from .scatter_connection import ScatterConnection, ScatterConnectionFunction  # noqa: F401
