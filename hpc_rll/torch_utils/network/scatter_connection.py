from di_hpc_b200.torch_utils.network.scatter_connection import ScatterConnection, ScatterConnectionFunction  # noqa: F401
