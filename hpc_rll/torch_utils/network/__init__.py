from di_hpc_b200.torch_utils.network.scatter_connection import ScatterConnection  # noqa: F401
