"""Host-side mirror of the reference package `hpc_rll.torch_utils` (module network.scatter_connection)."""
