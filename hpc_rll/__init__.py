"""`hpc_rll` -- the reference's package name, re-exporting the B200-native implementation.

DI-engine imports `hpc_rll.rl_utils.{gae,td,upgo,vtrace,ppo}` (see SURVEY.md 3.5); those module
paths resolve to `di_hpc_b200.rl_utils.*`.  `hpc_rll.torch_utils.network.scatter_connection` (ScatterConnection)
resolves to `di_hpc_b200.torch_utils.network.scatter_connection`.  `hpc_rll.origin` (the reference's PyTorch
oracle) and `hpc_rll.torch_utils.network.rnn` (LSTM) are intentionally absent: out of scope (DESIGN.md section 8).
"""
