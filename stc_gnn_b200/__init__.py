"""stc_gnn_b200 -- B200-native (sm_100a) implementation of STC-GNN's graph-convolution GRU cell.

Public surface:
  STC_Cell            drop-in for the reference class (framework/STC_GNN.py:51-79)
  stc_cell_forward    functional form (differentiable)
  CsrSupport          sparse spatial support: fixed pattern, constant or learnable edge values
  support_apply       the spatial mode product on its own
  support_apply_edge_grad  the adjoint CSR hop with the edge-value gradient fused in
  SparseGraphGenerator  the reference's spatial graph generator on a fixed CSR pattern (returns a learnable CsrSupport)
  pair_softmax_csr    its differentiable core: row softmax of relu(<U_n,V_m> - <V_n,U_m>) over the stored edges
  install / run_main  rebind STC_GNN.STC_Cell so Model_Trainer.py / Main.py run unchanged
  dp                  batch data-parallel gradient bucket (one flat all-reduce per step)
  halo                row-partitioned CSR support with per-hop halo exchange
  GraphedStep         CUDA-graph capture/replay of one forward+backward step (launch-bound small batches)
"""
from .cell import STC_Cell, GraphConvParams, stc_cell_forward  # noqa: F401
from .support import CsrSupport, support_apply, support_apply_edge_grad  # noqa: F401
from .install import install, run_main  # noqa: F401
from .stack import RecurrentStack  # noqa: F401
from .graph import GraphedStep  # noqa: F401
from .sparse_mgp import SparseGraphGenerator, pair_softmax_csr, pair_softmax_partitioned  # noqa: F401
from . import dp, halo, mgp  # noqa: F401
