"""hpc_b200 — B200-native CSR SpMM engine behind the PA4 `SpMM` operator surface.

Host-side mirror of the reference's operator interface (PA4/handout/include/spmm_base.h)
over the C ABI in include/spmm_b200.h. PyTorch is used only for device memory and streams.
"""
from ._lib import LIB_PATH, PlanInfo, SpmmB200Error  # noqa: F401
from .spmm import CSR, SpMM, SpMMB200, allocate, fill_normal, pack_light_host, plan_host, trim_memory, valid  # noqa: F401
from .graph import (  # noqa: F401
    GRAPH_SHAPES, RUN_ALL_DATASETS, gen_degrees, gen_graph, gen_named_graph, load_graph, partition_rows, plan_row_cost, rebase_ptr, set_host_threads,
    write_graph,
)
from .mg import MultiGpuSpMM  # noqa: F401
from .autograd import GraphAttention, GraphSpMM  # noqa: F401
