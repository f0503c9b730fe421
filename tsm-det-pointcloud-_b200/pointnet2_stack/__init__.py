"""The ``pointnet2_stack`` ops that SA layers >= 1 and the head's VSA module call (SURVEY.md 8 f3): ball query, voxel
query (+ dilated), stacked grouping, stacked furthest point sampling and the stacked 3-NN / interpolation -- same
names and arguments as ``/root/reference/pcdet/ops/pointnet2/pointnet2_stack`` (``pointnet2_stack_cuda`` = its pybind
module re-hosted on the C ABI, ``pointnet2_utils`` / ``voxel_query_utils`` = its Python wrappers, ``pointnet2_modules.StackSAModuleMSG`` = its
multi-scale set abstraction, ``pointnet2_modules.StackPointnetFPModule`` = its feature propagation,
``pointnet2_modules.VectorPoolAggregationModuleMSG`` = its vector-pool local aggregation (PV-RCNN++), all with a fused
eval path)."""
from .pointnet2_modules import (StackPointnetFPModule, StackSAModuleMSG, VectorPoolAggregationModule,  # noqa: F401
                                VectorPoolAggregationModuleMSG, build_local_aggregation_module)
