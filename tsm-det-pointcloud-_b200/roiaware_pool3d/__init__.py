"""The ``roiaware_pool3d`` ops (point-head target assignment, ground-truth sampling, PartA2's RoI pooling) -- same names
and arguments as ``/root/reference/pcdet/ops/roiaware_pool3d`` (``roiaware_pool3d_cuda`` = its pybind module re-hosted
on the C ABI, ``roiaware_pool3d_utils`` = its Python wrappers: ``points_in_boxes_cpu``, ``points_in_boxes_gpu``,
``RoIAwarePool3d``)."""
