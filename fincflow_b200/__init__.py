"""fincflow_b200 -- B200-native FInC invertible k x k convolution hot path.

Public surface (mirrors the reference's fastflow package for this path):

    FlowLayer, ModifiedGradFlowLayer, PreprocessingFlowLayer     fastflow/layers/flowlayer.py
    FlowSequential                                               fastflow/layers/flowsequential.py
    PaddedConv2d                                                 fastflow/layers/conv.py
    FastFlowUnit, clear_grad                                     fastflow/fastflow.py, train/experiment.py:16-18
    weight_grad_in_reverse                                       (reverse records a graph for the weights alone)
    flows.FastFlow (+ fastflow_mnist / _cifar10 / _imagenet32 / _imagenet64 builders)

Everything computes through the C ABI in include/fincflow_b200.h (libfincflow_b200.so, hand-written
sm_100a CUDA); there is no CPU fallback.  Importing the package does not load the library -- the
first kernel call does, and raises if it has not been built (`python -m fincflow_b200.build`).
"""
__version__ = "0.2.0"

_LAZY = {
    "FlowLayer": ("layers.flowlayer", "FlowLayer"),
    "ModifiedGradFlowLayer": ("layers.flowlayer", "ModifiedGradFlowLayer"),
    "PreprocessingFlowLayer": ("layers.flowlayer", "PreprocessingFlowLayer"),
    "FlowSequential": ("layers.flowsequential", "FlowSequential"),
    "PaddedConv2d": ("layers.conv", "PaddedConv2d"),
    "FastFlowUnit": ("fastflow", "FastFlowUnit"),
    "clear_grad": ("fastflow", "clear_grad"),
    "weight_grad_in_reverse": ("ops", "weight_grad_in_reverse"),
    "FastFlow": ("flows", "FastFlow"),
    "GaussianPrior": ("flows", "GaussianPrior"),
    "fastflow_mnist": ("flows", "fastflow_mnist"),
    "fastflow_cifar10": ("flows", "fastflow_cifar10"),
    "fastflow_imagenet32": ("flows", "fastflow_imagenet32"),
    "fastflow_imagenet64": ("flows", "fastflow_imagenet64"),
}
__all__ = sorted(_LAZY) + ["__version__"]


def __getattr__(name):
    if name in _LAZY:
        import importlib

        mod, attr = _LAZY[name]
        return getattr(importlib.import_module(f"{__name__}.{mod}"), attr)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
