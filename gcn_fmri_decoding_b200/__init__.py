"""B200-native graph-convolution hot path of GCN_fmri_decoding (see DESIGN.md).

``graphs`` / ``graclus`` / ``synth`` are host-side NumPy/SciPy (input contract);
``ops`` / ``models`` / ``train`` need PyTorch and the in-tree ``libgcnb200.so``
(sm_100a CUDA kernels, C ABI in ``include/gcnb200.h``).  There is no CPU
compute path: calling a layer without the library or without a GPU raises.
"""
from . import graclus, graphs, synth  # noqa: F401

__all__ = ["graclus", "graphs", "synth", "ops", "models", "finetune", "train", "plan"]


def __getattr__(name):  # lazy: importing the package must not require torch
    if name in ("ops", "models", "finetune", "train", "plan", "_lib"):
        import importlib

        return importlib.import_module("." + name, __name__)
    raise AttributeError(name)
