"""Helpers shared by the test modules: the committed golden fixtures (tests/golden/*.npz), error measures, and the
autouse fixtures of the GPU tests (a module imports them by name to use them)."""
import os

import numpy as np
import pytest
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def shapes_from(gold):
    return {str(k): tuple(int(s) for s in sh.split(",") if s) for k, sh in zip(gold["keys"], gold["shapes"])}


def rel_err(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def close(a, b, rel=1e-4, scale=0.0):
    """||a - b|| <= rel * max(||b||, 0.1 * scale).

    ``scale`` (the largest gradient norm of the module under test) gives a floor for gradients that
    are mathematically zero - e.g. a conv bias feeding a train-mode BatchNorm - where both sides hold
    nothing but rounding noise proportional to the other gradients.
    """
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm()) <= rel * max(float(b.norm()), 0.1 * scale)


@pytest.fixture(autouse=True)
def _exact_fp32_library_math():
    # the parity bar is fp32: keep cuDNN / cuBLAS off TF32 for the PyTorch layers around our kernels
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


OPTION_DEFAULTS = {"mr_fwd_form": 2, "mr_bwd_form": 2, "knn_epilogue": 0, "edge_bwd_row": 1, "gather_row": 1, "edge_row": 1,
                   "maxk_row": 1, "bn_reverse": 1, "bn_persistent": 1, "bn_l2_keep_mb": 80, "check_index": 0, "conv_gemm": 1}


@pytest.fixture(autouse=True)
def _default_kernel_options():
    """Kernel-selection options are process-wide: every test starts from, and leaves, the defaults."""
    from grafp_b200 import ops
    for name, value in OPTION_DEFAULTS.items():
        ops.set_option(name, value)
    yield
    for name, value in OPTION_DEFAULTS.items():
        ops.set_option(name, value)


def bn_moments(ws, C):
    """The per-channel (sum, sum of squares) doubles inside a BatchNorm workspace (256-byte aligned, bn_fused.cu)."""
    off = (-ws.data_ptr()) % 256
    return ws[off:off + 16 * C].view(torch.float64).view(2, C)
