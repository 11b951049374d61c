"""Host-side checks of precision 3 that need no GPU: workspace sizes and the three-way bf16 split."""
import ctypes as C
import os
import sys

import numpy as np
import torch

from avddpg_b200 import _lib
from avddpg_b200.model import make_dims

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))


def test_forward_workspace_bytes():
    lib = _lib.load()
    for d in (make_dims(4, 256, 48, 128), make_dims(3, 64, 16, 32)):
        for A, R in ((1, 64), (4, 1000), (3, 70)):
            for critic in (0, 1):
                F = d.l1 + (d.la if critic else 0)
                plain = A * R * (F + d.l2) * 4 + A * F * d.l2 * 2 + 512
                for prec in (0, 1, 2):
                    assert lib.avd_forward_workspace_bytes(C.byref(d), A, R, critic, prec) == plain
                assert lib.avd_forward_workspace_bytes(C.byref(d), A, R, critic, 3) == A * R * (6 * F + 4 * d.l2) + 3 * A * F * d.l2 * 2 + 512
    assert lib.avd_forward_workspace_bytes(None, 1, 1, 0, 0) == -1


def test_learn_workspace_covers_planes():
    lib = _lib.load()
    d = make_dims(4, 256, 48, 128)
    A, R = 4, 262_144
    N, F = A * R, d.l1 + d.la
    p0 = lib.avd_ddpg_workspace_bytes(C.byref(d), A, R, 0)
    p3 = lib.avd_ddpg_workspace_bytes(C.byref(d), A, R, 3)
    # 2 more bytes per element of H, H1a and dz2 (6 B instead of 4), three planes of the six 16-bit weight packs
    assert p3 - p0 == N * (F + d.l1 + d.l2) * 2 + 2 * A * (3 * F + 3 * d.l1) * d.l2 * 2
    assert lib.avd_ddpg_workspace_bytes(C.byref(d), A, R, 2) < p0          # the fused kernels keep activations on chip


def test_three_way_split_is_exact_for_fp32():
    import precision_model as P
    g = torch.Generator().manual_seed(3)
    x = torch.randn(100_000, generator=g) * torch.exp(torch.randn(100_000, generator=g) * 10)
    got = P.rnd(x.numpy(), "bf16x3")
    assert np.array_equal(got, x.numpy().astype(np.float64))
    assert not np.array_equal(P.rnd(x.numpy(), "bf16x2"), x.numpy().astype(np.float64))
