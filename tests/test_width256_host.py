"""The 256-wide denoiser without a GPU: the oracle-generated fixtures of tests/golden/w256_*.npz regenerate bit for bit
(tools/make_golden_width256.py), and d3d_create refuses every width / head / mode combination outside the supported set
with the documented code (-3) and a message that names the supported set."""
import ctypes
import os
import sys

import numpy as np
import pytest

from diff3dhpe_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def test_width256_fixtures_regenerate_bit_for_bit(golden):
    import make_golden_width256 as mk
    for name, arrays in mk.all_cases().items():
        g = golden(name)
        assert int(g["oracle_generated"]) == 1
        assert sorted(g) == sorted(arrays), name
        for k, v in arrays.items():
            assert np.array_equal(np.asarray(v), g[k]), f"{name}: {k} differs from the committed fixture"


def _create(F, J, C, heads, hidden, gemm_mode=_lib.GEMM_TC_F4C, attn_mode=_lib.ATTN_DEFAULT):
    lib = _lib.load()
    h = ctypes.c_void_p()
    cfg = _lib.Config(F, J, C, 8, heads, hidden, 1, 1, gemm_mode, attn_mode, 0, 1)
    rc = lib.d3d_create(ctypes.byref(cfg), ctypes.byref(h))
    if rc == 0:
        lib.d3d_destroy(h)
    return rc, lib.d3d_last_error(None).decode()


@pytest.mark.parametrize("C", [128, 384, 1024])
def test_create_refuses_widths_outside_256_512(C):
    rc, msg = _create(27, 17, C, 8, 2 * C)
    assert rc == -3 and "embed_dim 256 or 512" in msg and "8 heads" in msg


@pytest.mark.parametrize("heads,hidden", [(4, 512), (16, 512), (8, 1024), (8, 256)])
def test_create_refuses_other_heads_or_hidden_at_256(heads, hidden):
    rc, msg = _create(27, 17, 256, heads, hidden)
    assert rc == -3 and "embed_dim 256 or 512" in msg and "2 * embed_dim" in msg


@pytest.mark.parametrize("gemm_mode,attn_mode", [
    (_lib.GEMM_TC_SPLIT3, _lib.ATTN_DEFAULT), (_lib.GEMM_TC_FP16, _lib.ATTN_DEFAULT), (_lib.GEMM_SIMT_FP32, _lib.ATTN_DEFAULT),
    (_lib.GEMM_TC_F8C, _lib.ATTN_DEFAULT), (_lib.GEMM_SIMT_F8C, _lib.ATTN_DEFAULT), (_lib.GEMM_SIMT_F4C, _lib.ATTN_DEFAULT),
    (_lib.GEMM_TC_F4C, _lib.ATTN_SIMT), (_lib.GEMM_TC_F4C, _lib.ATTN_MMA_SYNC)])
def test_create_refuses_validation_modes_at_256(gemm_mode, attn_mode):
    rc, msg = _create(27, 17, 256, 8, 512, gemm_mode, attn_mode)
    assert rc == -3 and "D3D_GEMM_TC_F4C with attn_mode D3D_ATTN_DEFAULT only" in msg


def test_create_refuses_other_joint_counts_at_256():
    rc, msg = _create(27, 16, 256, 8, 512)
    assert rc == -3 and "num_joints 17" in msg
