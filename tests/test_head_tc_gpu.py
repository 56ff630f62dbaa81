"""Tensor-core projection head at shapes where the forward kernel's four warp groups get unequal tile counts.

head_fwd_tc_kernel hands the tiles of a persistent CTA to four warp groups in rotation (group g takes tiles g, g + 4,
...), so a CTA with 4 k + 1 .. 4 k + 3 tiles leaves some groups one tile short.  These planes give every CTA several
tiles, with both ragged and even splits across the 148 CTAs, at the widest channel count (C = 32: five K steps with
the ones column of b1) and the widest output (V = 8).  The checks are those of test_kernels_gpu.py's head test.
"""
import pytest

import test_kernels_gpu as K

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from fno_b200 import lib as L

    L.load()
    return L


@pytest.mark.parametrize("bwd_tc", [True, False], ids=["tcgen05", "fp32"])
@pytest.mark.parametrize("spatial,C,V,B", [
    ((64, 64), 20, 2, 40),      # 1280 tiles: 8 or 9 per CTA, groups of 2 / 2 / 2 / 2 or 3 / 2 / 2 / 2 tiles
    ((256, 256), 32, 3, 2),     # C = 32: 1024 tiles, 6 or 7 per CTA
    ((256, 256), 12, 8, 2),     # V = 8
])
def test_head_forward_backward_many_tiles(lib, monkeypatch, spatial, C, V, B, bwd_tc):
    K.test_head_forward_backward(lib, monkeypatch, spatial, C, V, B, bwd_tc)
