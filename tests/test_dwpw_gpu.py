"""The TMA-fed depthwise 5x5 -> 1x1 kernel (dwpw_tma_kernel) gives the bits of the cp.async kernel it replaces (dwpw_tc_kernel, the
-DYF_DWPW_TMA=0 build): conv5_4 / conv4_1_3 taps and both heads byte-equal, on every tile shape and on the maps that fall back."""
import os
import sys

import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))
import dwpw_ab  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="session")
def old_lib(tmp_path_factory):
    return dwpw_ab.build_old(str(tmp_path_factory.mktemp("dwpw_cpasync")))


# 512x640: small-batch (B = 1, 2), throughput with a ragged last wave (B = 37) and the bench batch; 256x320: TMA at 1/16, the 10-column
# 1/32 map falls back; 416x416: 26- and 13-column maps, fallback only; the 80-class network keeps its heads on the FFMA engine.
@pytest.mark.parametrize("res,B,nc", [("512x640", 1, 3), ("512x640", 2, 3), ("512x640", 37, 3), ("512x640", 256, 3),
                                      ("256x320", 3, 3), ("416x416", 2, 3), ("512x640", 2, 80)])
def test_dwpw_tma_bit_identical(old_lib, res, B, nc):
    import __graft_entry__ as ge
    new = dwpw_ab.run_child(ge.LIB, res, B, nc, profile=False)
    old = dwpw_ab.run_child(old_lib, res, B, nc, profile=False)
    assert new["sha"] == old["sha"], (new["sha"], old["sha"])
