"""The proposal-network density kernels compiled for an exact level count (``k_density_fwd<L, 16, KEEP, true>`` and
``k_density_bwd_tc<L, SPLIT>``, L = 1..7 at hidden 16) at the level counts ``test_density_field_gpu.py`` does not reach: 2, 3, 4 and
6.  Levels 2, 4 and 6 give input widths that are whole float4s of a weight row, level 3 a float2 tail after one float4.  Same cases, reference and bounds as ``test_density_field_gpu.py``."""
import ctypes as C

import pytest
import torch

import density_reference as dref
from test_density_field_gpu import TOL_FEAT, _abi, _check, _d_density, _reference, _rel_max, _run

from cropnerf_b200 import _lib as L

pytestmark = pytest.mark.gpu

LEVELS = [2, 3, 4, 6]


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
@pytest.mark.parametrize("contraction", [True, False], ids=["contract", "aabb"])
@pytest.mark.parametrize("nl", LEVELS)
def test_exact_levels(dev, record_property, nl, contraction, precision):
    """The public operator path (fwd, bwd through cnb_density_field_bwd) at 37 rays x 53 samples."""
    case = dref.make_case(37, 53, nl, 16, contraction, seed=100 * nl + 16)
    dd = _d_density(case.R * case.S, seed=nl + 16)
    _check(_run(case, dev, dd, precision), _reference(case, dd, dev), record_property, precision, True)


@pytest.mark.parametrize("precision", ["fp32", "mixed"])
@pytest.mark.parametrize("nl", LEVELS)
def test_exact_levels_kept_features(dev, record_property, nl, precision):
    """cnb_density_field_fwd_keep / cnb_density_field_bwd_kept at 300 rays x 96 samples (more tiles than one CTA's first pass)."""
    case = dref.make_case(300, 96, nl, 16, True, seed=40 + nl)
    N = case.R * case.S
    dd = _d_density(N, seed=41)
    ref = _reference(case, dd, dev)
    a = _abi(case, dev, L.PREC_MIXED if precision == "mixed" else L.PREC_FP32)
    density = torch.empty(N, device=dev)
    feat = torch.empty((nl, N, 2), device=dev)
    st = L.stream_ptr(dev)
    L.check(L.lib().cnb_density_field_fwd_keep(C.byref(a["f"]), C.byref(a["sm"]), density.data_ptr(), feat.data_ptr(), st), "fwd_keep")
    err = _rel_max(feat.permute(1, 0, 2).reshape(N, 2 * nl), ref["feat"])
    record_property("err_feat", err)
    assert err <= TOL_FEAT, f"kept features: {err:.3e}"
    ddv = dd.to(dev)
    L.check(L.lib().cnb_density_field_bwd_kept(C.byref(a["f"]), C.byref(a["sm"]), ddv.data_ptr(), feat.data_ptr(), st), "bwd_kept")
    _check({"density": density, **a["g"]}, ref, record_property, precision, True)
