"""Comparison with the REFERENCE's own torch GPU path (pytv/tv_GPU.py, pytv/tv_operators_GPU.py, unmodified) on the
same B200 - the four-way check of the reference's test-suite (tests.py:247-361) restated with seeded inputs.

The first test needs no copy of the reference: it reads the reference GPU path's float32 sub-gradient error per input,
recorded on a B200 by scripts/probe_ref_fp32.py (tests/golden/ref_gpu_fp32_err.json).  The direct output-to-output tests
need the git-ignored copy of the reference that travels with the repo (baseline/_ref); they are skipped when it is absent.

What the reference's float32 GPU path actually delivers on this hardware matters for the tolerance: its differences are
`torch.nn.functional.conv3d` calls, which run in TF32 by default (torch.backends.cudnn.allow_tf32 = True) - 10 mantissa
bits - so its float32 sub-gradient is 5e-3 .. 5e-1 away from its own float64 result (profiles/r02a_ref_fp32.json).  The
tests therefore (1) hold this library to max(1e-5, 2 x the reference GPU path's own error) against the float64 oracle, and
(2) with TF32 switched off - the reference at its best - compare the two GPU outputs with each other directly."""
import importlib
import json
import os
import sys
import warnings

import numpy as np
import pytest
import torch

import cases
import pytv_b200 as pytv
from oracle import tv_oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
SCHEMES = cases.SCHEMES


@pytest.fixture(scope="module")
def ref():
    if not os.path.isdir(os.path.join(REF_DIR, "pytv")):
        pytest.skip("baseline/_ref (the reference package) is not present")
    sys.path.insert(0, REF_DIR)
    warnings.filterwarnings("ignore")
    try:
        return importlib.import_module("pytv")
    except Exception as e:        # e.g. a dependency of the reference missing on the box
        pytest.skip("the reference does not import here: %r" % (e,))


@pytest.fixture(scope="module")
def ref_err():
    with open(os.path.join(ROOT, "tests", "golden", "ref_gpu_fp32_err.json")) as f:
        return json.load(f)["max_abs_err"]


@pytest.fixture
def no_tf32():
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = old


def _volumes():
    rs = np.random.RandomState(5)
    return {"readme": cases.readme_volume().astype(np.float32),
            "smooth64": (np.cumsum(rs.randn(6, 3, 64, 64), axis=-1) * 0.01).astype(np.float32)}


KWS = {"default": dict(), "rt": dict(reg_time=2 ** -5), "rz_rt": dict(reg_z_over_reg=0.5, reg_time=1.0)}


@pytest.mark.parametrize("kw_id", list(KWS))
@pytest.mark.parametrize("scheme", SCHEMES)
def test_subgradient_error_vs_reference_gpu_float32(ref_err, scheme, kw_id):
    kw = KWS[kw_id]
    for name, x in _volumes().items():
        tv_o, G_o = orc.tv(x.astype(np.float64), scheme, **kw)
        tv_m, G_m = getattr(pytv.tv_GPU, "tv_" + scheme)(x.copy(), **kw)
        ref_e = ref_err["%s/%s/%s" % (name, kw_id, scheme)]
        our_err = float(np.abs(G_m - G_o).max())
        assert our_err <= max(1e-5, 2.0 * ref_e), (name, our_err, ref_e)
        assert our_err <= 1e-5, (name, our_err)                 # and in fact within the north-star tolerance outright
        assert abs(float(tv_m) - tv_o) <= 1e-5 * tv_o, (name, float(tv_m), tv_o)


@pytest.mark.parametrize("scheme", SCHEMES)
def test_four_way_equality_float64(ref, scheme):
    """tests.py:304-361 (test_tv_D_DT_4D) with a seed: tv, G, D and D_T(D) of this library against the reference's GPU path,
    float64 (where TF32 plays no role), reg_time = 1 as in the reference's test."""
    rs = np.random.RandomState(8)
    for shape in ((20, 3, 12, 12), (1, 4, 16, 16), (6, 8, 9, 9)):
        x = rs.rand(*shape)
        kw = dict(reg_time=1.0)
        tv_r, G_r = getattr(ref.tv_GPU, "tv_" + scheme)(x.copy(), **kw)
        tv_m, G_m = getattr(pytv.tv_GPU, "tv_" + scheme)(x.copy(), **kw)
        assert float(tv_m) == pytest.approx(float(tv_r), rel=1e-12)
        np.testing.assert_allclose(G_m, G_r, rtol=0, atol=1e-11)
        D_r = getattr(ref.tv_operators_GPU, "D_" + scheme)(x, **kw)
        D_m = getattr(pytv.tv_operators_GPU, "D_" + scheme)(x, **kw)
        np.testing.assert_allclose(D_m, D_r, rtol=0, atol=1e-13)
        if shape[0] >= 5 or shape[0] == 1:      # the reference's D_T needs non-empty interior slices (SURVEY B5)
            try:
                DT_r = getattr(ref.tv_operators_GPU, "D_T_" + scheme)(D_r, **kw)
            except Exception:
                continue
            np.testing.assert_allclose(getattr(pytv.tv_operators_GPU, "D_T_" + scheme)(D_m, **kw), DT_r, rtol=0, atol=1e-12)


@pytest.mark.parametrize("scheme", SCHEMES)
def test_float32_against_reference_gpu_without_tf32(ref, scheme, no_tf32):
    """The reference GPU path at its best (TF32 off): the two float32 GPU results agree to the float32 rounding floor."""
    x = cases.readme_volume().astype(np.float32)
    kw = dict(reg_time=2 ** -5)
    tv_r, G_r = getattr(ref.tv_GPU, "tv_" + scheme)(x.copy(), **kw)
    tv_m, G_m = getattr(pytv.tv_GPU, "tv_" + scheme)(x.copy(), **kw)
    assert float(np.abs(G_m - G_r).max()) <= 1e-5
    assert abs(float(tv_m) - float(tv_r)) <= 1e-5 * abs(float(tv_r))
    D_r = getattr(ref.tv_operators_GPU, "D_" + scheme)(x, **kw)
    np.testing.assert_allclose(getattr(pytv.tv_operators_GPU, "D_" + scheme)(x, **kw), np.asarray(D_r, dtype=np.float32), rtol=0, atol=1e-5)
