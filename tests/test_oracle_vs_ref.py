"""CPU: the plain-C oracle against the reference's own translation units on inputs beyond
the committed fixtures: other shapes, up-sampling, edge cases.  The reference's outputs are
stored as digests (tests/golden/ref_cases.json, made by tests/golden/make_golden.py from the
cases in tests/ref_cases.py); every comparison is bit for bit."""
import numpy as np
import pytest

from openpano_b200 import synth
from openpano_b200._abi import default_params
from tests import golden_util as gu
from tests import ref_cases as rc


@pytest.mark.parametrize("w,h,seed", rc.SIFT_SHAPES)
def test_sift_every_stage(orc, w, h, seed):
    out = rc.sift_every_stage(orc, w, h, seed)
    rc.check(out, "sift_every_stage", w, h, seed)
    assert len(out["desc"]) > 20


def test_sift_other_params(orc):
    rc.check(rc.sift_other_params(orc), "sift_other_params")


@pytest.mark.parametrize("hist_scale,ori_radius", rc.WIDE_WINDOWS)
def test_sift_wide_windows(orc, hist_scale, ori_radius):
    """The parameter sets tests/test_gpu_sift.py::test_sift_wide_descriptor_windows runs on the GPU (descriptor
    windows wider than one interval-table block of the kernel, wide orientation windows): the restatement
    against the reference's own TUs, so that the GPU-vs-oracle result there is pinned to the reference too."""
    out = rc.sift_wide_windows(orc, hist_scale, ori_radius)
    rc.check(out, "sift_wide_windows", hist_scale, ori_radius)
    assert len(out["desc"]) > 100


def test_sift_flat_image(orc):
    out = rc.sift_flat_image(orc)
    rc.check(out, "sift_flat_image")
    assert out["n_desc"] == 0


def test_match_ragged_and_ties(orc):
    rc.check(rc.match_ragged_and_ties(orc), "match_ragged_and_ties")


@pytest.mark.parametrize("w,h,hf", rc.WARP_SHAPES)
def test_cyl_warp(orc, w, h, hf):
    rc.check(rc.cyl_warp(orc, w, h, hf), "cyl_warp", w, h, hf)


@pytest.mark.parametrize("projection", rc.PROJECTIONS)
@pytest.mark.parametrize("bands", rc.PROJECTION_BANDS)
def test_blend_projections(orc, projection, bands):
    out = rc.blend_projections(orc, projection, bands)
    rc.check(out, "blend_projections", projection, bands)
    assert (out["out"] >= 0).mean() > 0.3


def test_imgio_read_write(orc):
    """read_img / write_rgb through the reference's imgio.cc (lossless PNM files) vs the restatement."""
    rc.check(rc.imgio_read_write(orc), "imgio_read_write")


def test_imgio_crop(orc):
    out = rc.imgio_crop(orc)
    rc.check(out, "imgio_crop")
    for k, m in enumerate(rc.crop_cases()):
        x0, y0, cw, ch = orc.crop(m)[0]
        assert np.array_equal(out[f"crop{k}"], m[y0:y0 + ch, x0:x0 + cw])


@pytest.mark.parametrize("ratio,lo,hi", rc.RATIOS)
def test_match_other_ratios(orc, ratio, lo, hi):
    """MATCH_REJECT_NEXT_RATIO other than the default (the reference's side made in a fresh process
    per ratio: it freezes the value at its first match)."""
    out = rc.match_other_ratios(orc, ratio)
    rc.check(out, "match_other_ratios", ratio)
    assert lo <= len(out["ab"]) <= hi


@pytest.mark.parametrize("lazy,ordered", rc.LAZY_ORDERED)
def test_blend_scaled_resolution(orc, lazy, ordered):
    out = rc.blend_scaled_resolution(orc, lazy, ordered)
    rc.check(out, "blend_scaled_resolution", lazy, ordered)
    assert out["res_x"] > 2.0 and (out["linear"] >= 0).mean() > 0.5


def test_cyl_warp_other_focal(orc):
    rc.check(rc.cyl_warp_other_focal(orc), "cyl_warp_other_focal")


def test_oracle_mt_equals_oracle(orc):
    """oracle/liboracle_mt.so (independent loops under OpenMP, used by the BASELINE-size GPU
    parity tests) must be bit-identical to the single-thread restatement."""
    from tests.checker import get_checker, have
    if not have("orc_mt"):
        pytest.skip("oracle/liboracle_mt.so not built")
    mt = get_checker("orc_mt")
    rng = np.random.RandomState(21)
    a = synth.rootsift_like(900, 4)
    b = a[rng.permutation(900)][:700] + rng.randn(700, 128).astype(np.float32) * 25.0
    for x, y in ((a, b), (b, a), (a[:1], b), (a, a)):
        assert np.array_equal(orc.match(x, y), mt.match(x, y))
    imgs, org = synth.make_stack(5, 260, 200, 90, 77, rows=2, step_y=70)
    items, geom = synth.translation_blend_setup(org, 260, 200)
    for bands in (0, 2, 5):
        for lazy in (0, 1):
            p = default_params(lazy_read=lazy, multiband=bands)
            assert gu.same_bits(orc.blend(imgs, items, geom, bands, p), mt.blend(imgs, items, geom, bands, p)), (bands, lazy)


@pytest.mark.parametrize("n_match,n_hyp,seed", rc.RANSAC_CASES)
def test_ransac_scoring(orc, n_match, n_hyp, seed):
    """TransformEstimation::get_inliers itself (the reference TU, reached through the shim) against
    the restatement: per-hypothesis counts, first-maximum selection, inlier flags."""
    out = rc.ransac_scoring(orc, n_match, n_hyp, seed)
    rc.check(out, "ransac_scoring", n_match, n_hyp, seed)
    assert out["count"] > 0.5 * n_match


@pytest.mark.parametrize("n_cam,per_pair,seed,extra", rc.BA_CASES)
def test_ba_jacobian(orc, n_cam, per_pair, seed, extra):
    """IncrementalBundleAdjuster::calcJacobianSymbolic itself (the reference TU, compiled where it lies
    by oracle/refshim/ref_ba.cc) against the restatement: every J row and every J^T J entry, bit for bit —
    including reversed pairs, repeated camera pairs and the identity camera's small-angle branch.  The
    per-pair matrices the restatement takes are the reference's own (tests/golden/ref_ba_mats.npz)."""
    from tests.ba_util import ba_case
    _, pairs, pts = ba_case(n_cam, per_pair, seed, extra_pairs=extra)
    mats = gu.load(rc.BA_MATS)[rc.key("ba_jacobian", n_cam, per_pair, seed, extra)]
    rows, jtj = orc.ba_jacobian(n_cam, pairs, mats, pts[:, :2])
    rc.check({"input": pts, "rows": rows, "jtj": jtj}, "ba_jacobian", n_cam, per_pair, seed, extra)
    assert np.isfinite(rows).all() and (jtj != 0).any()
