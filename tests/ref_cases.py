"""The cases of tests/test_oracle_vs_ref.py: inputs beyond the committed fixtures (other
shapes, up-sampling, edge cases), each run through a checker and returned as named outputs.

tests/golden/make_golden.py runs every case through the reference's own translation units
and stores a digest of each output in tests/golden/ref_cases.json (and the BA pair matrices,
which are inputs of the restatement, in tests/golden/ref_ba_mats.npz); the tests run the same
cases through the plain-C restatement and compare digests, so equal digests mean bit-identical
results without the reference being present."""
import hashlib
import json
import math

import numpy as np

from openpano_b200 import synth
from openpano_b200._abi import default_params
from tests import golden_util as gu

GOLDEN_JSON = gu.GOLDEN / "ref_cases.json"
BA_MATS = "ref_ba_mats.npz"

SIFT_SHAPES = [(300, 200, 7), (200, 300, 8), (157, 211, 9)]
WIDE_WINDOWS = [(8, 4.5), (17, 9.0)]
WARP_SHAPES = [(200, 140, 1.0), (141, 173, 0.8), (160, 120, 1.3)]
PROJECTIONS = [0, 1, 2]
PROJECTION_BANDS = [0, 2]
RATIOS = [(0.6, 1, 60), (0.95, 150, 190)]
LAZY_ORDERED = [(0, 0), (1, 1)]
RANSAC_CASES = [(300, 200, 1), (8, 50, 2), (1200, 64, 3)]
BA_CASES = [(4, 50, 1, 2), (8, 300, 2, 6), (3, 1, 3, 0), (16, 1000, 4, 30)]


def key(name, *args):
    return f"{name}[{'-'.join(str(a) for a in args)}]"


def digest(a):
    """dtype, shape and a SHA-256 prefix of the bytes: equal digests <=> gu.same_bits."""
    a = np.ascontiguousarray(a)
    return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()[:16]}"


def summary(out):
    """Arrays -> digests, everything else as JSON stores it."""
    return json.loads(json.dumps({k: digest(v) if isinstance(v, np.ndarray) else v for k, v in out.items()}))


def golden(name, *args):
    if not hasattr(golden, "_cache"):
        golden._cache = json.loads(GOLDEN_JSON.read_text())
    return golden._cache[key(name, *args)]


def check(out, name, *args):
    """The restatement's outputs of one case against the reference's, output by output."""
    want, got = golden(name, *args), summary(out)
    assert got.keys() == want.keys()
    bad = [k for k in want if got[k] != want[k]]
    assert not bad, f"{key(name, *args)}: differs from the reference in {bad}"


# ----------------------------------------------------------------------------- SIFT
def _trace(tr, noct, nscale):
    out = {"working_size": list(tr.working_size()), "plane0": tr.plane(0)}
    for o in range(noct):
        out[f"octave_size_o{o}"] = list(tr.octave_size(o))
        for l in range(nscale):
            out[f"gauss_o{o}_l{l}"] = tr.plane(1, o, l)
        for l in range(nscale - 1):
            out[f"dog_o{o}_l{l}"] = tr.plane(2, o, l)
        for l in range(1, nscale):
            out[f"mag_o{o}_l{l}"] = tr.plane(3, o, l)
            out[f"ort_o{o}_l{l}"] = tr.plane(4, o, l)
    for st in range(3):
        out[f"points{st}"] = tr.points(st)
    out["coor"], out["desc"] = tr.descriptors()
    tr.close()
    return out


def sift_every_stage(chk, w, h, seed):
    img = synth.make_canvas(h, w, seed)
    return dict(input=img, **_trace(chk.sift_trace(img), 4, 7))


def sift_other_params(chk):
    img = synth.make_canvas(180, 260, 31)
    p = default_params(num_octave=3, num_scale=6, contrast_thres=3e-2, edge_ratio=10.0, sift_working_size=300)
    return dict(input=img, **_trace(chk.sift_trace(img, p), 3, 6))


def sift_wide_windows(chk, hist_scale, ori_radius):
    img = synth.make_canvas(200, 280, 41)
    coor, desc = chk.sift_detect(img, default_params(desc_hist_scale_factor=hist_scale, ori_radius=ori_radius))
    return {"input": img, "coor": coor, "desc": desc}


def sift_flat_image(chk):
    return {"n_desc": len(chk.sift_detect(np.full((120, 160, 3), 0.25, np.float32))[1])}


# ----------------------------------------------------------------------------- matcher
def match_ragged_and_ties(chk):
    rng = np.random.RandomState(3)
    a = synth.rootsift_like(260, 5)
    b = np.concatenate([a[:80], a[:80], a[150:]])                   # exact duplicates: zero-distance ties
    noisy = (a[rng.permutation(260)][:200] + rng.randn(200, 128).astype(np.float32) * 36).astype(np.float32)
    sets = ((a, b), (b, a), (a, noisy), (noisy, a), (a[:1], b), (b, a[:1]), (a[:2], a[:2]))
    out = {"a": a, "noisy": noisy}
    out.update({f"pairs{k}": chk.match(x, y) for k, (x, y) in enumerate(sets)})
    return out


def match_other_ratios(chk, ratio):
    """MATCH_REJECT_NEXT_RATIO is a config value (config.cfg:33).  The reference squares it into a
    function-local `static const` on the FIRST call (matcher.cc:16, :91), i.e. it is frozen per
    process exactly like the config file is: the reference side of this case runs in a fresh process."""
    rng = np.random.RandomState(21)
    a = synth.rootsift_like(220, 22)
    b = (a[rng.permutation(220)][:190] + rng.randn(190, 128).astype(np.float32) * 30).astype(np.float32)
    p = default_params(match_reject_next_ratio=ratio)
    return {"a": a, "b": b, "ab": chk.match(a, b, p), "ba": chk.match(b, a, p)}


# ----------------------------------------------------------------------------- warp / blend
def cyl_warp(chk, w, h, hf):
    img = synth.make_canvas(h, w, 61)
    k = np.array([[3.5, -2.25], [-60.0, 40.0]])
    out, kk = chk.cyl_warp(img, k, hf)
    return {"input": img, "shape": list(chk.cyl_warp_shape(w, h, hf)), "out": out, "kpts": kk}


def cyl_warp_other_focal(chk):
    img = synth.make_canvas(120, 180, 62)
    p = default_params(focal_length=24.0)
    k = np.array([[10.0, 5.0], [-80.0, -50.0]])
    out, kk = chk.cyl_warp(img, k, 1.0, p)
    return {"input": img, "shape": list(chk.cyl_warp_shape(180, 120, 1.0, p)), "out": out, "kpts": kk}


def blend_projections(chk, projection, bands):
    imgs, org = synth.make_stack(3, 160, 110, 60, 71)
    items = []
    for k, (x, y) in enumerate(org):
        if projection == 0:
            th = 0.003 * (k - 1)
            H = np.array([[math.cos(th), -math.sin(th), x - 80], [math.sin(th), math.cos(th), 2 * k], [1e-5 * k, -2e-5, 1.0]])
        else:
            f = 300.0
            H = np.array([[1 / f, 0, (x - 80) / f], [0, 1 / f, 0.004 * k], [0, 0, 1]])
        items.append((k * 60, 0, k * 60 + 160, 115, list(np.linalg.inv(H).ravel())))
    res = 1.0 if projection == 0 else 1 / 300.0
    pmin = (-80.0, -55.0) if projection == 0 else (-0.3, -0.2)
    geom = dict(projection=projection, res_x=res, res_y=res, proj_min_x=pmin[0], proj_min_y=pmin[1])
    return {"input": np.stack(imgs), "out": chk.blend(imgs, items, geom, bands)}


def blend_scaled_resolution(chk, lazy, ordered):
    """MAX_OUTPUT_SIZE shrinks the canvas through `resolution` (stitcher_image.cc:108-119): the
    blend map then samples the sources at a stride > 1."""
    imgs, org = synth.make_stack(3, 200, 150, 80, 73)
    items, geom = synth.translation_blend_setup(org, 200, 150, max_output_size=170)
    p = default_params(lazy_read=lazy, ordered_input=ordered)
    return {"input": np.stack(imgs), "res_x": geom["res_x"], "linear": chk.blend(imgs, items, geom, 0, p),
            "multiband3": chk.blend(imgs, items, geom, 3, p)}


# ----------------------------------------------------------------------------- 8-bit boundary
def random_mosaic(rng, h, w):
    m = rng.rand(h, w, 3).astype(np.float32)
    for _ in range(rng.randint(0, 6)):
        y0, x0 = rng.randint(0, h), rng.randint(0, w)
        m[y0:y0 + rng.randint(1, 8), x0:x0 + rng.randint(1, 10)] = -1
    if rng.rand() < 0.4:
        m[:rng.randint(0, 4)] = -1
        m[:, :rng.randint(0, 5)] = -1
    return m


def imgio_read_write(chk):
    """read_img / write_rgb (the reference's imgio.cc through lossless PNM files)."""
    rng = np.random.RandomState(11)
    allv = np.arange(256, dtype=np.uint8).reshape(16, 16)
    pixs = (rng.randint(0, 256, (37, 53, 3)).astype(np.uint8), np.stack([allv] * 3, -1), allv,
            rng.randint(0, 256, (9, 31)).astype(np.uint8))
    out = {f"read{k}": chk.read_img_rgb8(pix) for k, pix in enumerate(pixs)}
    m = random_mosaic(rng, 40, 60)
    m[0, 0] = (1.0, 0.0, 0.999999)
    m[0, 1] = np.float32(1.0) / np.float32(255.0) * np.arange(1, 4, dtype=np.float32)
    out.update(mosaic=m, write=chk.write_rgb8(m))
    return out


def crop_cases():
    rng = np.random.RandomState(12)
    cases = [random_mosaic(rng, rng.randint(5, 60), rng.randint(5, 90)) for _ in range(25)]
    cases.append(-np.ones((6, 7, 3), np.float32))                  # nothing valid: 0 x 1 result
    cases.append(rng.rand(8, 9, 3).astype(np.float32))              # everything valid
    return cases


def imgio_crop(chk):
    """Width / height of the rectangle and the cropped pixels (x0, y0 are -1 from the reference build)."""
    out = {}
    for k, m in enumerate(crop_cases()):
        rect, cropped = chk.crop(m)
        out[f"input{k}"], out[f"wh{k}"], out[f"crop{k}"] = m, rect[2:], cropped
    return out


# ----------------------------------------------------------------------------- host geometry
def ransac_scoring(chk, n_match, n_hyp, seed):
    from tests.ransac_util import ransac_case
    kp1, kp2, homos, thres = ransac_case(n_match, n_hyp, seed)
    best, count, counts, flags = chk.ransac_score(kp1, kp2, homos, thres)
    return {"input": np.concatenate([kp1.ravel(), kp2.ravel(), homos.ravel()]), "best": best, "count": count,
            "counts": counts, "flags": flags}
