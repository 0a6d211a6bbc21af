#!/usr/bin/env python
"""Generates tests/golden/*.npz from the REFERENCE's own translation units
(oracle/_ref/libopenpano_ref.so, built by oracle/Makefile from
/root/reference/src with -O2 -ffp-contract=off -msse3, single thread).

The reference ships no golden vectors for this path (SURVEY.md §4), so these
fixtures ARE the pin: the plain-C oracle and the CUDA engine are both compared
against them bit for bit.  Inputs come from openpano_b200.synth (seeded numpy);
each fixture stores a SHA-256 of its inputs so generator drift is detected.

Run in the build container (needs /root/reference):  python tests/golden/make_golden.py
"""
import hashlib
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))

from openpano_b200 import synth  # noqa: E402
from openpano_b200._abi import default_params  # noqa: E402
from tests.checker import get_checker  # noqa: E402

OUT = Path(__file__).resolve().parent


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def plane_crc(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest()[:8], np.uint64).copy()


def imgio(ref):
    """read_img / crop / write_rgb through the reference's own lib/imgio.cc + lib/imgproc.cc."""
    from tests.golden_util import imgio_inputs
    pix, grey, mos = imgio_inputs()
    rect, cropped = ref.crop(mos)
    np.savez_compressed(OUT / "imgio.npz", input_sha=np.array(sha(pix, grey, mos)),
                        read_rgb=ref.read_img_rgb8(pix), read_grey=ref.read_img_rgb8(grey),
                        crop_wh=rect[2:], cropped=cropped, write_full=ref.write_rgb8(mos),
                        write_cropped=ref.write_rgb8(cropped))
    print("imgio: crop", rect, cropped.shape)


def ba(ref):
    """The reference's own calcJacobianSymbolic (incremental_bundle_adjuster.cc:276-385) and the per-pair
    matrices, evaluated by the reference's own Homography / Camera operations (oracle/refshim/ref_ba.cc)."""
    from tests.ba_util import ba_case
    cams, pairs, pts = ba_case(5, 40, 5, extra_pairs=3)
    mats = ref.ba_pair_mats(cams, pairs)
    rows, jtj = ref.ba_jacobian_ref(cams, pairs, pts)
    np.savez_compressed(OUT / "ba_5cams.npz", input_sha=np.array(sha(cams, np.array(pairs), pts)),
                        mats=mats, rows=rows, jtj=jtj)
    print("ba:", len(pairs), "pairs,", len(pts), "matches")


_RATIO_SCRIPT = """
import json, sys
sys.path.insert(0, {root!r})
from tests import ref_cases as rc
from tests.checker import get_checker
print(json.dumps(rc.summary(rc.match_other_ratios(get_checker('ref'), {ratio}))))
"""


def ref_cases(ref):
    """The reference's outputs of every case of tests/test_oracle_vs_ref.py (tests/ref_cases.py)."""
    import json
    import subprocess
    from tests import ref_cases as rc
    from tests.ba_util import ba_case
    g = {}

    def put(fn, *args):
        g[rc.key(fn.__name__, *args)] = rc.summary(fn(ref, *args))

    for args in rc.SIFT_SHAPES:
        put(rc.sift_every_stage, *args)
    put(rc.sift_other_params)
    for args in rc.WIDE_WINDOWS:
        put(rc.sift_wide_windows, *args)
    put(rc.sift_flat_image)
    put(rc.match_ragged_and_ties)
    for args in rc.WARP_SHAPES:
        put(rc.cyl_warp, *args)
    put(rc.cyl_warp_other_focal)
    for projection in rc.PROJECTIONS:
        for bands in rc.PROJECTION_BANDS:
            put(rc.blend_projections, projection, bands)
    for args in rc.LAZY_ORDERED:
        put(rc.blend_scaled_resolution, *args)
    put(rc.imgio_read_write)
    put(rc.imgio_crop)
    for args in rc.RANSAC_CASES:
        put(rc.ransac_scoring, *args)
    for ratio, _, _ in rc.RATIOS:      # the reference freezes the ratio at its first match: one process each
        out = subprocess.run([sys.executable, "-c", _RATIO_SCRIPT.format(root=str(ROOT), ratio=ratio)],
                             capture_output=True, text=True, check=True)
        g[rc.key("match_other_ratios", ratio)] = json.loads(out.stdout.strip().splitlines()[-1])
    mats = {}
    for args in rc.BA_CASES:
        n_cam, per_pair, seed, extra = args
        cams, pairs, pts = ba_case(n_cam, per_pair, seed, extra_pairs=extra)
        k = rc.key("ba_jacobian", *args)
        mats[k] = ref.ba_pair_mats(cams, pairs)
        rows, jtj = ref.ba_jacobian_ref(cams, pairs, pts)
        g[k] = rc.summary({"input": pts, "rows": rows, "jtj": jtj})
    np.savez_compressed(OUT / rc.BA_MATS, **mats)
    rc.GOLDEN_JSON.write_text(json.dumps(g, indent=1, sort_keys=True) + "\n")
    print("ref_cases:", len(g), "cases")


def main():
    ref = get_checker("ref")
    assert ref.num_threads() == 1
    if sys.argv[1:] == ["imgio"]:      # add this fixture without rewriting the others
        imgio(ref)
        return
    if sys.argv[1:] == ["ba"]:
        ba(ref)
        return
    if sys.argv[1:] == ["ref_cases"]:
        ref_cases(ref)
        return
    imgio(ref)
    ba(ref)
    ref_cases(ref)

    # ---- SIFT chain on one 240x180 view
    img = synth.make_canvas(180, 240, 101)
    tr = ref.sift_trace(img)
    pts = [tr.points(s) for s in range(3)]
    coor, desc = tr.descriptors()
    planes = {f"gauss_o{o}_l{l}_crc": plane_crc(tr.plane(1, o, l)) for o in range(4) for l in range(7)}
    planes.update({f"dog_o{o}_l{l}_crc": plane_crc(tr.plane(2, o, l)) for o in range(4) for l in range(6)})
    np.savez_compressed(OUT / "sift_240x180.npz", input_sha=np.array(sha(img)),
                        working_size=np.array(tr.working_size()),
                        octave_sizes=np.array([tr.octave_size(o) for o in range(4)]),
                        dog_o0_l3=tr.plane(2, 0, 3)[40:60, 50:90].copy(),
                        raw=pts[0], refined=pts[1], oriented=pts[2], coor=coor, desc=desc, **planes)
    print("sift:", [len(p) for p in pts], desc.shape)

    # ---- matcher: two overlapping views + a noisy synthetic pair near the ratio threshold
    imgs, org = synth.make_stack(2, 240, 180, 90, 102)
    d0 = ref.sift_detect(imgs[0])[1]
    d1 = ref.sift_detect(imgs[1])[1]
    rng = np.random.RandomState(5)
    a = synth.rootsift_like(300, 6)
    b = (a[rng.permutation(300)][:260] + rng.randn(260, 128).astype(np.float32) * 28.0).astype(np.float32)
    c = (a[rng.permutation(300)][:280] + rng.randn(280, 128).astype(np.float32) * 38.0).astype(np.float32)
    np.savez_compressed(OUT / "match.npz", input_sha=np.array(sha(imgs[0], imgs[1], a, b, c)), d0=d0, d1=d1,
                        pairs_01=ref.match(d0, d1), pairs_10=ref.match(d1, d0), a=a, b=b, c=c,
                        pairs_ab=ref.match(a, b), pairs_ba=ref.match(b, a),
                        pairs_ac=ref.match(a, c), pairs_ca=ref.match(c, a))
    print("near-threshold pair:", len(ref.match(a, c)), "of 280")
    print("match:", len(d0), len(d1), len(ref.match(d0, d1)), len(ref.match(a, b)))

    # ---- cylinder warp
    wimg = synth.make_canvas(80, 120, 103)
    k = np.array([[10.5, -20.25], [-40.0, 30.0], [0.0, 0.0]])
    out, kk = ref.cyl_warp(wimg, k, 1.0)
    out2, kk2 = ref.cyl_warp(wimg, k, 0.9)
    np.savez_compressed(OUT / "cyl_warp_120x80.npz", input_sha=np.array(sha(wimg)),
                        shape=np.array(ref.cyl_warp_shape(120, 80)),
                        out=out, kpts_in=k, kpts_out=kk, out_h09=out2, kpts_out_h09=kk2)
    print("warp:", out.shape)

    # ---- blenders on 3 views of 120x80
    bimgs, borg = synth.make_stack(3, 120, 80, 40, 104)
    items, geom = synth.translation_blend_setup(borg, 120, 80)
    res = {}
    for lazy in (0, 1):
        for ordered in (0, 1):
            res[f"linear_lazy{lazy}_ord{ordered}"] = ref.blend(bimgs, items, geom, 0,
                                                               default_params(lazy_read=lazy, ordered_input=ordered))
    for bands in (1, 3, 5):
        res[f"multiband_{bands}"] = ref.blend(bimgs, items, geom, bands)
    np.savez_compressed(OUT / "blend_3x120x80.npz", input_sha=np.array(sha(*bimgs)), **res)
    print("blend:", {k: v.shape for k, v in res.items()})


if __name__ == "__main__":
    main()
