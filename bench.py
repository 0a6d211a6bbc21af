#!/usr/bin/env python
"""bench.py — SIFT + match + blend throughput of the hot path (BASELINE.json).

One "step" = one pass of the hot path over one synthetic stack of
BASELINE.json configs[1]: 13 ordered images 1500x1112 -> SIFT on every image,
the 13 adjacent-pair matches of linear_pairwise_match, and the LinearBlender
composite (reference defaults MULTIBAND 0, LAZY_READ 1; ORDERED_INPUT 1) with
generator-known homographies (RANSAC / bundle adjustment are host geometry
outside the hot path, SURVEY.md §8d).  Metric: megapixels of INPUT per second.

  python bench.py [--gpus N --steps K --warmup W]       our engine (one rank per GPU)
  python bench.py --impl reference [...]                 the reference's CPU path
  python bench.py --dump-outputs DIR [...]               also write what the last timed step
                                                         computed to DIR/*.npy (rank 0)

Prints ONE JSON line on rank 0 (contract in the task statement):
  value    : K steps with inputs resident in HBM (device-timed, max over ranks)
  e2e      : the same through the public API with pinned HOST inputs/outputs,
             H2D of the images and D2H of the mosaic + matches inside the timing.
             Host formats are the reference's file formats (8-bit pixels as read_img
             receives them, cropped 8-bit mosaic as write_rgb saves it; conversions
             and crop on the device, timed); e2e.mat32f_boundary is the same with
             f32 Mat32f buffers both ways (4x the PCIe bytes)
  roofline : dominant kernel, algorithmic bytes (SURVEY §8d) / event-timed duration
  cpu_baseline : oracle/_ref (the reference's own TUs, OpenMP) on this host
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

RESULT_OUT = sys.stdout
WORKLOAD = "ordered_13x1500x1112"
METRIC = "Mpixels/sec SIFT+match+blend"
UNIT = "Mpx/s"


# ----------------------------------------------------------------------------- workload
def make_workload(rank: int, bands: int):
    from openpano_b200 import synth
    from openpano_b200._abi import default_params
    from openpano_b200.synth import ordered_pairs

    cfg = dict(synth.CONFIGS[WORKLOAD])
    cfg["seed"] = cfg["seed"] + 1000 * rank          # each rank stitches its own stack (weak scaling)
    views, origins = synth.make_stack(**cfg)
    # The stack as the reference meets it: 8-bit decoded pixels (CImg<unsigned char>, imgio.cc:72)
    # turned into Mat32f by read_img's `(float)v / 255.0` (imgio.cc:79-81).  `pix` feeds the 8-bit
    # e2e boundary, `imgs` (bit-identical to read_img(pix)) every Mat32f leg and the CPU arms.
    pix = [(v * 255.0 + 0.5).astype(np.uint8) for v in views]
    imgs = [(p.astype(np.float32).astype(np.float64) / 255.0).astype(np.float32) for p in pix]
    items, geom = synth.translation_blend_setup(origins, cfg["w"], cfg["h"])
    params = default_params(ordered_input=1, multiband=bands)
    pairs = ordered_pairs(len(imgs))
    mpx = sum(im.shape[0] * im.shape[1] for im in imgs) / 1e6
    return imgs, pairs, items, geom, params, mpx, pix


def octave_dims(w, h, params):
    from tools.bench_configs import octave_dims as od
    return od(w, h, params)


def algorithmic_bytes(imgs, items, params, counts):
    """Per-launch algorithmic traffic of each kernel (SURVEY.md §8d model; tools/bench_configs.py)."""
    from tools.bench_configs import algorithmic_bytes as ab
    return ab([im.shape[:2] for im in imgs], items, params, counts, params.multiband)


DUMP_BYTES = 64_000_000
MOSAIC_SAMPLE_PIXELS = 1 << 20


def dump_outputs(out_dir, fs, match_total, mosaic):
    """What one step of the timed path hands its caller, so that two builds can be compared output
    for output on the same seeded workload: every image's keypoint coordinates (f64) and descriptors
    (f32), concatenated in image order, the per-image feature counts, the match total and the mosaic.
    The mosaic (7500x1112x3 f32, 100 MB) is written as a fixed, seeded sample of its pixels
    (mosaic_sample_index: the flat pixel indices, row-major) to keep the dump under DUMP_BYTES."""
    feats = [fs.download(i) for i in range(fs.n_images)]
    pixels = mosaic.reshape(-1, 3)
    pick = np.arange(len(pixels))
    if len(pixels) > MOSAIC_SAMPLE_PIXELS:
        pick = np.sort(np.random.default_rng(0).choice(len(pixels), MOSAIC_SAMPLE_PIXELS, replace=False))
    arrays = {"keypoints": np.concatenate([c for c, _ in feats]), "descriptors": np.concatenate([d for _, d in feats]),
              "feature_counts": np.array([len(c) for c, _ in feats], np.float64),
              "match_total": np.array([match_total], np.float64),
              "mosaic_sample": pixels[pick], "mosaic_sample_index": pick.astype(np.float64)}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"bench.py: outputs of one step take {total} bytes, more than the dump's {DUMP_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def config_dict(imgs, pairs, bands, world, extra=None):
    """The same keys on both arms (ours / reference), so the driver can compare them."""
    d = {"workload": WORKLOAD, "images": len(imgs), "image_wh": [imgs[0].shape[1], imgs[0].shape[0]],
         "pairs": len(pairs), "bands": bands, "blend": "linear" if bands == 0 else "multiband",
         "geometry": "generator-known homographies (flat projection)", "parallelism": f"dp{world}"}
    d.update(extra or {})
    return d


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.samples = []
        self._proc = None
        self._thr = None
        self._t0 = self._t1 = None

    def _run(self):
        # one long-lived `nvidia-smi -lms 100` (a fresh process per sample costs > 100 ms)
        for line in self._proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 7:
                self.samples.append((time.perf_counter(), parts))

    def launch(self):
        """Start the sampler process ahead of time; mark() / stop() bracket the timed region."""
        try:
            self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.FIELDS}",
                                           "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                          stderr=subprocess.DEVNULL, text=True)
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        except Exception:
            self._proc = None

    def start(self):
        if self._proc is None:
            self.launch()
        self._t0 = time.perf_counter()

    def stop(self):
        self._t1 = time.perf_counter()
        time.sleep(0.05)
        if self._proc is not None:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=3)
            except Exception:
                self._proc.kill()
        if self._thr:
            self._thr.join(timeout=3)
        inside = [p for (t, p) in self.samples if self._t0 <= t <= self._t1 + 0.03]
        self.samples = inside if inside else [p for (_, p) in self.samples[-3:]]
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- reference arm
def cpu_pass(checker, imgs, pairs, items, geom, bands, params):
    t = time.perf_counter()
    nf, nm, out, secs = checker.hotpath(imgs, pairs, items, geom, bands, params, use_flann=True)
    return time.perf_counter() - t, secs, int(nf.sum()), int(nm.sum())


def load_cpu_checker():
    from tests.checker import get_checker, have
    if have("ref_fast"):
        chk = get_checker("ref_fast")
        try:
            # every core this process may run on, whatever OMP_NUM_THREADS said when libgomp
            # was first initialised (another library may have done that long ago)
            chk.lib.omp_set_num_threads(len(os.sched_getaffinity(0)))
        except (AttributeError, OSError):
            pass
        return chk, "reference"
    if have("ref"):
        return get_checker("ref"), "reference"
    return get_checker("orc"), "port"


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 when it is unset; the reference's OpenMP
    path must get every host core (set before libgomp initialises)."""
    if os.environ.get("OMP_NUM_THREADS", "") in ("", "1") or "TORCHELASTIC_RUN_ID" in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)


def bind_to_gpu_numa_node(local_rank: int):
    """Best effort: run this rank (and allocate its pinned buffers) on the CPUs
    local to its GPU so H2D/D2H do not cross sockets."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        txt = Path(f"/sys/bus/pci/devices/{bus}/local_cpulist").read_text().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


def run_reference(args, rank, world):
    if rank != 0:
        return
    use_all_host_threads()
    imgs, pairs, items, geom, params, mpx, _ = make_workload(0, args.bands)
    chk, kind = load_cpu_checker()
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)                                 # the reference prints timers on stdout
    try:
        for _ in range(args.warmup):
            cpu_pass(chk, imgs, pairs, items, geom, args.bands, params)
        t0 = time.perf_counter()
        stage = np.zeros(3)
        for _ in range(args.steps):
            _, secs, nfeat, nmatch = cpu_pass(chk, imgs, pairs, items, geom, args.bands, params)
            stage += secs
        dt = (time.perf_counter() - t0) / args.steps
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    val = mpx / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(imgs, pairs, args.bands, args.gpus),
        "notes": {"matcher": "PairWiseMatcher (FLANN kd-forest)", "features": nfeat, "matches": nmatch,
                  "boundary": "Mat32f in / Mat32f out: read_img's, crop's and write_rgb's loops are NOT in the "
                              "timed region (less work than the CUDA arm's rgb8 e2e, which includes them; compare "
                              "with e2e.mat32f_value of the CUDA arm for the same boundary)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": chk.num_threads(), "kind": kind,
                         "sample": f"full {WORKLOAD} workload per step (host cores: {os.cpu_count()})",
                         "stage_ms": {"features": stage[0] / args.steps * 1e3, "match": stage[1] / args.steps * 1e3,
                                      "blend": stage[2] / args.steps * 1e3}},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=RESULT_OUT, flush=True)


# ----------------------------------------------------------------------------- our arm
SHARDED_TIMEOUT_S = 420          # watchdog of the N > 1 sharded legs (collectives: one failed rank would hang the rest)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bands", type=int, default=0, help="0 = LinearBlender (reference default), k = MultiBandBlender{k}")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lanes", type=int, default=3, help="concurrent stitch jobs per GPU in the e2e leg (StitchLanes)")
    ap.add_argument("--configs", default="all",
                    help="extra BASELINE.json configs measured in the same run at N=1 (comma list of 2mb,3,4,5; "
                         "'all'; 'none').  N>1 adds the sharded config-3 leg instead.")
    ap.add_argument("--sweep-sizes", default="10000,50000,100000,500000")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    # The contract is ONE JSON line on stdout.  Libraries chat on fd 1 (NCCL's version banner, the
    # reference's timers): keep a private handle to the real stdout for the line and point fd 1 at
    # stderr for everything else.
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the CUDA arm's outputs; the reference arm has none to write")
        args.warmup = min(args.warmup, 1)
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    from openpano_b200.capi import Engine
    from openpano_b200.stitcher import Stitcher

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa_cpus = bind_to_gpu_numa_node(local_rank)      # host threads + pinned buffers next to the GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    imgs, pairs, items, geom, params, mpx, pix = make_workload(rank, args.bands)
    shapes = [im.shape[:2] for im in imgs]
    out_w, out_h = max(it[2] for it in items), max(it[3] for it in items)

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        eng = Engine(local_rank, stream.cuda_stream)
        st = Stitcher(eng, params)
        # pinned host inputs / output for the e2e leg
        host = [torch.from_numpy(im).pin_memory() for im in imgs]
        host_out = torch.empty((out_h, out_w, 3), dtype=torch.float32).pin_memory()
        host_ptrs = [t.data_ptr() for t in host]
        h2d_bytes = sum(t.numel() * 4 for t in host)

        # ---- correctness guard + counts (untimed)
        st.upload(host_ptrs, shapes, (out_w, out_h))
        eng.sync()
        fs, matches = st.run_device(pairs, items, geom, args.bands, want_matches=True)
        counts = [fs.count(i) for i in range(len(imgs))]
        n_matches = sum(len(m) for m in matches)
        fs.free()
        if min(counts) == 0 or n_matches == 0:
            raise SystemExit("bench.py: degenerate workload (no features / matches)")

        # ---- value: inputs resident in HBM
        def step_device(keep=False):
            f, total = st.run_device(pairs, items, geom, args.bands, want_matches=False)
            if not keep:
                f.free()
            return f, total

        import gc
        gc.collect()
        gc.disable()                       # no collector pauses inside the timed regions
        for _ in range(args.warmup):
            step_device()
        torch.cuda.synchronize()
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.launch()
            time.sleep(0.3)                      # let nvidia-smi start sampling
            sampler.start()
        l0 = eng.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            last = step_device(keep=bool(args.dump_outputs) and i == args.steps - 1)
        e1.record(stream)
        torch.cuda.synchronize()
        barrier()
        launches = eng.launch_count() - l0
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs:
            if rank == 0:
                mosaic = np.empty((out_h, out_w, 3), np.float32)
                eng.dev_download(mosaic, st._d_out)          # the e2e legs below reuse the stitcher's canvas
                dump_outputs(args.dump_outputs, last[0], last[1], mosaic)
            last[0].free()
        exact_rows = eng.match_last_exact_rows()
        ms = e0.elapsed_time(e1)
        t_dev = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        ms_total = float(t_dev.item())
        ms_per_step = ms_total / args.steps
        value = world * mpx / (ms_per_step / 1e3)

        # ---- e2e: pinned host images in, host mosaic + matches out, every step.
        # (a) one job at a time: Stitcher.build() — the latency of a single stitch
        d2h_bytes = out_w * out_h * 3 * 4
        for _ in range(2):
            st.build(host_ptrs, shapes, pairs, items, geom, host_out.data_ptr(), args.bands)
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        nm_e2e = 0
        n_lat = max(3, min(args.steps, 10))
        for _ in range(n_lat):
            m = st.build(host_ptrs, shapes, pairs, items, geom, host_out.data_ptr(), args.bands)
            nm_e2e = sum(len(x) for x in m)
        torch.cuda.synchronize()
        e2e_latency = (time.perf_counter() - t0) / n_lat
        assert float(host_out[out_h // 2, out_w // 2, 0]) >= 0.0      # the mosaic really came back
        # (b) throughput: consecutive jobs pipelined (PipelinedStitcher): job i+1's H2D and
        # job i-1's D2H overlap job i's kernels; every step still uploads its own inputs
        # from pinned host memory and downloads its own mosaic + match lists.
        from openpano_b200.stitcher import PipelinedStitcher, unpack_rgb8_mosaic

        class Leg:
            """One e2e configuration, set up once and timed in several trials of `steps` jobs."""

            def __init__(self, rgb8, n_lanes):
                from openpano_b200.stitcher import StitchLanes
                self.rgb8, self.n_out = rgb8, 3 * n_lanes
                self.lanes = StitchLanes(local_rank, params, lanes=n_lanes, depth=3 if n_lanes == 1 else 2, rgb8=rgb8,
                                         crop=True)
                if rgb8:
                    self.src = [torch.from_numpy(p).pin_memory() for p in pix]
                    self.outs = [torch.empty(self.lanes.out_bytes((out_w, out_h)), dtype=torch.uint8).pin_memory()
                                 for _ in range(self.n_out)]
                else:
                    self.src = host
                    self.outs = [torch.empty_like(host_out).pin_memory() for _ in range(self.n_out)]
                self.ptrs = [t.data_ptr() for t in self.src]
                self.h2d = self.lanes.in_bytes(shapes)
                self.d2h = self.lanes.out_bytes((out_w, out_h)) + nm_e2e * 8 + len(imgs) * 8
                self.trials = []
                self.gaps = []        # per trial: the longest pause between two consecutive job completions (ms)
                self.lanes.map(self.jobs(2 * self.n_out))           # warm-up

            def jobs(self, n):
                return [(self.ptrs, shapes, (out_w, out_h), pairs, items, geom, self.outs[i % self.n_out].data_ptr(),
                         args.bands) for i in range(n)]

            def trial(self):
                torch.cuda.synchronize()
                barrier()
                t0 = time.perf_counter()
                res = self.lanes.map(self.jobs(args.steps))
                torch.cuda.synchronize()
                secs = time.perf_counter() - t0
                dt = np.diff(np.sort(np.array([t0] + list(self.lanes.done_times))))
                self.gaps.append(float(dt.max()) * 1e3 if len(dt) else 0.0)
                nm_pipe = sum(sum(len(x) for x in m) for m in res)
                assert nm_pipe == args.steps * nm_e2e, (nm_pipe, nm_e2e)      # every job returned the same matches
                last = self.outs[(args.steps - 1) % self.n_out]
                if self.rgb8:
                    rect, px = unpack_rgb8_mosaic(last.numpy(), (out_w, out_h))
                    assert rect[2] > out_w // 2 and rect[3] > out_h // 2 and int(px[rect[3] // 2, rect[2] // 2].max()) > 0
                else:
                    assert float(last[out_h // 2, out_w // 2, 0]) >= 0.0
                t = torch.tensor([secs], device="cuda")
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                self.trials.append(float(t.item()) / args.steps)

            def median(self):
                return float(np.median(self.trials))

        # headline: the reference's file formats at the boundary (8-bit pixels in, cropped 8-bit
        # mosaic out; conversions and crop on the device).  Beside it one lane, and the Mat32f
        # boundary.  The GPU box is shared: other tenants' PCIe traffic slows whole legs down for
        # seconds at a time (seen: 2.3 -> 5+ ms/job with identical kernel times), so every leg is
        # timed in E2E_TRIALS (9) trials of `steps` jobs, interleaved with the other legs, and the MEDIAN
        # trial is reported (all trials are in the JSON line).
        E2E_TRIALS = 9
        legs = {"lanes": Leg(True, args.lanes)}
        legs["one"] = Leg(True, 1) if args.lanes != 1 else legs["lanes"]
        legs["f32"] = Leg(False, 1)
        for _ in range(E2E_TRIALS):
            for key in ("lanes", "one", "f32"):
                if key == "one" and args.lanes == 1:
                    continue
                legs[key].trial()
        e2e_per_step, h2d_bytes, d2h_bytes = legs["lanes"].median(), legs["lanes"].h2d, legs["lanes"].d2h
        e2e_value = world * mpx / e2e_per_step
        one_lane_per_step = legs["one"].median()
        f32_per_step, f32_h2d, f32_d2h = legs["f32"].median(), legs["f32"].h2d, legs["f32"].d2h
        e2e_trials = {k: [round(x * 1e3, 3) for x in v.trials] for k, v in legs.items()}
        e2e_gaps = {k: [round(x, 2) for x in v.gaps] for k, v in legs.items()}
        for v in {id(v): v for v in legs.values()}.values():
            v.lanes.close()

        # ---- roofline of the dominant kernel (event-timed per launch, separate untimed pass)
        roof = None
        kernels = {}
        if rank == 0:
            st.upload(host_ptrs, shapes, (out_w, out_h))
            eng.sync()
            st._overlap = False                 # per-kernel times: every kernel of the step on the profiled context
            eng.profile(True)
            eng.profile_reset()
            PROF_STEPS = 5
            for _ in range(PROF_STEPS):
                step_device()
            prof = eng.profile_read()
            eng.profile(False)
            st._overlap = True
            ab = algorithmic_bytes(imgs, items, params, counts)
            peaks = {}
            pk = ROOT / "MEASURED_PEAKS.json"
            peak_src = "fallback"
            if pk.exists():
                peaks = json.loads(pk.read_text())
                peak_src = "measured"
            hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
            tf_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
            tot = sum(v[1] for v in prof.values())
            for name, (cnt, tms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
                avg = tms / max(cnt, 1)
                ent = {"launches_per_step": cnt / PROF_STEPS, "avg_ms": avg, "share": tms / tot if tot else 0}
                if name in ("k_match_top2", "k_tc_top2"):
                    flops = sum(2.0 * counts[i] * counts[j] * 128 for i, j in pairs)   # §8d: 2·N·M·128 per pair
                    ent.update(bound="tensor", achieved=flops / (avg * 1e-3) / 1e12, peak=tf_peak, unit="TFLOP/s")
                elif ab.get(name):
                    ent.update(bound="hbm", achieved=ab[name] / (avg * 1e-3) / 1e9, peak=hbm_peak, unit="GB/s")
                if "achieved" in ent:
                    ent["frac"] = ent["achieved"] / ent["peak"]
                kernels[name] = ent
            top = max(kernels, key=lambda k: kernels[k]["share"])
            t = kernels[top]
            # DRAM bytes per launch of that kernel from the committed `ncu --set full` capture of this
            # same workload (profiles/*_traffic.json, written by tools/ncu_summary.py); null if absent
            traffic, issue = None, None
            # captures are tagged r02a .. r02z, r02aa ..: shorter tags are older
            tr_files = sorted((ROOT / "profiles").glob("*_traffic.json"), key=lambda f: (len(f.name), f.name))
            if tr_files and not args.bands:
                ent = json.loads(tr_files[-1].read_text()).get(top, {})
                traffic = ent.get("dram_bytes_per_launch")
                wi = ent.get("warp_instructions_per_launch")
                if wi:
                    # issue-slot roofline: a kernel cannot finish before its warp instructions have gone through
                    # the 148 x 4 schedulers (one instruction per scheduler per cycle) at the SM clock seen in this run
                    sm_hz = float((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
                    floor_ms = wi / (148 * 4 * sm_hz) * 1e3
                    issue = {"warp_instructions": wi, "floor_ms": floor_ms, "frac": floor_ms / t["avg_ms"],
                             "source": tr_files[-1].name}
            roof = {"kernel": top, "bound": t.get("bound"), "achieved": t.get("achieved"), "peak": t.get("peak"),
                    "unit": t.get("unit"), "frac": t.get("frac"), "traffic": traffic, "peak_source": peak_src,
                    "share_of_step": t["share"], "avg_ms": t["avg_ms"], "issue": issue}
            # the dominant kernel (k_descriptor) is issue-bound: its §8d bytes are only its outputs, so its
            # HBM fraction says little.  Beside it, the largest kernel that IS bandwidth-limited.
            bw = [k for k, v in kernels.items() if v.get("bound") == "hbm" and (v.get("frac") or 0) >= 0.05]
            if bw:
                k2 = max(bw, key=lambda k: kernels[k]["share"])
                v2 = kernels[k2]
                roof["largest_bandwidth_bound_kernel"] = {
                    "kernel": k2, "achieved": v2["achieved"], "peak": v2["peak"], "unit": v2["unit"], "frac": v2["frac"],
                    "share_of_step": v2["share"], "avg_ms": v2["avg_ms"]}

        # ---- CPU baseline (rank 0, N == 1): the reference's own TUs on this host
        cpu = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                os.sched_setaffinity(0, all_cpus)          # the CPU arm gets every core again
                use_all_host_threads()
                chk, kind = load_cpu_checker()
                devnull = os.open(os.devnull, os.O_WRONLY)
                saved = os.dup(1)
                os.dup2(devnull, 1)
                try:
                    dt, secs, _, _ = cpu_pass(chk, imgs, pairs, items, geom, args.bands, params)
                finally:
                    os.dup2(saved, 1)
                    os.close(devnull)
                cpu = {"value": mpx / dt, "unit": UNIT, "cores": chk.num_threads(), "kind": kind,
                       "sample": f"one full pass of {WORKLOAD} ({dt:.2f} s; host has {os.cpu_count()} cores)",
                       "stage_ms": {"features": secs[0] * 1e3, "match": secs[1] * 1e3, "blend": secs[2] * 1e3}}
            except Exception as ex:  # the checker is optional equipment on the box
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(ex)}

        # ---- the other BASELINE.json configs (N == 1) / the sharded path (N > 1), same run, same engine
        configs, sharded = None, None
        st.release_images()
        want = [] if args.configs == "none" else (["1", "2mb", "3", "4", "5"] if args.configs == "all" else args.configs.split(","))
        if world == 1 and want:
            from openpano_b200 import synth as _synth
            from openpano_b200._abi import default_params as _dp
            from tools import bench_configs as bc
            loader = None if args.no_cpu_baseline else load_cpu_checker
            use_all_host_threads()
            configs = {}

            def leg(key, fn):
                try:
                    configs[key] = fn()
                except Exception as ex:      # one failing leg must not take the headline line down
                    configs[key] = {"error": repr(ex)}
            if "1" in want:
                leg("config1_cmu0_cylinder", lambda: bc.run_cylinder(
                    eng, "cmu0_8x600x400, cylinder mode: SIFT + 7 adjacent matches + cylinder warp + linear blend",
                    "cmu0_8x600x400", _dp(ordered_input=1), cpu_loader=loader, all_cpus=all_cpus))
            if "2mb" in want:
                leg("config2_multiband5", lambda: bc.run_stack(
                    eng, "ordered_13x1500x1112, MULTIBAND 5", "ordered_13x1500x1112", _synth.ordered_pairs, 5,
                    _dp(ordered_input=1, multiband=5), cpu_loader=loader, all_cpus=all_cpus))
            if "3" in want:
                leg("config3_unordered38", lambda: bc.run_stack(
                    eng, "unordered_38x1300x867, all 703 pairs, linear blend", "unordered_38x1300x867", _synth.all_pairs, 0,
                    _dp(), cpu_loader=loader, all_cpus=all_cpus))
            if "4" in want:
                leg("config4_match_sweep", lambda: bc.run_sweep(eng, [int(x) for x in args.sweep_sizes.split(",")], _dp()))
            if "5" in want:
                leg("config5_uav64_multiband5", lambda: bc.run_stack(
                    eng, "uav_64x4000x3000, MULTIBAND 5, LAZY_READ 0, MAX_OUTPUT_SIZE 8000", "uav_64x4000x3000",
                    lambda n: [(i, i + 1) for i in range(n - 1)], 5, _dp(multiband=5, lazy_read=0), steps=3,
                    max_output=8000, cpu_views=16, cpu_loader=loader, all_cpus=all_cpus))

        def build_line(sharded):
            return {
                "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config_dict(imgs, pairs, args.bands, world),
                "notes": {"cpu_affinity_cpus": numa_cpus,
                          "l2_policy": "inputs_exceed_l2 (260 MB of images + 0.9 GB pyramid arena per step)",
                          "features": int(sum(counts)), "matches": int(n_matches),
                          "match_rows_rescanned_exactly": int(exact_rows)},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes),
                        "d2h_bytes_per_step": int(d2h_bytes), "ms_per_step": e2e_per_step * 1e3,
                        "mode": f"StitchLanes: {args.lanes} concurrent pipelined jobs per GPU (one host thread each); every job "
                                "uploads its own images and downloads its own mosaic + match lists",
                        "one_lane": {"value": world * mpx / one_lane_per_step, "ms_per_step": one_lane_per_step * 1e3},
                        "reported": f"median of {E2E_TRIALS} trials of {args.steps} jobs each (trials interleaved across legs)",
                        "trials_ms_per_step": e2e_trials,
                        "best_trial_ms_per_step": min(e2e_trials["lanes"]),
                        "boundary": "rgb8: decoded 8-bit pixels in (read_img's input), crop()+write_rgb 8-bit mosaic out; "
                                    "u8<->f32 conversions and crop run on the device inside the timed region",
                        "mat32f_boundary": {"value": world * mpx / f32_per_step, "ms_per_step": f32_per_step * 1e3,
                                            "h2d_bytes_per_step": int(f32_h2d), "d2h_bytes_per_step": int(f32_d2h)},
                        "single_job_latency_ms_mat32f": e2e_latency * 1e3,
                        "single_job_value_mat32f": world * mpx / e2e_latency,
                        # the same figures as flat scalars (nested objects get dropped by some JSON consumers)
                        "one_lane_ms_per_step": one_lane_per_step * 1e3, "one_lane_value": world * mpx / one_lane_per_step,
                        "mat32f_ms_per_step": f32_per_step * 1e3, "mat32f_value": world * mpx / f32_per_step,
                        "mat32f_h2d_bytes_per_step": int(f32_h2d), "mat32f_d2h_bytes_per_step": int(f32_d2h),
                        "single_job_ms": e2e_latency * 1e3, "single_job_value": world * mpx / e2e_latency,
                        "lanes_trials_ms": e2e_trials["lanes"], "lanes_worst_trial_ms": max(e2e_trials["lanes"]),
                        # a slow trial is ONE long pause between two job completions (a descheduled host thread /
                        # another tenant's PCIe burst on the shared box), not a uniformly slower pipeline:
                        "longest_pause_between_jobs_ms": e2e_gaps},
                "gpu_launches": int(launches * world),
                "roofline": roof,
                "cpu_baseline": cpu,
                "kernels": kernels,
                "configs": configs,
                "sharded": sharded,
            }

        if world > 1:
            # The sharded legs are collectives over all ranks: if one rank fails inside them the others would
            # wait for ever.  A watchdog prints the line without them (rank 0) and leaves, so the headline survives.
            import threading

            def _bail():
                if rank == 0:
                    print(json.dumps(build_line({"error": f"sharded legs did not finish within {SHARDED_TIMEOUT_S} s"})),
                          file=RESULT_OUT, flush=True)
                os._exit(0)
            dog = threading.Timer(SHARDED_TIMEOUT_S, _bail)
            dog.daemon = True
            dog.start()
            from openpano_b200._abi import default_params as _dp
            from tools import bench_configs as bc
            try:
                sharded = bc.run_sharded(eng, rank, world, _dp())
            except Exception as ex:
                sharded = {"error": repr(ex)}
            try:
                sweep = bc.run_sharded_sweep(eng, rank, world, _dp())
            except Exception as ex:
                sweep = {"error": repr(ex)}
            dog.cancel()
            if rank == 0 and isinstance(sharded, dict):
                sharded["match_sweep_100k_row_sharded"] = sweep

        line = build_line(sharded) if rank == 0 else None
        st.close()
        eng.close()

    if rank == 0:
        print(json.dumps(line), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
