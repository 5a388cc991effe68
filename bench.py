#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 backend for yuki's per-pixel rendering hot path.

Metric (BASELINE.json): Msamples/s (and Mrays/s) of the path-traced Cornell box, config[1]:
1024x1024, Path integrator with Russian roulette (max_depth 8), 1024 spp stratified 32x32, on N B200s.
A "step" is one complete render of that film. At N > 1 the reference's spiral tile list is interleaved over the
ranks (tile i -> rank i mod N, no data-path collective) and the film is summed to rank 0 with one NCCL reduce.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference      # the CPU restatement of yuki's renderer on the host cores

`value` is measured with the scene and the film resident in HBM (CUDA events on the renderer's stream, max over
ranks). `e2e` is the same metric through the C-ABI call with host buffers: scene upload, tile/job upload and the
film read-back are all inside its timed region.

The line also carries `large_scene`: BASELINE.json configs[4]'s geometry (the 10 M-triangle scene at 3840x2160, Path 8) at
64 spp, run by ALL ranks (tiles interleaved, film reduced to rank 0) — the workload whose BVH cannot live in the caches,
with its own clocks, roofline (algorithmic bytes next to the ncu-measured DRAM / L2 bytes per launch) and per-rank busy
times. Films are checked against stored digests (tests/golden/bench_film_digests.json) outside the timed regions.

`--dump-outputs DIR` writes the headline leg's film and counters of its last timed step as DIR/*.npy (dump_outputs()): the
inputs are fixed, so two builds' dumps of the same command can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# stdout carries the one JSON line and nothing else: whatever libraries write to file descriptor 1 while the bench runs
# (NCCL's version banner under NCCL_DEBUG=VERSION, NCCL_DEBUG=INFO output) is sent to stderr; emit() writes the line to
# the real stdout.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
_REAL_STDOUT = None  # main() moves file descriptor 1 aside


def emit(line: dict):
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        print(json.dumps(line), flush=True)
    else:
        os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

from yuki_b200 import desc as D  # noqa: E402

WORKLOAD = "cornell-box 1024x1024, Path max_depth 8 (Russian roulette after 3 bounces), 1024 spp stratified 32x32"
RES = (1024, 1024)
SPP_NX = SPP_NY = 32
MAX_DEPTH = 8
CPU_SAMPLE_SPP = 32  # bounded CPU sample: sample indices 0..31 of every pixel (accumulate-mode tiles), ~10 s on 15 host threads
SCENE = "cornell"
# The device-resident leg (`value`, `roofline`) runs on one pipe so that the CUDA-event time of a kernel launch is the kernel's
# own; the end-to-end leg (`e2e`) makes the call a user makes, with the library's default of two overlapping pipes.
VALUE_PIPES = 1


def select_workload(name, spp_side):
    """The default (and the driver's) workload is BASELINE.json configs[1]. `--workload c5` switches to configs[4] (the
    10 M-triangle scene at 3840x2160, Path 8, 64x64 = 4096 spp) for scaling studies; `--spp-side` shortens either."""
    global WORKLOAD, RES, SPP_NX, SPP_NY, SCENE, CPU_SAMPLE_SPP, VALUE_PIPES
    if name == "c5":
        VALUE_PIPES = 0  # scaling studies: the library's default (two pipes) on every leg
        SCENE, RES, SPP_NX, SPP_NY = "terrain", (3840, 2160), 64, 64
        CPU_SAMPLE_SPP = 1  # one sample index of every pixel: 8.3 M samples
        WORKLOAD = "10M-triangle terrain + material objects 3840x2160, Path max_depth 8, 4096 spp stratified 64x64"
    if spp_side:
        SPP_NX = SPP_NY = spp_side
        CPU_SAMPLE_SPP = min(CPU_SAMPLE_SPP, spp_side * spp_side)
        WORKLOAD = WORKLOAD.split(",")[0] + f", Path max_depth 8, {spp_side * spp_side} spp stratified {spp_side}x{spp_side} (--spp-side override)"


def workload(xf):
    from yuki_b200 import scenes
    scene, cam = scenes.terrain_room(xf) if SCENE == "terrain" else scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings(RES, 16)
    sampler = D.SamplerType.stratified(SPP_NX, SPP_NY, jitter=True)
    integ = D.IntegratorType.path(MAX_DEPTH)
    return scene, cam, film, sampler, integ


def kernel_source_hash():
    """sha256 over the CUDA sources the kernels are compiled from: what a committed ncu capture is valid for."""
    import hashlib
    h = hashlib.sha256()
    src = os.path.join(ROOT, "yuki_b200", "csrc")
    for name in sorted(os.listdir(src)):
        # the wavefront kernels, their device headers and the driver that sizes their grids (not the loaders, the display passes
        # or the device-group layer, none of which can change what the profiled kernel does)
        if name.endswith(".cuh") or name in ("render.cu", "yk_libm.h", "yk_fastdiv.h"):
            with open(os.path.join(src, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def ncu_traffic(workload):
    """DRAM and L2 bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this command
    (profiles/<round>/traffic.json, written by scripts/gpu_bench_profile.sh + scripts/ncu_traffic.py). A capture is only
    reported when it was taken from the kernels that are running now (its kernel_hash equals the hash of today's sources):
    a stale capture yields None and says so."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    for rnd in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        f = os.path.join(pdir, rnd, "traffic.json")
        if os.path.exists(f):
            with open(f) as fh:
                best = json.load(fh)
    entry = (best or {}).get(workload) if isinstance((best or {}).get(workload), dict) else None
    if entry is None:
        return {"dram_bytes_per_launch": None, "l2_bytes_per_launch": None, "traffic_state": "no capture for this workload"}
    now = kernel_source_hash()
    if entry.get("kernel_hash") != now:
        return {"dram_bytes_per_launch": None, "l2_bytes_per_launch": None,
                "traffic_state": f"stale: captured at kernel_hash {entry.get('kernel_hash')} (commit {entry.get('commit')}), sources are {now}"}
    return {"dram_bytes_per_launch": entry.get("dram_bytes_per_launch"), "l2_bytes_per_launch": entry.get("l2_bytes_per_launch"),
            "traffic_state": "current", "traffic_commit": entry.get("commit"), "traffic_kernel_hash": now, "traffic_source": entry.get("source"),
            "ncu": entry.get("ncu")}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._t.start()

    def stop(self):
        self._stop.set()
        self._t.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = []
        for name, col in (("hw_slowdown", 2), ("hw_thermal_slowdown", 3), ("sw_thermal_slowdown", 4), ("sw_power_cap", 5)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


CPU_TILES = 128        # bounded CPU sample of the headline workload: ~128 tiles spread evenly over the spiral list, all of their samples


def cpu_sample_tiles(film, first_sample=0, n=CPU_SAMPLE_SPP):
    """Accumulate-mode tile list covering sample indices [first, first+n) of every pixel (render_manager.rs:135-143)."""
    from oracle import oracle as O
    base = O.film_tiles(film)
    out = []
    for s in range(first_sample, first_sample + n):
        t = base.copy()
        t["sample"] = s
        out.append(t)
    return np.concatenate(out)


def time_cpu(threads=0, first_sample=0, step=0):
    """Times the CPU restatement of yuki's renderer (oracle) on a bounded sample of the workload. Headline workload: the way a
    headless 1024-spp render runs in the reference — non-accumulating, one task = one 16x16 tile with all of its samples
    (render_manager.rs:135-143 replicates tiles per sample only for accumulating films) — on ~CPU_TILES tiles spread evenly over
    the spiral list (a whole number per worker thread; ~34 M samples, ~10 s on 15 threads). Measured on this container's 7 worker threads the
    accumulate-mode micro-tasks round 1 timed are ~10 % slower per sample (0.90 vs 1.00 Msamples/s): queue and film mutex
    per 256 samples. `--workload c5` keeps one accumulate-mode sample index of every pixel (a 4096-spp tile is 1 M samples)."""
    from oracle import oracle as O
    scene, cam, film, sampler, integ = workload(O.transforms)
    osc = O.OracleScene(scene)
    if SCENE == "cornell":
        # a whole number of tiles per worker (the reference runs hardware_concurrency() - 1 of them), so that the sample's tail does not
        # penalise the CPU arm: a full render has 4096 tiles and no such tail
        workers = threads or max(1, (os.cpu_count() or 2) - 1)
        all_tiles = O.film_tiles(film)
        n = min(len(all_tiles), workers * max(1, round(CPU_TILES / workers)))
        pick = (np.arange(n) * len(all_tiles) // n + step) % len(all_tiles)
        tiles = np.ascontiguousarray(all_tiles[pick])
        _, _, st = osc.render(cam, film, sampler, integ, tiles=tiles, threads=threads)
        return st
    acc = D.FilmSettings(film.res, film.tile_dim, accumulate=True)
    tiles = cpu_sample_tiles(film, first_sample)
    _, _, st = osc.render(cam, acc, sampler, integ, tiles=tiles, threads=threads)
    return st


def cpu_sample_text(samples):
    if SCENE == "cornell":
        return (f"{samples // (256 * SPP_NX * SPP_NY)} 16x16 tiles spread evenly over the spiral list with all {SPP_NX * SPP_NY} samples of their pixels, "
                f"non-accumulating like a headless render of the reference ({samples} samples), same scene/sampler/integrator")
    return f"{CPU_SAMPLE_SPP} of the {SPP_NX * SPP_NY} samples of every pixel ({samples} samples), same scene/sampler/integrator"


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path. The Rust renderer cannot be built in
    this image (no cargo/rustc, DESIGN.md), so this is the line-by-line C++ restatement (oracle/, kind "port") with the
    reference's threading model: hardware_concurrency()-1 workers popping 16x16 spiral tiles from one queue."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.warmup > 0:
        time_cpu(first_sample=0)  # one untimed pass warms caches/page tables; repeating it W times would only burn minutes
    t_total, samples, rays, shadow, threads = 0.0, 0, 0, 0, 0
    for k in range(args.steps):
        st = time_cpu(first_sample=(k * CPU_SAMPLE_SPP) % max(1, SPP_NX * SPP_NY - CPU_SAMPLE_SPP), step=k)
        t_total += st.seconds
        samples += st.samples
        rays += st.ray_count
        shadow += st.shadow_rays
        threads = st.threads
    v = samples / t_total / 1e6
    sample = cpu_sample_text(samples // max(args.steps, 1)) + " per step"
    line = {
        "impl": "reference", "metric": "Msamples/s", "value": v, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "each step is a bounded sample of the workload; throughput is per sample"},
        "mrays_per_s": rays / t_total / 1e6, "mrays_per_s_total": (rays + shadow) / t_total / 1e6,
        "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


C5_SPP_SIDE = 8          # the large-scene leg: 8 x 8 = 64 spp of configs[4]'s 4096 (at 16 spp an 8-rank step is one 20 ms batch per rank:
                         # per-launch tails and the hash-table set-up, which the real config amortises over 4096 spp, cost 10 % there)
C5_STEPS, C5_WARMUP = 5, 2
C5_DIGEST = f"c5_{C5_SPP_SIDE * C5_SPP_SIDE}spp"
DIGESTS = os.path.join(ROOT, "tests", "golden", "bench_film_digests.json")


def film_digest(t):
    """sha256 of a film tensor's bytes. Renders are bit-reproducible (DESIGN.md: no result depends on the processing order)
    and tiles are disjoint, so the digest is the same at every N."""
    import hashlib
    return hashlib.sha256(t.detach().cpu().numpy().tobytes()).hexdigest()[:32]


def check_digest(key, digest, update):
    """Compares with the stored digest of this workload (tests/golden/bench_film_digests.json). Returns 'ok' / 'written' /
    'absent'; raises on a mismatch — a bench that timed the wrong picture must not print a line."""
    stored = {}
    if os.path.exists(DIGESTS):
        with open(DIGESTS) as f:
            stored = json.load(f)
    if update:
        stored[key] = digest
        with open(DIGESTS, "w") as f:
            json.dump(stored, f, indent=1, sort_keys=True)
        return "written"
    if key not in stored:
        return "absent"
    if stored[key] != digest:
        raise SystemExit(f"bench.py: film digest of '{key}' is {digest}, expected {stored[key]} (tests/golden/bench_film_digests.json)")
    return "ok"


DUMP_COUNTERS = ("ray_count", "shadow_rays", "samples", "closest_nodes", "closest_tris", "any_nodes", "any_tris")
DUMP_LIMIT = 64 << 20    # bytes, all files of one --dump-outputs together
DUMP_SAMPLE_PIXELS = 1 << 20


def dump_outputs(directory, film, counters):
    """--dump-outputs: what the timed leg's caller receives after its last timed step, so that two builds' runs with the same
    arguments can be compared output for output. film.npy is the (height, width, 3) float32 film; a film larger than the budget
    (--workload c5) is replaced by film_sample.npy, the pixels at a fixed seeded choice of DUMP_SAMPLE_PIXELS flat pixel indices
    (film_sample_index.npy). counters.npy holds the step's DUMP_COUNTERS in that order as float64 (exact below 2**53)."""
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "counters.npy"), np.asarray(counters, np.float64))
    film = np.asarray(film, np.float32)
    if film.nbytes <= DUMP_LIMIT // 2:
        np.save(os.path.join(directory, "film.npy"), film)
        return
    pixels = film.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(0).choice(len(pixels), DUMP_SAMPLE_PIXELS, replace=False))
    np.save(os.path.join(directory, "film_sample.npy"), pixels[idx])
    np.save(os.path.join(directory, "film_sample_index.npy"), idx.astype(np.float64))


def shared_host_scene(api, scene, world, local, tag, big):
    """One host BVH build per node: local rank 0 builds and (for the 10 M-triangle scene, `big`) leaves the flattened arrays under
    /dev/shm; the other ranks map them (api.HostScene.save / load) instead of repeating the 6 s build N times on contended cores.
    Returns (host scene, clean-up function to call once every rank holds its device copy)."""
    import torch.distributed as dist
    if world == 1 or not big:
        return api.HostScene(scene), (lambda: None)
    base = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    share_dir = os.path.join(base, f"yuki_b200_{tag}_{os.environ.get('MASTER_PORT', '0')}_{kernel_source_hash()}")
    host = None
    if local == 0:
        host = api.HostScene(scene)
        host.save(share_dir)
    dist.barrier()
    if local != 0:
        host = api.HostScene.load(share_dir)

    def done():
        dist.barrier()
        if local == 0:
            import shutil
            shutil.rmtree(share_dir, ignore_errors=True)
    return host, done


def large_scene_leg(args, api, capi, xf, ctx, stream, rank, world, local, peak):
    """BASELINE.json configs[4]'s geometry — the 10 M-triangle terrain + material objects at 3840x2160, Path max_depth 8 — at
    64 spp, on every rank: spiral tiles interleaved over the ranks, the scene built and uploaded once per rank OUTSIDE the
    timed region, the film summed to rank 0 (NCCL) inside it. Timed like the main leg (barrier + synchronize on both sides,
    CUDA events, max over ranks, L2 flushed between steps). Then, on one pipe (exclusive kernel times), the closest-hit
    kernel's roofline on this scene: its BVH (554 MB of records + 480 MB of triangles) cannot live in the 126 MB L2."""
    import torch
    import torch.distributed as dist
    from yuki_b200 import scenes
    t0 = time.perf_counter()
    scene, cam = scenes.terrain_room(xf)
    host, shared_done = shared_host_scene(api, scene, world, local, "c5leg", True)
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    dev = api.Scene(ctx, scene, host=host)
    t_upload = time.perf_counter() - t0
    shared_done()
    rn = api.Renderer(ctx)
    film = D.FilmSettings((3840, 2160), 16)
    sampler, integ = D.SamplerType.stratified(C5_SPP_SIDE, C5_SPP_SIDE, jitter=True), D.IntegratorType.path(MAX_DEPTH)
    all_tiles = api.film_tiles(film)
    my_tiles = np.ascontiguousarray(all_tiles[rank::world])
    n_pix = film.res[0] * film.res[1]
    total_samples = n_pix * sampler.samples_per_pixel()
    with torch.cuda.stream(stream):
        d_film = torch.zeros(n_pix * 3, dtype=torch.float32, device="cuda")
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

        def step(pipes=0):
            flush.zero_()
            d_film.zero_()
            r = rn.render(dev, cam, film, sampler, integ, tiles=my_tiles, device_film_ptr=d_film.data_ptr(), pipes=pipes)
            if world > 1:
                dist.reduce(d_film, dst=0, op=dist.ReduceOp.SUM)
            return r.stats

        for _ in range(C5_WARMUP):
            step()
        torch.cuda.synchronize()
        digest_state = check_digest(C5_DIGEST, film_digest(d_film), args.write_digests) if rank == 0 else None
        if world > 1:
            dist.barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        busy_ms, rays, shadow, launches = 0.0, 0, 0, 0
        for _ in range(C5_STEPS):
            st = step()
            busy_ms += st.device_ms; rays += st.ray_count; shadow += st.shadow_rays; launches += st.kernel_launches
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clk = clocks.stop() if rank == 0 else None
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        counts = torch.tensor([rays, shadow, launches], dtype=torch.float64, device="cuda")
        per_rank = torch.zeros(world, dtype=torch.float64, device="cuda")
        per_rank[rank] = busy_ms / C5_STEPS
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(counts, op=dist.ReduceOp.SUM)
            dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
        ms_total = float(ms.item())
        # roofline pass: rank 0, its own tiles, one pipe
        roof = None
        if rank == 0:
            cms, nodes, tris, r_rays, cl = 0.0, 0, 0, 0, 0
            dms = 0.0
            for _ in range(3):
                st = step(pipes=1) if world == 1 else rn.render(dev, cam, film, sampler, integ, tiles=my_tiles, device_film_ptr=d_film.data_ptr(), pipes=1).stats
                cms += st.trace_closest_ms; nodes += st.closest_nodes; tris += st.closest_tris; r_rays += st.ray_count
                cl += st.trace_closest_launches; dms += st.device_ms
            alg = 32 * nodes + 36 * tris
            achieved = alg / (max(cms, 1e-9) / 1e3) / 1e9
            tr = ncu_traffic("c5")
            roof = {"bound": "latency/issue", "roofline_axis": "hbm", "kernel": "k_trace_closest", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "algorithmic_bytes_per_launch": alg / max(cl, 1), "avg_launch_ms": cms / max(cl, 1), "launches": cl,
                    "share_of_step": cms / max(dms, 1e-9), "nodes_per_ray": nodes / max(r_rays, 1), "shape_tests_per_ray": tris / max(r_rays, 1),
                    "dram_bytes_per_launch": tr["dram_bytes_per_launch"], "l2_bytes_per_launch": tr["l2_bytes_per_launch"],
                    "traffic": tr["dram_bytes_per_launch"], "traffic_state": tr["traffic_state"], "traffic_commit": tr.get("traffic_commit"),
                    "ncu": tr.get("ncu"),
                    "note": "achieved = (32 B x node visits + 36 B x shape tests) / CUDA-event time of the closest-hit launches, one pipe, rank 0's tiles. "
                            "ncu on this scene: DRAM 4-6 % of peak, L1 hit 43-57 %, L2 hit 62-65 %, 16-17.5 of 32 lanes, issue-active 53-63 %, "
                            "long-scoreboard 3-6.5 warps per issue, L1TEX pipe 68-80 % (profiles/r02): the walk is bound by the load pipe, dependent-load latency and issue slots, "
                            "most algorithmic bytes are served by L1/L2, so frac is a throughput in the roofline's unit, not DRAM utilisation"}
        if world > 1:
            dist.barrier()
    n_tris, n_nodes = dev.host.n_tris, dev.host.n_nodes
    dev.close()
    host.close()
    if rank != 0:
        return None
    s = ms_total / 1e3
    return {"workload": f"configs[4] geometry: 10M-triangle terrain + material objects 3840x2160, Path max_depth 8, {C5_SPP_SIDE * C5_SPP_SIDE} spp "
                        f"stratified {C5_SPP_SIDE}x{C5_SPP_SIDE}, spiral tiles interleaved over {world} rank(s), film summed to rank 0",
            "triangles": n_tris, "bvh_nodes": n_nodes, "host_build_s": t_build, "upload_s": t_upload, "steps": C5_STEPS, "warmup": C5_WARMUP,
            "msamples_per_s": total_samples * C5_STEPS / s / 1e6, "c5_msamples_per_s": total_samples * C5_STEPS / s / 1e6,
            "ms_per_step": ms_total / C5_STEPS, "mrays_per_s": float(counts[0].item()) / s / 1e6,
            "mrays_per_s_total": float((counts[0] + counts[1]).item()) / s / 1e6, "gpu_launches": int(counts[2].item()),
            "per_rank_device_ms": [float(v) for v in per_rank.tolist()], "clocks": clk, "film_digest": digest_state,
            "pipes": "library default (two) for msamples_per_s; one for the roofline pass", "roofline": roof}


def published_config_leg(api, xf, ctx):
    """The one configuration the reference publishes a number for (BASELINE.md §1): its README screenshot — Scene::cornell()
    (37 shapes), 1920x1080, Path max_depth 10, indirect clamp 2.0, Stratified 32x32, tile 32 — "272.10 s, 20.47 Mrays/s"
    (closest-hit rays / wall time, app/window.rs:907-916) on the author's CPU. Rendered here end to end (host film out) with the
    library defaults, after one warm-up; tests/test_screenshot_pin.py checks the same render against the screenshot itself."""
    from yuki_b200 import scenes
    fx_path = os.path.join(ROOT, "tests", "golden", "reference_screenshot_regions.json")
    with open(fx_path) as f:
        fx = json.load(f)
    st = fx["settings"]
    scene, _ = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_SAH, back_wall_albedo=(0.85, 0.85, 0.80))
    cam = D.CameraParameters(tuple(st["camera_position"]), tuple(st["camera_target"]), fov_axis=D.FOV_X, fov_deg=st["fov_x_deg"])
    film = D.FilmSettings(tuple(fx["film"]), st["tile_dim"])
    sampler, integ = D.SamplerType.stratified(32, 32, jitter=True), D.IntegratorType.path(st["max_depth"], indirect_clamp=st["indirect_clamp"])
    dev = api.Scene(ctx, scene)
    rn = api.Renderer(ctx)
    out = np.zeros((film.res[1], film.res[0], 3), np.float32)
    rn.render(dev, cam, film, sampler, integ, film_out=out)
    t0 = time.perf_counter()
    r = rn.render(dev, cam, film, sampler, integ, film_out=out)
    sec = time.perf_counter() - t0
    dev.close()
    pub = fx["published"]
    mrays = r.stats.ray_count / sec / 1e6
    return {"workload": "the reference's README screenshot: Scene::cornell() 1920x1080, Path max_depth 10, indirect clamp 2.0, 1024 spp stratified 32x32",
            "seconds": sec, "msamples_per_s": r.stats.samples / sec / 1e6, "mrays_per_s": mrays, "rays_per_sample": r.stats.ray_count / r.stats.samples,
            "published": {"seconds": pub["render_seconds"], "mrays_per_s": pub["mrays_per_s"], "rays_per_sample": pub["mrays_per_s"] * 1e6 * pub["render_seconds"] / r.stats.samples,
                          "hardware": "the author's CPU (not stated; sampling/mod.rs:92-96 mentions a Ryzen 5900X)", "source": "screenshot.png via readme.md:3"},
            "vs_published": mrays / pub["mrays_per_s"], "timing": "host clock around the blocking call, host film out, one GPU"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from yuki_b200 import api, capi, transforms as xf

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the backend has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    scene, cam, film, sampler, integ = workload(xf)
    ctx = api.Context(local)
    stream = torch.cuda.ExternalStream(capi.lib().yk_context_stream(ctx._h), device=torch.device("cuda", local))
    host_scene, shared_done = shared_host_scene(api, scene, world, local, "main", SCENE != "cornell")
    dev = api.Scene(ctx, scene, host=host_scene)
    shared_done()
    rn = api.Renderer(ctx)
    all_tiles = api.film_tiles(film)
    my_tiles = np.ascontiguousarray(all_tiles[rank::world])  # spiral order interleaved over ranks (render_manager.rs:206-210 TODO)
    n_pix = film.res[0] * film.res[1]
    spp = sampler.samples_per_pixel()
    total_samples = n_pix * spp

    with torch.cuda.stream(stream):
        d_film = torch.zeros(n_pix * 3, dtype=torch.float32, device="cuda")
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

        def step():
            flush.zero_()
            d_film.zero_()
            r = rn.render(dev, cam, film, sampler, integ, tiles=my_tiles, device_film_ptr=d_film.data_ptr(), pipes=VALUE_PIPES)
            if world > 1:
                dist.reduce(d_film, dst=0, op=dist.ReduceOp.SUM)  # tiles are disjoint: sum == gather, bit-exact
            return r.stats

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        # the film the timed steps produce (every step renders the same picture), checked outside the timed region
        digest_state = None
        if rank == 0 and args.warmup > 0 and not args.spp_side:
            digest_state = check_digest("c2_1024spp" if SCENE == "cornell" else "c5_4096spp", film_digest(d_film), args.write_digests)
        if world > 1:
            dist.barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        agg = {"ray_count": 0, "shadow_rays": 0, "closest_nodes": 0, "closest_tris": 0, "trace_closest_ms": 0.0, "trace_any_ms": 0.0,
               "shade_ms": 0.0, "kernel_launches": 0, "trace_closest_launches": 0, "any_nodes": 0, "any_tris": 0}
        for _ in range(args.steps):
            st = step()
            for k in agg:
                agg[k] += getattr(st, k)
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clk = clocks.stop() if rank == 0 else None
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        counts = torch.tensor([agg["ray_count"], agg["shadow_rays"], agg["kernel_launches"]], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        ms_total = float(ms.item())
        value = total_samples * args.steps / (ms_total / 1e3) / 1e6
        if args.dump_outputs:  # d_film and st hold the last timed step's film and counters
            last = torch.tensor([getattr(st, k) for k in DUMP_COUNTERS], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.reduce(last, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                dump_outputs(args.dump_outputs, d_film.cpu().numpy().reshape(film.res[1], film.res[0], 3), last.tolist())

        # ---- e2e: public API with host buffers; scene upload + job upload + film read-back inside the timed region ----
        film_host = np.zeros((film.res[1], film.res[0], 3), np.float32)
        flat = host_scene.flat
        scene_bytes = flat.n_nodes * 32 + flat.n_tris * (36 + 4 + 4 + 4 + 1)
        h2d = scene_bytes + len(my_tiles) * (12 + 8) + 8 + 2 * 64   # scene arrays, tile list + tile-area prefix sums, camera matrices
        d2h = n_pix * 12
        e2e_steps = max(1, min(args.steps, 2))

        film_pinned = torch.empty(n_pix * 3, dtype=torch.float32).pin_memory() if world > 1 and rank == 0 else None

        def e2e_step():
            d2 = api.Scene(ctx, scene, host=host_scene)       # yk_scene_create: host arrays -> HBM
            if world == 1:
                rn.render(d2, cam, film, sampler, integ, tiles=my_tiles, film_out=film_host)   # jobs H2D, film D2H
            else:  # every rank renders its tiles, the film is assembled on rank 0 over NVLink and read back there
                d_film.zero_()
                rn.render(d2, cam, film, sampler, integ, tiles=my_tiles, device_film_ptr=d_film.data_ptr())
                dist.reduce(d_film, dst=0, op=dist.ReduceOp.SUM)
                if rank == 0:
                    film_pinned.copy_(d_film)
            d2.close()

        e2e_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = total_samples * e2e_steps / float(e2e_s.item()) / 1e6

    large = None
    if not args.no_large_scene and SCENE == "cornell":
        large = large_scene_leg(args, api, capi, xf, ctx, stream, rank, world, local, peaks()[0])

    if rank == 0:
        peak, peak_src = peaks()
        traffic = ncu_traffic("c2" if SCENE == "cornell" else "c5")
        alg_bytes = 32 * agg["closest_nodes"] + 36 * agg["closest_tris"]
        launches = max(agg["trace_closest_launches"], 1)
        t_closest = max(agg["trace_closest_ms"], 1e-9) / 1e3
        achieved = alg_bytes / t_closest / 1e9
        line = {
            "metric": "Msamples/s", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tile_dim": 16, "partition": f"spiral tiles interleaved over {world} rank(s)",
                       "l2": "256 MB L2 flush between steps; wavefront state (tens of GB per batch) exceeds the 126 MB L2" + ("; the 37-node scene is cache-resident by nature" if SCENE == "cornell" else ""),
                       "wavefront": "up to 64 Mi paths per batch (~24 GB of wavefront state per pipe), queue lengths on the device (no host sync per bounce)",
                       "pipes": ("value / roofline: one pipe, so that a kernel's event-bracketed time is its own; e2e: the library default, "
                                 "two pipes overlapping one batch's shading with the other's traversal") if VALUE_PIPES == 1
                       else "library default (two pipes) on every leg"},
            "mrays_per_s": float(counts[0].item()) / (ms_total / 1e3) / 1e6,
            "mrays_per_s_total": float((counts[0] + counts[1]).item()) / (ms_total / 1e3) / 1e6,
            "gpu_launches": int(counts[2].item()),
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "includes": "yk_scene_create + yk_render with host film (pinned staging inside the library)" if world == 1 else
                    "per rank yk_scene_create + yk_render of its tiles, NCCL sum-reduce of the film to rank 0, read-back to pinned host memory there"},
            "film_digest": digest_state,
            "roofline": {"bound": "issue (cache-resident scene)" if SCENE == "cornell" else "latency/issue", "roofline_axis": "hbm",
                         "kernel": "k_trace_closest", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic["dram_bytes_per_launch"], "dram_bytes_per_launch": traffic["dram_bytes_per_launch"],
                         "l2_bytes_per_launch": traffic["l2_bytes_per_launch"], "traffic_state": traffic["traffic_state"],
                         "traffic_commit": traffic.get("traffic_commit"), "traffic_source": traffic.get("traffic_source"),
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes / launches, "avg_launch_ms": 1e3 * t_closest / launches,
                         "launches": launches, "share_of_step": agg["trace_closest_ms"] / ms_total,
                         "note": "rank 0; 32 B per node visit + 36 B per triangle test (SURVEY.md §8d). The 37-node scene is L1-resident: no node byte comes from HBM, the kernel is "
                                 "instruction-issue bound (ncu: issue-active 74-77 %, l1tex hit 85-92 %, DRAM 3-9 %), so achieved is a throughput in the roofline's unit and can "
                                 "exceed the HBM peak; the bandwidth-relevant roofline is large_scene.roofline"},
            "stage_ms_per_step": {k: v / args.steps for k, v in (("trace_closest", agg["trace_closest_ms"]), ("trace_any", agg["trace_any_ms"]),
                                                                 ("shade", agg["shade_ms"])) if v > 0},  # any / shade only with YK_STAGE_TIMING=2
        }
        # CPU baseline (rank 0, N == 1 only): bounded sample of the same workload on the host cores.
        if world == 1 and not args.no_cpu_baseline:
            st = time_cpu()
            sample = cpu_sample_text(st.samples)
            line["cpu_baseline"] = {"value": st.samples / st.seconds / 1e6, "unit": "Msamples/s", "cores": st.threads, "kind": "port",
                                    "sample": sample, "seconds": st.seconds}
        if large is not None:
            line["large_scene"] = large
        if world == 1 and not args.no_large_scene and SCENE == "cornell":
            line["published_config"] = published_config_leg(api, xf, ctx)
        emit(line)
    dev.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args):
    """`python bench.py --gpus N` WITHOUT torchrun: all N devices behind one handle (yk_multi_*, csrc/multi.inl) — one host
    thread per device inside the library, tiles popped from one shared cursor, the film assembled on device 0 by peer stores.
    Timed on the host around the blocking calls (each returns with every device synchronised); per-device busy times come
    from the library's CUDA events. The driver's N > 1 runs use torchrun (run_ours); this is the in-process alternative a
    host binding the C ABI gets."""
    import torch
    from yuki_b200 import api, transforms as xf
    n = args.gpus
    if torch.cuda.device_count() < n:
        raise SystemExit(f"bench.py --gpus {n}: only {torch.cuda.device_count()} CUDA devices")
    mctx = api.MultiContext(list(range(n)))
    out = {}
    for key in ("c2", "c5"):
        if key == "c5" and args.no_large_scene:
            continue
        if key == "c2":
            scene, cam, film, sampler, integ = workload(xf)
            steps, warmup, name = args.steps, args.warmup, WORKLOAD
        else:
            from yuki_b200 import scenes
            scene, cam = scenes.terrain_room(xf)
            film = D.FilmSettings((3840, 2160), 16)
            sampler, integ = D.SamplerType.stratified(C5_SPP_SIDE, C5_SPP_SIDE, jitter=True), D.IntegratorType.path(MAX_DEPTH)
            steps, warmup, name = C5_STEPS, C5_WARMUP, f"configs[4] geometry at {C5_SPP_SIDE * C5_SPP_SIDE} spp"
        host = api.HostScene(scene)
        ms = api.MultiScene(mctx, scene, host=host)
        n_pix = film.res[0] * film.res[1]
        total = n_pix * sampler.samples_per_pixel()
        with torch.cuda.device(0):
            d_film = torch.zeros(n_pix * 3, dtype=torch.float32, device="cuda:0")
            for _ in range(max(warmup, 1)):
                api.multi_render(mctx, ms, cam, film, sampler, integ, device_film_ptr=d_film.data_ptr())
            digest = check_digest("c2_1024spp" if key == "c2" else C5_DIGEST, film_digest(d_film), False) if not args.spp_side else None
            clocks = ClockSampler(0)
            clocks.start()
            t0 = time.perf_counter()
            busy = [0.0] * n
            rays = shadow = launches = 0
            for _ in range(steps):
                r, per = api.multi_render(mctx, ms, cam, film, sampler, integ, device_film_ptr=d_film.data_ptr())
                busy = [b + p.device_ms for b, p in zip(busy, per)]
                rays += r.stats.ray_count; shadow += r.stats.shadow_rays; launches += r.stats.kernel_launches
            sec = time.perf_counter() - t0
            clk = clocks.stop()
            if key == "c2" and args.dump_outputs:
                dump_outputs(args.dump_outputs, d_film.cpu().numpy().reshape(film.res[1], film.res[0], 3),
                             [getattr(r.stats, k) for k in DUMP_COUNTERS])
            film_host = np.zeros((film.res[1], film.res[0], 3), np.float32)
            e2e_steps = max(1, min(steps, 2))
            for k in range(e2e_steps + 1):  # the first pass warms up (pinned staging buffers of the upload, first touch of film_host)
                if k == 1:
                    t0 = time.perf_counter()
                ms2 = api.MultiScene(mctx, scene, host=host)
                api.multi_render(mctx, ms2, cam, film, sampler, integ, film_out=film_host)
                ms2.close()
            e2e_sec = time.perf_counter() - t0
        out[key] = {"workload": name, "value": total * steps / sec / 1e6, "ms_per_step": 1e3 * sec / steps, "steps": steps,
                    "per_device_busy_ms": [b / steps for b in busy], "peer_stores": mctx.peer_stores(), "film_digest": digest, "clocks": clk,
                    "mrays_per_s": rays / sec / 1e6, "mrays_per_s_total": (rays + shadow) / sec / 1e6, "gpu_launches": int(launches),
                    "e2e": total * e2e_steps / e2e_sec / 1e6}
        ms.close()
        host.close()
    c2 = out["c2"]
    line = {"metric": "Msamples/s", "value": c2["value"], "unit": "Msamples/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": c2["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tile_dim": 16, "mode": "single process: yk_multi_render, one host thread per device, tiles from one shared cursor, "
                       "film on device 0 written by peer (NVLink) stores", "timing": "host clock around blocking calls"},
            "mrays_per_s": c2["mrays_per_s"], "mrays_per_s_total": c2["mrays_per_s_total"], "gpu_launches": c2["gpu_launches"], "clocks": c2["clocks"],
            "per_device_busy_ms": c2["per_device_busy_ms"], "peer_stores": c2["peer_stores"], "film_digest": c2["film_digest"],
            "e2e": {"value": c2["e2e"], "unit": "Msamples/s", "includes": "yk_multi_scene_create + yk_multi_render with a host film"}}
    if "c5" in out:
        line["large_scene"] = out["c5"]
    emit(line)
    mctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-large-scene", action="store_true", help="skip the 10 M-triangle leg (large_scene)")
    ap.add_argument("--write-digests", action="store_true", help="store the films' digests in tests/golden/bench_film_digests.json instead of checking them")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"], help="c2 = BASELINE.json configs[1] (default, the contract's line); c5 = configs[4]")
    ap.add_argument("--spp-side", type=int, default=0, help="override the stratified grid side (spp = side^2); the line's config says so")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the film and counters of the last timed step as DIR/*.npy (GPU arms)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm renders a sample of the tiles")
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    select_workload(args.workload, args.spp_side)
    if args.impl == "reference":
        run_reference(args)
    elif args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        run_single_process(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
