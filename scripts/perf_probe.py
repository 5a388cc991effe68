"""Quick throughput probe of the wavefront renderer (not the bench contract)."""
import sys, os, time
os.environ.setdefault("YK_STAGE_TIMING", "2")  # per-stage times for analysis (the library default times the closest-hit kernel only)
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from yuki_b200 import api, desc as D, scenes, transforms as xf

def probe(name, scene, cam, film, sampler, integ, reps=2, **kw):
    ctx = api.Context(0)
    t0 = time.time(); dev = api.Scene(ctx, scene); t_scene = time.time() - t0
    rn = api.Renderer(ctx)
    best = None
    for i in range(max(reps, 1) + 2):  # the first renders of a process allocate and warm up: report the fastest
        r = rn.render(dev, cam, film, sampler, integ, **kw)
        if best is None or r.stats.device_ms < best.stats.device_ms:
            best = r
        if os.environ.get("YK_PROBE_VERBOSE"):
            print(f"    rep {i}: device {r.stats.device_ms:.2f} ms, lib wall {1e3 * r.stats.seconds:.2f} ms", flush=True)
    st = best.stats
    s = st.device_ms / 1e3
    bytes_closest = 32 * st.closest_nodes + 36 * st.closest_tris
    print(f"{name}: scene {t_scene:.2f}s tris {dev.host.n_tris} nodes {dev.host.n_nodes} | {st.samples/s/1e6:.1f} Msamples/s "
          f"{st.ray_count/s/1e6:.1f} Mrays/s(closest) {(st.ray_count+st.shadow_rays)/s/1e6:.1f} Mrays/s(total) | device {st.device_ms:.1f} ms "
          f"closest {st.trace_closest_ms:.1f} any {st.trace_any_ms:.1f} shade {st.shade_ms:.1f} | launches {st.kernel_launches} | "
          f"closest roofline {bytes_closest/ (max(st.trace_closest_ms, 1e-9)/1e3) /1e9:.0f} GB/s nodes/ray {st.closest_nodes/max(st.ray_count,1):.1f}", flush=True)
    dev.close(); ctx.close()

which = sys.argv[1] if len(sys.argv) > 1 else "cornell"
if which == "cornell16":  # one short render for ncu captures
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    probe("cornell 1024^2 path8 16spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=1)
if which == "c16":
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    probe("cornell 1024^2 path8 16spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=3)
if which == "capsweep":
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    for cap in (1 << 25, 1 << 24, 1 << 23, 1 << 22, 1 << 21):
        probe(f"cornell 1024^2 path8 64spp cap {cap}", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8), reps=2, wavefront_paths=cap)
if which == "capsweep2":  # larger batches than the default 16 Mi paths (HBM is 180 GB): Cornell at 256 spp and the 10 M-triangle scene at 16 spp
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    for pipes in (2, 1):
        for cap in (1 << 24, 1 << 25, 1 << 26):
            probe(f"cornell 1024^2 path8 256spp pipes {pipes} cap {cap >> 20} Mi", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(16, 16), D.IntegratorType.path(8), reps=1, wavefront_paths=cap, pipes=pipes)
    s, c = scenes.terrain_room(xf)
    for cap in (1 << 24, 1 << 25, 1 << 26):
        probe(f"terrain 10M path8 4K 16spp pipes 2 cap {cap >> 20} Mi", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=1, wavefront_paths=cap, pipes=2)
if which == "terrain":
    import time as _t
    t0 = _t.time(); s, c = scenes.terrain_room(xf); print(f"terrain scene desc {_t.time()-t0:.1f}s", flush=True)
    probe("terrain 10M path8 3840x2160 4spp", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8), reps=2)
    probe("terrain 10M bvh-intersections 3840x2160", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections(), reps=2)
if which == "hf16":
    s, c = scenes.heightfield(xf, 708, 708)
    probe("heightfield 1M path8 1920x1080 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=2)
    probe("heightfield 1M bvh 1920x1080 uniform 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.uniform(16), D.IntegratorType.bvh_intersections(), reps=2)
if which == "hf4":
    s, c = scenes.heightfield(xf, 708, 708)
    probe("heightfield 1M path8 1920x1080 4spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8), reps=1)
if which in ("cornell", "all"):
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    probe("cornell 1024^2 path8 16spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    probe("cornell 1024^2 path8 64spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8))
    probe("cornell 512^2 whitted3 16spp", s, c, D.FilmSettings((512, 512), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.whitted(3))
if which in ("hf", "all"):
    for sm in (D.SPLIT_SAH, D.SPLIT_MIDDLE, D.SPLIT_EQUAL_COUNTS):
        s, c = scenes.heightfield(xf, 708, 708, split_method=sm)
        probe(f"heightfield 1M split{sm} bvh 1920x1080", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    s, c = scenes.heightfield(xf, 708, 708)
    probe("heightfield 1M path8 1920x1080 4spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8))
if which in ("room", "all"):
    s, c = scenes.material_room(xf)
    probe("room 1080p path8 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
if which == "ab":  # one line per scene class, for A/B builds (YUKI_GPU_LIB=...)
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    probe("cornell 1024^2 path8 64spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8))
    s, c = scenes.material_room(xf)
    probe("room 1080p path8 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    s, c = scenes.heightfield(xf, 708, 708)
    probe("heightfield 1M path8 1920x1080 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=2)
    s, c = scenes.terrain_room(xf)
    probe("terrain 10M path8 3840x2160 4spp", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8), reps=2)
if which == "terrain1":  # one short path-traced render of the 10 M-triangle scene for ncu captures
    s, c = scenes.terrain_room(xf)
    probe("terrain 10M path8 3840x2160 1spp", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(1, 1), D.IntegratorType.path(8), reps=1)
if which == "jitter":  # run-to-run variation of one render (device time between the library's events, and wall time)
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    ctx = api.Context(0); dev = api.Scene(ctx, s); rn = api.Renderer(ctx)
    for i in range(12):
        t0 = time.time()
        r = rn.render(dev, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8))
        print(f"rep {i}: device {r.stats.device_ms:.1f} ms wall {1e3*(time.time()-t0):.1f} ms closest {r.stats.trace_closest_ms:.1f} any {r.stats.trace_any_ms:.1f} shade {r.stats.shade_ms:.1f}", flush=True)
if which == "jitter_hf4":
    s, c = scenes.heightfield(xf, 708, 708)
    ctx = api.Context(0); dev = api.Scene(ctx, s); rn = api.Renderer(ctx)
    for i in range(8):
        t0 = time.time()
        r = rn.render(dev, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8))
        print(f"rep {i}: device {r.stats.device_ms:.1f} ms wall {1e3*(time.time()-t0):.1f} ms closest {r.stats.trace_closest_ms:.1f} any {r.stats.trace_any_ms:.1f} shade {r.stats.shade_ms:.1f} launches {r.stats.kernel_launches}", flush=True)
if which == "query":  # the ray-query ABI on 8 Mi incoherent rays on the 1 M-triangle mesh: host arrays (copies included), then device arrays
    import subprocess
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True).stdout.strip(), flush=True)
    s, c = scenes.heightfield(xf, 708, 708)
    ctx = api.Context(0); dev = api.Scene(ctx, s)
    rng = np.random.default_rng(1)
    n = 1 << 23
    o = rng.uniform((-0.7, -0.4, -0.7), (0.7, 0.6, 0.7), (n, 3)).astype(np.float32)
    d = (rng.uniform((-0.7, -0.4, -0.7), (0.7, 0.6, 0.7), (n, 3)).astype(np.float32) - o)
    def best_of(name, fn, where):  # host clock around the blocking call, best of 4 after a warm-up call
        fn()
        best = 1e9
        for i in range(4):
            t0 = time.perf_counter(); r = fn(); best = min(best, time.perf_counter() - t0)
        print(f"{name}: {n / best / 1e6:.1f} Mrays/s end to end ({n} incoherent rays, {where}), {1e3 * best:.1f} ms", flush=True)
    host = "host arrays in and out"
    for name, fn in (("yk_trace", lambda: dev.intersect(o, d)), ("yk_trace (no counters)", lambda: dev.intersect(o, d, counts=False)), ("yk_occluded", lambda: dev.occluded(o, d)),
                     ("yk_query_intersect surface", lambda: dev.surface(o, d))):
        best_of(name, fn, host)
    import torch
    to, td = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    torch.cuda.synchronize()
    dv = "torch CUDA tensors in and out"
    for name, fn in (("yk_query_intersect t + id + counts", lambda: dev.intersect(to, td)), ("yk_query_intersect t + id", lambda: dev.intersect(to, td, counts=False)),
                     ("yk_query_intersect surface", lambda: dev.surface(to, td)), ("yk_query_occluded", lambda: dev.occluded(to, td))):
        best_of(name + " (device)", fn, dv)
    dev.close(); ctx.close()
if which == "whitted":  # config 1 (Cornell 512^2, Whitted depth 3, 16 spp) and a deeper tree
    s, c = scenes.cornell(xf, light="point", tall_box="glass")
    probe("cornell 512^2 whitted3 16spp", s, c, D.FilmSettings((512, 512), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.whitted(3), reps=4)
    probe("cornell 1024^2 whitted3 64spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.whitted(3), reps=3)
    probe("cornell 1024^2 whitted6 16spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.whitted(6), reps=3)
if which == "sortab":  # ray-queue sort A/B (yk_render_opts.ray_sort): every scene class, sort off / leaf-slot key / Morton key, both orders
    names = {1: "off", 2: "slot", 3: "morton", 2 | 16: "slot/trace-only", 3 | 16: "morton/trace-only"}
    only = sys.argv[2].split(",") if len(sys.argv) > 2 else ["cornell", "room", "hf", "terrain"]
    def sweep(name, s, c, film, smp, integ):
        ctx = api.Context(0); dev = api.Scene(ctx, s); rn = api.Renderer(ctx)
        ref = None
        for pipes in (1, 2):
            for mode in (1, 2, 3, 2 | 16, 3 | 16):
                best = None
                for i in range(4):
                    r = rn.render(dev, c, film, smp, integ, ray_sort=mode, pipes=pipes)
                    if best is None or r.stats.device_ms < best.stats.device_ms:
                        best = r
                st = best.stats
                if ref is None:
                    ref = best.film.copy()
                same = bool(np.array_equal(ref.view(np.uint32), best.film.view(np.uint32)))
                print(f"{name} pipes {pipes} sort {names[mode]:18s}: {st.samples / st.device_ms / 1e3:8.1f} Msamples/s device {st.device_ms:7.2f} ms closest {st.trace_closest_ms:6.2f} "
                      f"any {st.trace_any_ms:6.2f} shade {st.shade_ms:6.2f} launches {st.kernel_launches} film==unsorted {same}", flush=True)
        dev.close(); ctx.close()
    if "cornell" in only:
        s, c = scenes.cornell(xf, light="rect", tall_box="glass")
        sweep("cornell 1024^2 path8 64spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8))
    if "room" in only:
        s, c = scenes.material_room(xf)
        sweep("room 1080p path8 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    if "hf" in only:
        s, c = scenes.heightfield(xf, 708, 708)
        sweep("heightfield 1M path8 1080p 16spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    if "terrain" in only:
        s, c = scenes.terrain_room(xf)
        sweep("terrain 10M path8 4K 4spp", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8))
if which == "room4":  # one batch of the material room for ncu captures
    s, c = scenes.material_room(xf)
    probe("room 1080p path8 4spp", s, c, D.FilmSettings((1920, 1080), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8), reps=0, pipes=1)
if which == "whitted1":
    s, c = scenes.cornell(xf, light="point", tall_box="glass")
    probe("cornell 1024^2 whitted4 4spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(4), reps=0)
if which == "terrain16":  # the render of bench.py's large_scene leg (one pipe), for its ncu capture
    s, c = scenes.terrain_room(xf)
    probe("terrain 10M path8 3840x2160 16spp", s, c, D.FilmSettings((3840, 2160), 16), D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), reps=0, pipes=1)
if which == "c64":
    s, c = scenes.cornell(xf, light="rect", tall_box="glass")
    probe("cornell 1024^2 path8 64spp", s, c, D.FilmSettings((1024, 1024), 16), D.SamplerType.stratified(8, 8), D.IntegratorType.path(8), reps=3)
