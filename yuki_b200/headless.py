"""Headless render, the counterpart of `yuki --out=foo.exr` (yuki/src/main.rs:94-118 -> app/headless.rs:24-111):
load a scene file by its extension (app/util.rs:15-66), launch the renderer, print the reference's progress line while
polling `check_status`, apply the selected tone map and write an uncompressed f32 EXR.

    python -m yuki_b200.headless --scene box.pbrt --out box.exr --integrator path --max-depth 8 --sampler stratified 4 4

The reference takes integrator / sampler / film / tone-map choices from settings.yaml (app/mod.rs:17-25); here they are
flags with the reference's defaults (Whitted depth 3, Stratified 1x1 jittered, the scene file's film settings, filmic
tone map with exposure 1). The camera is the pinhole, as the reference's, unless --thin-lens (the pbrt file's `lensradius` /
`focaldistance`) or --lens-radius asks for depth of field."""
from __future__ import annotations

import argparse
import os
import sys
import time

import numpy as np

from . import api, capi, desc as D, scenes, transforms as xf

INTEGRATORS = {"whitted": D.INTEGRATOR_WHITTED, "path": D.INTEGRATOR_PATH, "bvh-intersections": D.INTEGRATOR_BVH_INTERSECTIONS,
               "geometry-normals": D.INTEGRATOR_GEOMETRY_NORMALS, "shading-normals": D.INTEGRATOR_SHADING_NORMALS,
               "shading-uvs": D.INTEGRATOR_SHADING_UVS}
SPLITS = {"sah": D.SPLIT_SAH, "middle": D.SPLIT_MIDDLE, "equal-counts": D.SPLIT_EQUAL_COUNTS}


def try_load_scene(path: str, max_shapes_in_node: int = 1, split_method: int = D.SPLIT_SAH, with_lens: bool = False):
    """app/util.rs:15-66: (SceneDesc, CameraParameters, FilmSettings) by file extension; an empty path is the built-in
    Cornell box (`Scene::cornell`, scene/mod.rs:154-531). `with_lens`: also the file's D.ThinLens (a pbrt camera's
    lensradius / focaldistance; radius 0 for the other formats)."""
    if with_lens:
        if os.path.splitext(path)[1] == ".pbrt" and os.path.exists(path):
            return api.load_pbrt(path, max_shapes_in_node, split_method, with_lens=True)
        return (*try_load_scene(path, max_shapes_in_node, split_method), D.ThinLens(0.0))
    if path == "":
        scene, cam = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_MIDDLE)
        return scene, cam, D.FilmSettings()
    if not os.path.exists(path):
        raise FileNotFoundError(f"Scene not found at '{path}'")
    ext = os.path.splitext(path)[1]
    if ext == "":
        raise ValueError("Expected a file with an extension")
    if ext == ".ply":
        scene, cam = scenes.ply(xf, path, split_method=split_method, max_shapes_in_node=max_shapes_in_node)
        return scene, cam, D.FilmSettings()
    if ext == ".xml":
        return api.load_mitsuba(path, max_shapes_in_node, split_method)
    if ext == ".pbrt":
        return api.load_pbrt(path, max_shapes_in_node, split_method)
    raise ValueError(f"Unknown extension '{ext[1:]}'")


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="python -m yuki_b200.headless", description=__doc__.split("\n\n")[0])
    ap.add_argument("--scene", default="", help=".pbrt / .xml / .ply file; empty = the built-in Cornell box")
    ap.add_argument("--out", required=True, help="EXR file to write")
    ap.add_argument("--integrator", choices=sorted(INTEGRATORS), default="whitted")
    ap.add_argument("--max-depth", type=int, default=3)
    ap.add_argument("--indirect-clamp", type=float, default=None)
    ap.add_argument("--sampler", nargs="+", default=["stratified", "1", "1"], metavar=("KIND", "N"),
                    help="'stratified NX NY' or 'uniform SPP'")
    ap.add_argument("--no-jitter", action="store_true")
    ap.add_argument("--seed", type=lambda s: int(s, 0), default=None)
    ap.add_argument("--res", type=int, nargs=2, default=None, metavar=("W", "H"), help="overrides the scene file's film resolution")
    ap.add_argument("--tile-dim", type=int, default=16)
    ap.add_argument("--split", choices=sorted(SPLITS), default="sah")
    ap.add_argument("--max-shapes-in-node", type=int, default=1)
    ap.add_argument("--tone-map", choices=["raw", "filmic", "heatmap"], default="filmic")
    ap.add_argument("--exposure", type=float, default=1.0)
    ap.add_argument("--heatmap-channel", type=int, default=0, help="0 R, 1 G, 2 B, 3 luminance")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--aov", type=aov_arg, action="append", default=[], metavar="NAME=PATH",
                    help=f"also write a companion film of the same render as a raw EXR (Path / Whitted); NAME is one of "
                         f"{', '.join(capi.AOV_NAMES)}; repeatable")
    ap.add_argument("--adaptive", type=float, default=None, metavar="REL",
                    help="adaptive sampling (Path / Whitted): stop a pixel once the standard error of its mean is at most "
                         "REL * mean + --adaptive-abs in every channel; the sampler's spp is each pixel's maximum")
    ap.add_argument("--adaptive-abs", type=float, default=0.0, metavar="A")
    ap.add_argument("--adaptive-min", type=int, default=16, metavar="N", help="first check after N samples (>= 2)")
    ap.add_argument("--adaptive-step", type=int, default=16, metavar="N", help="then a check every N samples")
    ap.add_argument("--sample-counts", default=None, metavar="PATH",
                    help="with --adaptive: write each pixel's sample count (in all three channels) as a raw EXR")
    ap.add_argument("--denoise", action="store_true",
                    help="denoise the film before the tone map (Path / Whitted): an a-trous filter guided by the render's own "
                         "radiance_sq and shading_normals companion films and, with --adaptive, its sample counts")
    ap.add_argument("--denoise-sigma", type=float, default=D.Denoise.sigma, metavar="S")
    ap.add_argument("--denoise-iterations", type=int, default=D.Denoise.iterations, metavar="K", help="1 ... 10")
    ap.add_argument("--thin-lens", action="store_true",
                    help="depth of field with the scene file's lens (pbrt: Camera lensradius / focaldistance); default: pinhole")
    ap.add_argument("--lens-radius", type=float, default=None, metavar="R",
                    help="depth of field through a thin lens of radius R (scene units); 0 = pinhole")
    ap.add_argument("--focal-distance", type=float, default=None, metavar="F",
                    help="with --lens-radius or --thin-lens: distance of the plane of focus (default: the scene file's, else 1e6)")
    args = ap.parse_args(argv)
    if args.focal_distance is not None and args.lens_radius is None and not args.thin_lens:
        ap.error("--focal-distance needs --lens-radius or --thin-lens")
    try:
        D.ThinLens(0.0 if args.lens_radius is None else args.lens_radius, 1e6 if args.focal_distance is None else args.focal_distance)
    except ValueError as e:
        ap.error(str(e))
    if args.sample_counts is not None and args.adaptive is None:
        ap.error("--sample-counts needs --adaptive")
    if args.denoise:
        if args.integrator not in ("path", "whitted"):
            ap.error("--denoise needs the Path or Whitted integrator")
        try:
            denoise_from_args(args)
            sampler, _ = settings_from_args(args)
        except ValueError as e:
            ap.error(str(e))
        if args.adaptive is None and sampler.samples_per_pixel() < 2:
            ap.error("--denoise needs at least 2 samples per pixel")
    return args


def lens_from_args(args, file_lens: D.ThinLens):
    """--thin-lens / --lens-radius R [--focal-distance F] -> D.ThinLens, each value the scene file's unless given; None
    (the pinhole) without either."""
    if not args.thin_lens and args.lens_radius is None:
        return None
    return D.ThinLens(file_lens.radius if args.lens_radius is None else args.lens_radius,
                      file_lens.focal_distance if args.focal_distance is None else args.focal_distance)


def denoise_from_args(args):
    """--denoise [--denoise-sigma S --denoise-iterations K] -> D.Denoise, or None."""
    if not args.denoise:
        return None
    return D.Denoise(args.denoise_iterations, args.denoise_sigma)


def adaptive_from_args(args):
    """--adaptive REL [--adaptive-abs A --adaptive-min N --adaptive-step N] -> D.Adaptive, or None."""
    if args.adaptive is None:
        return None
    return D.Adaptive(args.adaptive_min, args.adaptive_step, args.adaptive, args.adaptive_abs)


def aov_arg(text):
    """--aov NAME=PATH -> (name, path)."""
    name, sep, path = text.partition("=")
    if not sep or not path:
        raise argparse.ArgumentTypeError(f"expected NAME=PATH, got '{text}'")
    if name not in capi.AOV_NAMES:
        raise argparse.ArgumentTypeError(f"unknown companion film '{name}' (one of {', '.join(capi.AOV_NAMES)})")
    return name, path


def settings_from_args(args):
    kind = args.sampler[0]
    if kind == "stratified" and len(args.sampler) == 3:
        sampler = D.SamplerType.stratified(int(args.sampler[1]), int(args.sampler[2]), jitter=not args.no_jitter)
    elif kind == "uniform" and len(args.sampler) == 2:
        sampler = D.SamplerType.uniform(int(args.sampler[1]))
    else:
        raise ValueError("--sampler takes 'stratified NX NY' or 'uniform SPP'")
    if args.seed is not None:
        sampler = D.SamplerType(sampler.kind, sampler.nx, sampler.ny, sampler.jitter, args.seed)
    ik = INTEGRATORS[args.integrator]
    if ik == D.INTEGRATOR_PATH:
        integrator = D.IntegratorType.path(args.max_depth, indirect_clamp=args.indirect_clamp)
    elif ik == D.INTEGRATOR_WHITTED:
        integrator = D.IntegratorType.whitted(args.max_depth)
    elif ik == D.INTEGRATOR_BVH_INTERSECTIONS:
        integrator = D.IntegratorType.bvh_intersections()
    else:
        integrator = D.IntegratorType.debug(ik)
    return sampler, integrator


def render(args, out=sys.stdout) -> np.ndarray:
    sampler, integrator = settings_from_args(args)
    t0 = time.perf_counter()
    scene, cam, film_settings, file_lens = try_load_scene(args.scene, args.max_shapes_in_node, SPLITS[args.split], with_lens=True)
    lens = lens_from_args(args, file_lens)
    if args.res is not None or args.tile_dim != film_settings.tile_dim:
        film_settings = D.FilmSettings(tuple(args.res) if args.res is not None else tuple(film_settings.res), args.tile_dim)
    ctx = api.Context(args.device)
    dev = api.Scene(ctx, scene)
    print(f"Scene loaded in {time.perf_counter() - t0:.2f}s", file=out)
    film = api.Film(film_settings)
    rn = api.Renderer(ctx)
    start = time.perf_counter()
    denoise = denoise_from_args(args)
    aovs = [name for name, _ in args.aov] + (["radiance_sq", "shading_normals"] if denoise else [])
    if lens is not None:
        print(f"Thin lens: radius {lens.radius:g}, focal distance {lens.focal_distance:g}", file=out)
    rn.launch(dev, cam, film, sampler, integrator, aovs=aovs, adaptive=adaptive_from_args(args), lens=lens)
    width = 0
    while True:   # headless.rs:51-110
        st = rn.check_status()
        elapsed = time.perf_counter() - start
        if isinstance(st, api.RenderFinished):
            print(file=out)
            if rn.last_error is not None:
                raise rn.last_error
            print(f"Render finished in {elapsed:.2f}s", file=out)
            break
        if isinstance(st, api.RenderProgress):
            line = (f"Tile {st.tiles_done}/{st.tiles_total} | {elapsed:.1f}s elapsed, ~{st.approx_remaining_s:.0f}s remaining | "
                    f"{st.current_rays_per_s * 1e-6:>4.2f} Mrays/s")
            width = max(width, len(line))
            print(f"\r{line:<{width}}", end="", file=out, flush=True)
        time.sleep(0.01)
    pixels = film.pixels
    if denoise is not None:
        res = rn.last_result
        pixels = api.denoise(ctx, pixels, res.aovs["radiance_sq"], spp=sampler.samples_per_pixel(), sample_counts=res.sample_counts,
                             normals=res.aovs["shading_normals"], params=denoise)
        print(f"Denoised: {denoise.iterations} iterations, sigma {denoise.sigma:g}", file=out)
    if args.tone_map == "filmic":
        pixels = api.tonemap_filmic(ctx, pixels, args.exposure)
    elif args.tone_map == "heatmap":
        pixels, bounds = api.heatmap(ctx, pixels, args.heatmap_channel)
        print(f"Heatmap bounds {bounds[0]:g} .. {bounds[1]:g}", file=out)
    api.write_exr(args.out, pixels)
    for name, path in args.aov:
        api.write_exr(path, rn.last_result.aovs[name])
        print(f"wrote {name} to {path}", file=out)
    if args.sample_counts is not None:
        counts = rn.last_result.sample_counts.astype(np.float32)
        api.write_exr(args.sample_counts, np.repeat(counts[:, :, None], 3, axis=2))
        print(f"wrote sample counts to {args.sample_counts} ({int(rn.last_result.stats.samples)} samples)", file=out)
    st = rn.last_result.stats
    print(f"{st.samples / max(st.device_ms, 1e-9) * 1e-3:.1f} Msamples/s, {st.ray_count / max(st.device_ms, 1e-9) * 1e-3:.1f} Mrays/s on the device; "
          f"wrote {args.out}", file=out)
    dev.close()
    ctx.close()
    return pixels


def main(argv=None):
    render(parse_args(argv))


if __name__ == "__main__":
    main()
