"""Generates tests/golden/reference_screenshot_regions.json from the reference's only published render, screenshot.png of a
yuki checkout (embedded by readme.md:3): python tests/golden/make_screenshot_regions.py <yuki>/screenshot.png. The tests only
read the committed JSON. No pixels are copied: the fixture holds the mean colour of a few flat regions, two floor
profiles, the box opening's edges and the light quad's bounding box, i.e. measurements of the picture.

What the screenshot shows (every setting is visible in its UI panel; window client area = 1920 x 1080 at (1, 38), so the film
is displayed 1:1): scene "Cornell Box" (Scene::cornell(), scene/mod.rs:154-531: 36 triangles + the copper sphere = 37 shapes),
film 1920 x 1080, tile 32, Stratified 32 x 32 jittered = 1024 spp, camera position (0.278, 0.273, 0.8) -> target (0.278,
0.273, -0.26) (shown rounded to one decimal) with FoV X 64, SurfaceAreaHeuristic / 1 shape per leaf, Path max_depth 10,
indirect clamp 2.0, Filmic tone map, exposure 1.0; status "Render finished in 272.10s / 20.47 Mrays/s"."""
import json
import os
import sys

import numpy as np
from PIL import Image

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_screenshot_regions.json")
CLIENT_X, CLIENT_Y, W, H = 1, 38, 1920, 1080

# film-pixel boxes (x0, y0, x1, y1), chosen inside flat, directly or indirectly lit surfaces, away from edges, objects and the UI
REGIONS = {
    "red wall": (470, 300, 600, 800),
    "green wall": (1330, 300, 1460, 800),
    "ceiling left": (600, 60, 850, 200),
    "ceiling right": (1080, 60, 1330, 200),
    "floor front": (600, 980, 900, 1040),
    "floor right": (1150, 1000, 1300, 1040),
    "sphere shadow": (1050, 980, 1180, 1010),
    "light": (900, 130, 1020, 155),
    "outside the box": (1600, 300, 1800, 800),
    # the back wall carries the marble texture whose PNG is missing from the checkout: used only to fit the substitute albedo
    "back wall": (700, 300, 1200, 420),
}


def main(src):
    im = np.array(Image.open(src).convert("RGB")).astype(np.float64)
    assert im.shape == (1119, 1922, 3), im.shape
    film = im[CLIENT_Y:CLIENT_Y + H, CLIENT_X:CLIENT_X + W]
    out = {"source": "screenshot.png (readme.md:3)", "film": [W, H], "client_origin": [CLIENT_X, CLIENT_Y],
           "settings": {"scene": "Scene::cornell()", "shapes": 37, "camera_position": [0.278, 0.273, 0.8], "camera_target": [0.278, 0.273, -0.26],
                        "fov_x_deg": 64.0, "tile_dim": 32, "sampler": "stratified 32x32 jittered", "integrator": "path", "max_depth": 10,
                        "indirect_clamp": 2.0, "tone_map": "filmic", "exposure": 1.0},
           "published": {"render_seconds": 272.10, "mrays_per_s": 20.47, "note": "status line of the screenshot; hardware not stated "
                         "(sampling/mod.rs:92-96 mentions the author's Ryzen 5900X)"},
           "regions": {}}
    for name, (x0, y0, x1, y1) in REGIONS.items():
        px = film[y0:y1, x0:x1]
        out["regions"][name] = {"box": [x0, y0, x1, y1], "mean_rgb8": [round(float(v), 2) for v in px.mean(axis=(0, 1))],
                                "std_rgb8": [round(float(v), 2) for v in px.std(axis=(0, 1))]}
    # geometry: the box opening (first / last non-black pixel of a row / column through the middle), the light quad's extent
    lit = film.sum(axis=2) > 30
    row, col = lit[562], lit[:, 960]
    cols = np.where(row)[0]
    cols = cols[cols > 380]   # right of the settings panel
    rows = np.where(col)[0]
    out["box_opening"] = {"x_first": int(cols[0]), "x_last": int(cols[-1]), "y_first": int(rows[0]), "y_last": int(rows[-1])}
    sat = (film.min(axis=2) >= 250)
    sat[:, :400] = False
    ys, xs = np.where(sat[:400])
    out["light_quad"] = {"x_min": int(xs.min()), "x_max": int(xs.max()), "y_min": int(ys.min()), "y_max": int(ys.max())}
    # two floor profiles (mean of 16 x 16 blocks along a row): they carry the shadows of the sphere and the box
    for name, y in (("floor profile y=1030", 1030), ("floor profile y=960", 960)):
        xs0 = list(range(480, 1440, 32))
        out[name] = {"y": y, "x": xs0, "block": 16, "mean_rgb8": [[round(float(v), 2) for v in film[y:y + 16, x:x + 16].mean(axis=(0, 1))] for x in xs0]}
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", OUT, out["box_opening"], out["light_quad"])


if __name__ == "__main__":
    main(sys.argv[1])
