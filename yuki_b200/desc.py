"""Plain-Python scene description shared by every front end (no native code involved).

Mirrors the pieces of yuki's `Scene` a loader fills in (yuki/src/scene/mod.rs:41-49): meshes with an
object-to-world transform (shapes/mesh.rs:8-18), textures, materials, lights and the BVH build
settings (`SceneLoadSettings`, scene/mod.rs:25-39). Transforms are (m, m_inv) pairs of row-major
f32[16] exactly like `math::Transform` (math/transform.rs:12-19); they are produced by a transform
backend (`yuki_b200.transforms` — the C ABI's yk_xf_* helpers) so the f32 arithmetic is the
reference's, not numpy's.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

# enums (values match include/yuki_gpu.h)
SPLIT_SAH, SPLIT_MIDDLE, SPLIT_EQUAL_COUNTS = 0, 1, 2
INTEGRATOR_WHITTED, INTEGRATOR_PATH, INTEGRATOR_BVH_INTERSECTIONS = 0, 1, 2
INTEGRATOR_GEOMETRY_NORMALS, INTEGRATOR_SHADING_NORMALS, INTEGRATOR_SHADING_UVS = 3, 4, 5
SAMPLER_UNIFORM, SAMPLER_STRATIFIED = 0, 1
MAT_MATTE, MAT_GLASS, MAT_METAL, MAT_GLOSSY = 0, 1, 2, 3
LIGHT_POINT, LIGHT_SPOT, LIGHT_RECT, LIGHT_DISTANT = 0, 1, 2, 3
TEX_CONSTANT, TEX_IMAGE = 0, 1
FOV_X, FOV_Y = 0, 1


@dataclass
class Transform:
    m: np.ndarray      # (16,) float32 row-major
    m_inv: np.ndarray  # (16,) float32


@dataclass
class Texture:
    kind: int = TEX_CONSTANT
    value: tuple = (0.0, 0.0, 0.0)           # f32 textures use value[0]
    image: Optional[np.ndarray] = None       # (H, W, 3) float32, row 0 = top row of the file

    @staticmethod
    def constant(r, g=None, b=None) -> "Texture":
        if g is None:
            g = b = r
        return Texture(TEX_CONSTANT, (float(np.float32(r)), float(np.float32(g)), float(np.float32(b))))

    @staticmethod
    def from_image(img: np.ndarray) -> "Texture":
        return Texture(TEX_IMAGE, (0.0, 0.0, 0.0), np.ascontiguousarray(img, dtype=np.float32))


@dataclass
class Material:
    kind: int
    tex: tuple                 # texture indices, see yk_material_desc
    eta: float = 1.5
    remap_roughness: bool = False


@dataclass
class Light:
    kind: int
    light_to_world: Transform
    intensity: tuple = (1.0, 1.0, 1.0)
    total_width_deg: float = 0.0
    falloff_start_deg: float = 0.0
    size: tuple = (0.0, 0.0)
    direction: tuple = (0.0, 0.0, 0.0)


@dataclass
class Mesh:
    object_to_world: Transform
    points: np.ndarray                      # (N, 3) float32, object space
    indices: np.ndarray                     # (T*3,) uint32
    material: int
    normals: Optional[np.ndarray] = None    # (N, 3) float32
    uvs: Optional[np.ndarray] = None        # (N, 2) float32
    area_light: int = -1


@dataclass
class Sphere:                               # Sphere::new, shapes/sphere.rs:23-33
    object_to_world: Transform
    radius: float
    material: int


@dataclass
class SceneDesc:
    meshes: List[Mesh] = field(default_factory=list)
    spheres: List[Sphere] = field(default_factory=list)   # shapes = mesh triangles in order, then the spheres ...
    objects: Optional[List[int]] = None     # ... unless given: declaration order, mesh index or -1 - sphere index
    textures: List[Texture] = field(default_factory=list)
    materials: List[Material] = field(default_factory=list)
    lights: List[Light] = field(default_factory=list)
    background: tuple = (0.0, 0.0, 0.0)
    max_shapes_in_node: int = 1             # scene/mod.rs:36
    split_method: int = SPLIT_SAH           # scene/mod.rs:35

    def add_texture(self, t: Texture) -> int:
        self.textures.append(t)
        return len(self.textures) - 1

    def add_material(self, m: Material) -> int:
        self.materials.append(m)
        return len(self.materials) - 1

    def n_triangles(self) -> int:
        return sum(len(m.indices) // 3 for m in self.meshes)


@dataclass
class CameraParameters:                     # camera.rs:23-29
    position: tuple
    target: tuple
    up: tuple = (0.0, 1.0, 0.0)
    fov_axis: int = FOV_X
    fov_deg: float = 40.0


@dataclass
class FilmSettings:                         # film.rs:13-38 (defaults 640x480, tile 16)
    res: tuple = (640, 480)
    tile_dim: int = 16
    accumulate: bool = False


@dataclass
class SamplerType:                          # sampling/mod.rs:15-19
    kind: int = SAMPLER_STRATIFIED
    nx: int = 1
    ny: int = 1
    jitter: bool = True
    seed: int = 0x73B9642E74AC471C          # the reference's commented-out debug seed (uniform.rs:35)

    @staticmethod
    def stratified(nx=1, ny=1, jitter=True, seed=0x73B9642E74AC471C) -> "SamplerType":
        return SamplerType(SAMPLER_STRATIFIED, nx, ny, jitter, seed)

    @staticmethod
    def uniform(pixel_samples=1, seed=0x73B9642E74AC471C) -> "SamplerType":
        return SamplerType(SAMPLER_UNIFORM, pixel_samples, 1, True, seed)

    def samples_per_pixel(self) -> int:
        return self.nx if self.kind == SAMPLER_UNIFORM else self.nx * self.ny


@dataclass
class IntegratorType:                       # integrators/mod.rs:33-40
    kind: int = INTEGRATOR_WHITTED
    max_depth: int = 3                      # whitted.rs:21-25, path.rs:25-32
    indirect_clamp: Optional[float] = None

    @staticmethod
    def whitted(max_depth=3) -> "IntegratorType":
        return IntegratorType(INTEGRATOR_WHITTED, max_depth)

    @staticmethod
    def path(max_depth=3, indirect_clamp=None) -> "IntegratorType":
        return IntegratorType(INTEGRATOR_PATH, max_depth, indirect_clamp)

    @staticmethod
    def bvh_intersections() -> "IntegratorType":
        return IntegratorType(INTEGRATOR_BVH_INTERSECTIONS, 0)

    @staticmethod
    def debug(kind) -> "IntegratorType":
        return IntegratorType(kind, 0)


@dataclass
class Adaptive:                             # yk_adaptive (include/yuki_gpu.h): no counterpart in the reference
    """Adaptive sampling: the sampler's samples per pixel become each pixel's maximum. After `min_samples` samples and then
    every `step`, a pixel stops once, in every channel, the squared standard error of its mean is at most
    (rel_error * mean + abs_error)^2."""
    min_samples: int = 16
    step: int = 16
    rel_error: float = 0.05
    abs_error: float = 0.0


@dataclass(frozen=True)
class ThinLens:                             # yk_thin_lens (include/yuki_gpu.h): pbrt-v3's lensradius / focaldistance
    """Depth of field: camera rays leave from a disk of `radius` (scene units) around the camera position and meet on the
    plane of focus at `focal_distance` along the view axis. Radius 0 is the pinhole."""
    radius: float
    focal_distance: float = 1e6

    def __post_init__(self):
        with np.errstate(over="ignore"):
            r, f = float(np.float32(self.radius)), float(np.float32(self.focal_distance))
        if not 0.0 <= r <= float(np.finfo(np.float32).max):   # (NaN fails the comparison)
            raise ValueError(f"ThinLens.radius must be >= 0 and finite in float32, got {self.radius}")
        if not 0.0 < f <= float(np.finfo(np.float32).max):
            raise ValueError(f"ThinLens.focal_distance must be > 0 and finite in float32, got {self.focal_distance}")


@dataclass(frozen=True)
class Denoise:                              # yk_denoise_params (include/yuki_gpu.h): no counterpart in the reference
    """The a-trous denoiser's settings: `iterations` passes (1 ... 10) at steps 1, 2, 4, ...; colour weights
    (1 + |dc|^2 / (sigma^2 (var_p + var_q) + eps))^-2."""
    iterations: int = 5
    sigma: float = 2.0
    eps: float = 1e-4

    def __post_init__(self):
        if isinstance(self.iterations, bool) or int(self.iterations) != self.iterations or not 1 <= int(self.iterations) <= 10:
            raise ValueError(f"Denoise.iterations must be an integer in 1 ... 10, got {self.iterations!r}")
        for name in ("sigma", "eps"):
            v = float(getattr(self, name))
            with np.errstate(over="ignore"):
                f = float(np.float32(v))
            if not 0.0 < f <= float(np.finfo(np.float32).max):   # (NaN fails the comparison)
                raise ValueError(f"Denoise.{name} must be > 0 and finite in float32, got {v}")
