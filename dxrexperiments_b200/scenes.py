"""Synthetic scenes for the BASELINE.json configurations (SURVEY.md section 8d).

Every generator returns a :class:`Mesh` whose vertex buffer has the reference's interleaved layout
(``{float3 position, float3 normal}``, stride 24 — libs/DXRFramework/RtModel.cpp:13-17) and a
uint32 index buffer.  Triangles are wound so that ``cross(v1-v0, v2-v0)`` points away from the
solid; that is the orientation the Fallback Layer treats as front facing
(FallbackLayerUnitTests/fallbacklayerunittests.cpp:3630-3663 with TraverseFunction.hlsli:229-241).

Everything is a pure function of its arguments and an explicit seed (numpy ``PCG64`` streams are
stable across numpy versions), so the oracle and the CUDA path always see the same bytes.
"""
from dataclasses import dataclass, field

import numpy as np

from .types import VERTEX_DTYPE


@dataclass
class Mesh:
    vertices: np.ndarray  # (V,) VERTEX_DTYPE
    indices: np.ndarray   # (3*T,) uint32

    @property
    def num_triangles(self) -> int:
        return self.indices.size // 3

    def triangles(self) -> np.ndarray:
        """(T, 3, 3) float32 triangle soup."""
        return self.vertices["position"][self.indices.reshape(-1, 3)]


def _pack(positions: np.ndarray, normals: np.ndarray, indices: np.ndarray) -> Mesh:
    v = np.zeros(positions.shape[0], dtype=VERTEX_DTYPE)
    v["position"] = positions.astype(np.float32)
    v["normal"] = normals.astype(np.float32)
    return Mesh(v, np.ascontiguousarray(indices, dtype=np.uint32).reshape(-1))


def merge(meshes) -> Mesh:
    """Concatenate meshes the way RtModel merges Assimp meshes (RtModel.cpp:35-58): vertex offset per mesh."""
    verts, idx, base = [], [], 0
    for m in meshes:
        verts.append(m.vertices)
        idx.append(m.indices + np.uint32(base))
        base += m.vertices.shape[0]
    return Mesh(np.concatenate(verts), np.concatenate(idx).astype(np.uint32))


def quad(p0, p1, p2, p3) -> Mesh:
    """Quad p0-p1-p2-p3 (counter-clockwise seen from the side its normal points to)."""
    p = np.array([p0, p1, p2, p3], dtype=np.float32)
    n = np.cross(p[1] - p[0], p[2] - p[0])
    n = n / np.linalg.norm(n)
    return _pack(p, np.tile(n, (4, 1)), np.array([0, 1, 2, 0, 2, 3]))


def box(lo, hi, inward=False) -> Mesh:
    lo, hi = np.array(lo, np.float32), np.array(hi, np.float32)
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    faces = [
        ((x1, y0, z0), (x1, y1, z0), (x1, y1, z1), (x1, y0, z1)),  # +x
        ((x0, y0, z0), (x0, y0, z1), (x0, y1, z1), (x0, y1, z0)),  # -x
        ((x0, y1, z0), (x0, y1, z1), (x1, y1, z1), (x1, y1, z0)),  # +y
        ((x0, y0, z0), (x1, y0, z0), (x1, y0, z1), (x0, y0, z1)),  # -y
        ((x0, y0, z1), (x1, y0, z1), (x1, y1, z1), (x0, y1, z1)),  # +z
        ((x0, y0, z0), (x0, y1, z0), (x1, y1, z0), (x1, y0, z0)),  # -z
    ]
    quads = []
    for f in faces:
        quads.append(quad(f[0], f[3], f[2], f[1]) if inward else quad(*f))
    return merge(quads)


def cornell_box() -> Mesh:
    """Procedural Cornell box: 5 walls + a ceiling light quad + 2 boxes = 36 triangles (config C1)."""
    room = box((-1, -1, -1), (1, 1, 1), inward=True)
    # drop the +z face (open towards the camera at z = +3.5): faces are emitted in order +x,-x,+y,-y,+z,-z
    keep = np.ones(room.indices.size // 6, dtype=bool)
    keep[4] = False
    idx = room.indices.reshape(-1, 6)[keep].reshape(-1)
    room = Mesh(room.vertices, idx)
    light = quad((-0.25, 0.995, -0.25), (0.25, 0.995, -0.25), (0.25, 0.995, 0.25), (-0.25, 0.995, 0.25))
    tall = box((-0.65, -1.0, -0.6), (-0.1, 0.2, -0.05))
    short = box((0.1, -1.0, 0.0), (0.65, -0.4, 0.55))
    return merge([room, light, tall, short])


def icosphere(subdivisions: int, radius: float = 1.0) -> Mesh:
    t = (1.0 + 5.0 ** 0.5) / 2.0
    v = np.array([(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
                  (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)], dtype=np.float64)
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    f = np.array([(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2),
                  (10, 7, 6), (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11),
                  (6, 2, 10), (8, 6, 7), (9, 8, 1)], dtype=np.int64)
    for _ in range(subdivisions):
        edges = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
        edges.sort(axis=1)
        uniq, inv = np.unique(edges, axis=0, return_inverse=True)
        inv = inv.reshape(-1)
        mid = v[uniq[:, 0]] + v[uniq[:, 1]]
        mid /= np.linalg.norm(mid, axis=1, keepdims=True)
        base = v.shape[0]
        v = np.concatenate([v, mid])
        nf = f.shape[0]
        a, b, c = base + inv[:nf], base + inv[nf:2 * nf], base + inv[2 * nf:]
        f = np.concatenate([np.stack([f[:, 0], a, c], 1), np.stack([f[:, 1], b, a], 1), np.stack([f[:, 2], c, b], 1),
                            np.stack([a, b, c], 1)])
    return _pack(v * radius, v, f.reshape(-1))


def _smooth_normals(pos: np.ndarray, idx: np.ndarray) -> np.ndarray:
    tri = idx.reshape(-1, 3)
    fn = np.cross(pos[tri[:, 1]] - pos[tri[:, 0]], pos[tri[:, 2]] - pos[tri[:, 0]])
    n = np.zeros_like(pos, dtype=np.float64)
    for k in range(3):
        np.add.at(n, tri[:, k], fn)
    ln = np.linalg.norm(n, axis=1, keepdims=True)
    ln[ln == 0] = 1.0
    return n / ln


def bunny_scale(subdivisions: int = 6, seed: int = 1234, amplitude: float = 0.1) -> Mesh:
    """Config C2: displaced icosphere (20*4^s triangles; s=6 -> 81 920) standing on a 2-triangle ground.

    The radial displacement is a sum of a few seeded low-frequency sinusoids, so the surface has
    concavities (self-shadowing, inter-reflection) like a scanned model."""
    s = icosphere(subdivisions)
    p = s.vertices["position"].astype(np.float64)
    rng = np.random.Generator(np.random.PCG64(seed))
    disp = np.zeros(p.shape[0])
    for _ in range(6):
        k = rng.normal(size=3) * 3.0
        ph = rng.uniform(0, 2 * np.pi)
        disp += np.sin(p @ k + ph)
    disp *= amplitude / 6.0 * 2.0
    p = p * (1.0 + disp)[:, None]
    # Framed by the reference camera (eye (8,10,30) -> (0,1.5,0)): the model fills about half of a 16:9 frame.  The
    # ground sits at y = -0.5 so that the reference's point light at the origin lies between the ground and the
    # model's underside instead of exactly in the ground plane (in-plane shadow rays have a zero direction
    # component, which turns the y slab of every box test into NaN and makes those rays visit the whole column).
    p = p * 7.0 + np.array([0.0, 7.6, 0.0])
    n = _smooth_normals(p, s.indices.astype(np.int64))
    body = _pack(p, n, s.indices)
    ground = quad((-25, -0.5, 25), (25, -0.5, 25), (25, -0.5, -25), (-25, -0.5, -25))
    return merge([body, ground])


def column_hall(grid: int = 16, tris_per_column: int = 1000, seed: int = 1234) -> Mesh:
    """Config C3 ("sponza-scale"): grid x grid fluted columns inside a box, ~grid^2 * tris_per_column triangles."""
    rng = np.random.Generator(np.random.PCG64(seed))
    seg = 20
    rings = max(2, tris_per_column // (2 * seg))
    meshes = []
    span = 4.0
    ang = np.linspace(0, 2 * np.pi, seg, endpoint=False)
    ys = np.linspace(0.0, 10.0, rings + 1)
    for gx in range(grid):
        for gz in range(grid):
            cx, cz = (gx - grid / 2 + 0.5) * span, (gz - grid / 2 + 0.5) * span
            r0 = 0.5 + 0.3 * rng.random()
            flute = 0.05 + 0.1 * rng.random()
            prof = r0 * (1.0 + 0.15 * np.sin(ys * rng.uniform(0.5, 2.0)))
            rr = prof[:, None] * (1.0 + flute * np.cos(8 * ang)[None, :])
            x = cx + rr * np.cos(ang)[None, :]
            z = cz + rr * np.sin(ang)[None, :]
            y = np.repeat(ys[:, None], seg, 1)
            pos = np.stack([x, y, z], -1).reshape(-1, 3)
            i0 = (np.arange(rings)[:, None] * seg + np.arange(seg)[None, :])
            i1 = (np.arange(rings)[:, None] * seg + (np.arange(seg)[None, :] + 1) % seg)
            a, b, c, d = i0, i1, i1 + seg, i0 + seg
            idx = np.stack([a, d, c, a, c, b], -1).reshape(-1)
            meshes.append(_pack(pos, _smooth_normals(pos, idx), idx))
    half = grid * span / 2 + 2
    meshes.append(box((-half, 0, -half), (half, 12, half), inward=True))
    return merge(meshes)


def triangle_soup(n: int, seed: int = 1234, extent: float = 500.0, edge: float = 1.0) -> Mesh:
    """Config C4 build workload: n small triangles with uniform centroids in [-extent, extent]^3."""
    rng = np.random.Generator(np.random.PCG64(seed))
    c = rng.uniform(-extent, extent, size=(n, 1, 3)).astype(np.float32)
    off = rng.uniform(-edge / 2, edge / 2, size=(n, 3, 3)).astype(np.float32)
    p = (c + off).reshape(-1, 3)
    tri = p.reshape(-1, 3, 3)
    fn = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    ln = np.linalg.norm(fn, axis=1, keepdims=True)
    ln[ln == 0] = 1
    nrm = np.repeat(fn / ln, 3, axis=0)
    return _pack(p, nrm, np.arange(3 * n))


def random_rigid_transforms(count: int, seed: int = 10, extent: float = 100.0, scale=(0.5, 2.0)) -> np.ndarray:
    """(count, 12) object->world 3x4 row-major transforms: random rotation, uniform scale, translation
    (the shape of GenerateRandomTranformation in the reference's TLAS tests, UT:123-157)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    q = rng.normal(size=(count, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    R = np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                  2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                  2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1).reshape(count, 3, 3)
    s = rng.uniform(scale[0], scale[1], size=(count, 1, 1))
    t = rng.uniform(-extent, extent, size=(count, 3, 1))
    return np.concatenate([R * s, t], axis=2).reshape(count, 12).astype(np.float32)


IDENTITY_3X4 = np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32)


def sky_cube(size: int = 64, seed: int = 7) -> np.ndarray:
    """Procedural HDR environment cube, (6, size, size, 4) float32, D3D face order +X,-X,+Y,-Y,+Z,-Z.

    Stands in for assets/textures/CathedralRadiance.dds (a 256^2 fp16 cube) on machines that do not
    have the reference checkout: a vertical gradient plus a warm "sun" lobe."""
    s = (np.arange(size, dtype=np.float64) + 0.5) / size * 2 - 1
    u, v = np.meshgrid(s, s)  # u along x (columns), v along y (rows)
    one = np.ones_like(u)
    dirs = [np.stack([one, -v, -u], -1), np.stack([-one, -v, u], -1), np.stack([u, one, v], -1),
            np.stack([u, -one, -v], -1), np.stack([u, -v, one], -1), np.stack([-u, -v, -one], -1)]
    out = np.zeros((6, size, size, 4), dtype=np.float32)
    sun = np.array([0.4, 0.7, 0.6])
    sun /= np.linalg.norm(sun)
    for f, d in enumerate(dirs):
        d = d / np.linalg.norm(d, axis=-1, keepdims=True)
        up = d[..., 1] * 0.5 + 0.5
        sky = np.stack([0.25 + 0.35 * up, 0.3 + 0.45 * up, 0.35 + 0.65 * up], -1)
        lobe = np.clip(d @ sun, 0, 1) ** 64
        out[f, ..., :3] = sky + lobe[..., None] * np.array([6.0, 5.0, 3.5])
        out[f, ..., 3] = 1.0
    return out


# ---------------------------------------------------------------------------------------------
# Host-side frame constants (src/ProgressiveRaytracingPipeline.cpp:151-213) in numpy, for tests/bench.

@dataclass
class Camera:
    eye: tuple = (8.0, 10.0, 30.0)   # src/DXRExperimentsApp.cpp:63
    at: tuple = (0.0, 1.5, 0.0)
    up: tuple = (0.0, 1.0, 0.0)
    fov_y: float = float(np.float32(np.pi / 4))  # libs/MiniEngine/Camera.h:141-156

    def uvw(self, aspect: float):
        """calculateCameraVariables(): w = forward (unit), u = normalize(w x up) * ulen, v = normalize(u x w) * vlen."""
        f32 = np.float32
        eye, at, up = (np.array(a, dtype=f32) for a in (self.eye, self.at, self.up))
        w = at - eye
        w = (w / f32(np.sqrt(f32(np.dot(w, w))))).astype(f32)
        right = np.cross(w, up).astype(f32)
        right = (right / f32(np.linalg.norm(right))).astype(f32)
        cam_up = np.cross(right, w).astype(f32)  # BaseCamera::SetLookDirection
        u = np.cross(w, cam_up).astype(f32)
        u = (u / f32(np.linalg.norm(u))).astype(f32)
        v = np.cross(u, w).astype(f32)
        v = (v / f32(np.linalg.norm(v))).astype(f32)
        vlen = f32(np.linalg.norm(w)) * f32(np.tan(f32(0.5) * f32(self.fov_y)))
        ulen = f32(vlen * f32(aspect))
        return (u * ulen).astype(f32), (v * vlen).astype(f32), w.astype(f32)


def orbit(camera: Camera, degrees: float) -> Camera:
    """`camera` with its eye rotated by `degrees` about its `at` point around +y (right-handed: +x turns towards -z)."""
    a = np.radians(float(degrees))
    c, s = float(np.cos(a)), float(np.sin(a))
    dx, dz = camera.eye[0] - camera.at[0], camera.eye[2] - camera.at[2]
    eye = (camera.at[0] + c * dx + s * dz, camera.eye[1], camera.at[2] - s * dx + c * dz)
    return Camera(eye=eye, at=camera.at, up=camera.up, fov_y=camera.fov_y)


SLIDING_BOX_START = (-0.6, -0.999, 0.7)  # the box's translation at frame 0: on the floor, in front of the two Cornell boxes


def sliding_box(frame: int, step=(0.08, 0.0, 0.0)):
    """A moving-instance scene: (meshes, transforms) of a small box (instance 0, 0.3 wide) sliding across the floor of the
    Cornell room (instance 1, fixed).  At `frame` the box is translated by SLIDING_BOX_START + frame * step."""
    t = np.array(IDENTITY_3X4, np.float64)
    t[[3, 7, 11]] = np.array(SLIDING_BOX_START, np.float64) + frame * np.array(step, np.float64)
    return [box((-0.15, 0.0, -0.15), (0.15, 0.3, 0.15)), cornell_box()], [t.astype(np.float32), IDENTITY_3X4.copy()]


def sheared_positions(positions, offset) -> np.ndarray:
    """(V, 3) float32: every vertex moved by offset * h, h its height normalised to [0, 1] over the mesh (a shear that
    keeps the lowest vertices fixed), in float64 and rounded once.  dxr_headless --deform computes the same."""
    p = np.asarray(positions, np.float32).astype(np.float64)
    lo, hi = p[:, 1].min(), p[:, 1].max()
    h = (p[:, 1] - lo) / (hi - lo) if hi > lo else np.zeros(p.shape[0])
    return (p + h[:, None] * np.asarray(offset, np.float64)).astype(np.float32)


def sheared_box(frame: int, step=(0.08, 0.0, 0.0)):
    """A deforming-mesh scene: sliding_box(0)'s (meshes, transforms) with the box's top vertices moved by frame * step
    and its bottom vertices fixed (normals unchanged).  The deformation is affine, so an instance transform can express
    it too: sliding_box(0)'s transform times the shear x += (frame * step) * y / 0.3."""
    meshes, transforms = sliding_box(0)
    v = meshes[0].vertices.copy()
    v["position"] = sheared_positions(v["position"], frame * np.asarray(step, np.float64))
    return [Mesh(v, meshes[0].indices), meshes[1]], transforms


def waving_sheet(frame: float, amplitude: float = 0.15, wavelength: float = 1.6, speed: float = 0.5, cells=(48, 24)):
    """A deforming-mesh scene: (meshes, transforms) of an upright sheet (instance 0, x in [-0.7, 0.7], y in [-0.95, 0.45],
    facing the camera at z = 0.8) in the open front of the Cornell room (instance 1), with a travelling wave
    z = 0.8 + amplitude * sin(k x - speed * frame), k = 2 pi / wavelength, on a grid of cells[0] x cells[1] quads.  The
    defaults turn a normal by at most amplitude * k * speed = 0.29 rad (17 degrees) per frame, under the temporal
    denoiser's arccos(normal_cos = 0.9) = 26 degrees, and move a point by up to 0.075 along z per frame, more than
    position_tolerance * distance (0.02 * ~2.8), so without its vertex motion the sheet loses history."""
    nx, ny = cells
    k = 2.0 * np.pi / wavelength
    xs, ys = np.linspace(-0.7, 0.7, nx + 1), np.linspace(-0.95, 0.45, ny + 1)
    x, y = np.meshgrid(xs, ys)
    ph = k * x - speed * frame
    p = np.stack([x, y, 0.8 + amplitude * np.sin(ph)], -1).reshape(-1, 3)
    n = np.stack([-amplitude * k * np.cos(ph), np.zeros_like(x), np.ones_like(x)], -1).reshape(-1, 3)
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    i = np.arange((ny + 1) * (nx + 1)).reshape(ny + 1, nx + 1)
    a, b, c, d = i[:-1, :-1], i[:-1, 1:], i[1:, 1:], i[1:, :-1]  # counter-clockwise seen from +z: front faces the camera
    idx = np.stack([a, b, c, a, c, d], -1).reshape(-1)
    return [_pack(p, n, idx), cornell_box()], [IDENTITY_3X4.copy(), IDENTITY_3X4.copy()]


@dataclass
class FrameSetup:
    """Deterministic replacement of the wall-clock driven parts of update() (SURVEY.md A6)."""
    camera: Camera = field(default_factory=Camera)
    seed: int = 1234
    elapsed_time: float = 142.0  # mAnimationPaused
    dir_light_color: tuple = (0.9, 0.9, 0.9, 1.0)
    point_light_color: tuple = (0.2, 0.8, 0.6, 2.0)
    point_light_pos: tuple = (0.0, 0.0, 0.0, 1.0)

    def directional_forward(self):
        f32 = np.float32
        ang = f32(np.sin(f32(self.elapsed_time) * f32(0.2))) * f32(3.14) * f32(0.5)
        c, s = f32(np.cos(ang)), f32(np.sin(ang))
        x, y, z = f32(0.3), f32(-0.2), f32(-1.0)
        # XMVector4Transform(v, XMMatrixRotationY(a)) — row vector times matrix
        return np.array([x * c + z * s, y, -x * s + z * c, 0.0], dtype=f32)


def jitter_sequence(seed: int, frames: int, width: int, height: int) -> np.ndarray:
    """(frames, 2) jitters = (U[0,1) - 0.5) / dim, drawn x then y per frame from one seeded stream."""
    rng = np.random.Generator(np.random.PCG64(seed))
    u = rng.random(size=(frames, 2), dtype=np.float32)
    return ((u - np.float32(0.5)) / np.array([width, height], dtype=np.float32)).astype(np.float32)


# Camera of the C2/C5 benchmark scene: the bunny-scale model covers ~36 % of a 16:9 frame, the ground ~28 %.
BUNNY_CAMERA = Camera(eye=(6.0, 10.0, 19.0), at=(0.0, 7.0, 0.0))

REFERENCE_MATERIAL = dict(albedo=(0.95, 0.05, 0.0, 1.0), specular=(0.58, 0.58, 0.58, 1.0), emissive=(0, 0, 0, 0),
                          reflectivity=0.7, roughness=0.5, IoR=0.0, type=1)  # src/DXRExperimentsApp.cpp:98-103


def make_material(**kw):
    from .types import MaterialParams
    m = MaterialParams()
    d = dict(REFERENCE_MATERIAL)
    d.update(kw)
    m.albedo[:] = d["albedo"]
    m.specular[:] = d["specular"]
    m.emissive[:] = d["emissive"]
    m.reflectivity, m.roughness, m.IoR, m.type = d["reflectivity"], d["roughness"], d["IoR"], d["type"]
    return m


def default_options():
    """mShaderDebugOptions defaults: src/ProgressiveRaytracingPipeline.cpp:74-84."""
    from .types import DebugOptions
    o = DebugOptions()
    o.maxIterations = 1024
    o.cosineHemisphereSampling = 1
    o.environmentStrength = 1.0
    return o


def make_frame(setup: FrameSetup, width: int, height: int, frame_count: int, accum_count: int, jitter=(0.0, 0.0),
               options=None):
    """PerFrameConstants exactly as ProgressiveRaytracingPipeline::update fills them (:177-213), with the
    wall-clock inputs (jitter, frameCount) made explicit."""
    from .types import PerFrameConstants
    f = PerFrameConstants()
    u, v, w = setup.camera.uvw(width / height)
    f.cameraParams.worldEyePos[:] = [*setup.camera.eye, 1.0]
    f.cameraParams.U[:] = [*u, 0.0]
    f.cameraParams.V[:] = [*v, 0.0]
    f.cameraParams.W[:] = [*w, 0.0]
    f.cameraParams.jitters[:] = [float(jitter[0]), float(jitter[1])]
    f.cameraParams.frameCount = frame_count
    f.cameraParams.accumCount = accum_count
    f.directionalLight.forwardDir[:] = setup.directional_forward().tolist()
    f.directionalLight.color[:] = setup.dir_light_color
    f.pointLight.worldPos[:] = setup.point_light_pos
    f.pointLight.color[:] = setup.point_light_color
    f.options = options if options is not None else default_options()
    return f


# ---------------------------------------------------------------------------------------------
# The BASELINE.json workloads (SURVEY.md 8d), shared by bench.py and the full-size tests.

HALL_CAMERA = Camera(eye=(-29.0, 6.0, -29.0), at=(0.0, 4.0, 0.0))
CLOUD_CAMERA = Camera(eye=(0.0, 40.0, 330.0), at=(0.0, 0.0, 0.0))


@dataclass
class Workload:
    name: str
    description: str
    meshes: list
    transforms: list
    instance_mesh: list
    materials: list
    setup: FrameSetup
    width: int
    height: int
    spp: int
    realtime: bool = False

    @property
    def num_triangles(self) -> int:
        return int(sum(self.meshes[k].num_triangles for k in self.instance_mesh))


def workload(name: str, subdiv: int = 6) -> Workload:
    """C2: bunny-scale mesh, 1080p, 16 spp progressive.  C3: sponza-scale column hall (~260 k tris), 4K, 64 spp.
    C4: 512 instances (random rigid transforms, seed 10) of one 20 480-triangle BLAS = 10.5 M triangles, 1080p, 4 spp.
    C5: the C2 scene through the realtime pipeline (1 spp + DenoiseCompositor), 1080p."""
    if name in ("C2", "C5"):
        m = bunny_scale(subdiv)
        return Workload(name, f"{name} bunny-scale synthetic mesh ({m.num_triangles} tris) 1920x1080 " +
                        ("16 spp progressive (Phong, 2 lights, 1 indirect-diffuse + 1 Phong-lobe bounce)" if name == "C2" else
                         "realtime pipeline: 1 spp + shadow rays + Phong-lobe bounce + DenoiseCompositor"),
                        [m], [IDENTITY_3X4], [0], [make_material()], FrameSetup(camera=BUNNY_CAMERA), 1920, 1080,
                        16 if name == "C2" else 1, realtime=(name == "C5"))
    if name == "C1M":  # the north-star target scene: >= 1 Grays/s of incoherent secondary rays on ~1 M triangles at 1080p
        m = bunny_scale(8)
        return Workload(name, f"C1M 1M-triangle-scale synthetic mesh ({m.num_triangles} tris, flat BLAS, traversal section "
                        "~200 MB > L2) 1920x1080 4 spp progressive", [m], [IDENTITY_3X4], [0], [make_material()],
                        FrameSetup(camera=BUNNY_CAMERA), 1920, 1080, 4)
    if name == "C3":
        m = column_hall(16, 1000)
        setup = FrameSetup(camera=HALL_CAMERA, point_light_pos=(0.0, 8.0, 0.0, 1.0))
        return Workload(name, f"C3 sponza-scale column hall ({m.num_triangles} tris) 3840x2160 64 spp progressive", [m],
                        [IDENTITY_3X4], [0], [make_material()], setup, 3840, 2160, 64)
    if name == "C4":
        s = icosphere(5, 4.0)
        xf = random_rigid_transforms(512, seed=10, extent=100.0)
        setup = FrameSetup(camera=CLOUD_CAMERA, point_light_pos=(0.0, 0.0, 0.0, 1.0))
        return Workload(name, f"C4 instanced scene: 512 instances x {s.num_triangles}-tri BLAS = {512 * s.num_triangles} tris "
                        "(TLAS over BLAS), 1920x1080 4 spp progressive", [s], list(xf), [0] * 512, [make_material()], setup,
                        1920, 1080, 4)
    raise ValueError(name)
