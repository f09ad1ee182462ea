"""A float64 restatement of the wavefront shading kernels, vectorised over hit slots.

It follows the same lines of the application's shaders that csrc/shade.cuh and csrc/pipeline.cu cite ("S/" below):
k_shade_primary (depth-0 shade(): lights, AO view, indirect-diffuse and Phong-lobe samples, the queued rays),
k_shade_secondary (depth-1 shade() of a secondary hit: its two shadow rays and its radiance terms), secondary_radiance and
k_resolve (the expression trees of shade() / shadeAOV() and the running mean of write_pixel), for the progressive and the
realtime program.

Everything is computed in float64 from the float32 values the kernels receive, except the kernels' discrete decisions,
which take the kernel's own float32 value so that a decision never flips on rounding:
  * the RNG (TEA + 24-bit LCG) is integer arithmetic and exact; `next_rand() < 0.5f` compares its exact float32 value;
  * perpendicular()'s axis choice uses the float32 normal / mirror vector, restated bit for bit (the library builds with
    -fmad=false and these paths have no transcendental function);
  * material `type` and `reflectivity > 0.001f` use the float32 material;
  * the hit position o + t * d is taken in float32, restated bit for bit: it is the origin of the kernel's queued rays,
    and its rounding would otherwise dominate the light terms of hits close to the point light;
  * sample_env's cube face uses the float32 direction when the kernel's direction is known bit for bit (camera rays and
    captured rays); for a direction the reference samples itself the face choice cannot be reproduced, and such directions
    are flagged ill-conditioned when their two largest |components| lie within ENV_FACE_REL of each other;
  * 0 * brdf / pdf and fmaxf's clamp keep IEEE semantics (a zero pdf gives NaN, the clamp turns NaN into 0).
"""
import numpy as np

from test_independent_answers import tea16

F32 = np.float32
M_PI = float(F32(3.1415927))         # RT_M_PI, S/RaytracingUtils.hlsli:22
SAMPLER_PI = float(F32(3.14159265))  # RT_SAMPLER_PI, :69,92,103
RAY_MAX_T = float(F32(1.0e38))       # S/RaytracingCommon.hlsli:8
RAY_EPSILON = float(F32(1e-4))       # :9
NO_HIT = 0xFFFFFFFF
ENV_FACE_REL = 1e-6

# slot flags of k_shade_primary (pipeline.cu)
SLOT_DEBUG2_DIR, SLOT_DEBUG2_POINT, SLOT_HAS_SPEC, SLOT_HAS_DIFFUSE, SLOT_UNIFORM, SLOT_AO = 1, 2, 4, 8, 16, 32


class NS:
    def __init__(self, **kw):
        self.__dict__.update(kw)


# ---------------------------------------------------------------------------------------------- vector helpers
# Written once for both precisions: on float32 arrays every operation rounds like the -fmad=false kernel.
def dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def cross(a, b):
    return np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                     a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)


def normalize(a):
    inv = a.dtype.type(1) / np.sqrt(dot(a, a))
    return a * inv[..., None]


def saturate(x):
    return np.minimum(np.maximum(x, 0.0), 1.0)


def reflect(i, n):
    return i - (2.0 * n) * dot(i, n)[..., None]


# ---------------------------------------------------------------------------------------------- RNG (S/RaytracingUtils.hlsli:26-45)
class Rng:
    """Per-slot LCG states; draw(mask) advances only the masked slots and returns their float32 value (exact in float64)."""

    def __init__(self, pixel_index, frame_count):
        self.s = tea16(np.asarray(pixel_index, np.uint32), np.full(np.shape(pixel_index), frame_count, np.uint32)).astype(np.uint64)

    def draw(self, mask=None):
        nxt = (np.uint64(1664525) * self.s + np.uint64(1013904223)) & np.uint64(0xFFFFFFFF)
        if mask is not None:
            nxt = np.where(mask, nxt, self.s)
        self.s = nxt
        return (nxt & np.uint64(0xFFFFFF)).astype(np.float64) / 16777216.0


# ---------------------------------------------------------------------------------------------- scene and frame
class Scene:
    """Hit records (2 * instance + ray type, RtScene.cpp:29) with their meshes and float32 materials, and the environment."""

    def __init__(self, meshes, materials, env, instance_mesh=None, n_instances_bound=None):
        instance_mesh = list(range(len(meshes))) if instance_mesh is None else list(instance_mesh)
        n_inst = len(instance_mesh) if n_instances_bound is None else n_instances_bound
        pos, nrm, idx, voff, ioff = [], [], [], [], []
        nv = ni = 0
        for k, m in enumerate(meshes):
            pos.append(np.asarray(m.vertices["position"], np.float32))
            nrm.append(np.asarray(m.vertices["normal"], np.float32))
            idx.append(np.asarray(m.indices, np.int64))
            voff.append(nv), ioff.append(ni)
            nv += m.vertices.shape[0]
            ni += m.indices.size
        self.positions, self.normals, self.indices = np.concatenate(pos), np.concatenate(nrm), np.concatenate(idx)
        rec_mesh = np.repeat(np.asarray(instance_mesh[:n_inst], np.int64), 2)
        self.n_recs = rec_mesh.size
        self.rec_voff, self.rec_ioff = np.asarray(voff)[rec_mesh], np.asarray(ioff)[rec_mesh]
        mats = [materials[k] for k in rec_mesh]
        self.albedo = np.array([list(m.albedo)[:3] for m in mats], np.float32)
        self.specular = np.array([list(m.specular)[:3] for m in mats], np.float32)
        self.emissive = np.array([list(m.emissive) for m in mats], np.float32)
        self.reflectivity = np.array([m.reflectivity for m in mats], np.float32)
        self.roughness = np.array([m.roughness for m in mats], np.float32)
        self.type = np.array([m.type for m in mats], np.uint32)
        self.env = None if env is None else np.ascontiguousarray(env, np.float32)

    def clamp_record(self, rec):
        """A hit on an instance without a bound record is shaded with record 0 (pipeline.cu:323)."""
        rec = np.asarray(rec, np.int64)
        return np.where(rec < self.n_recs, rec, 0)

    def has_spec(self, rec):
        t = self.type[rec]
        return ((t == 1) | (t == 2)) & (self.reflectivity[rec] > F32(0.001))

    def triangle(self, rec, prim):
        i = self.rec_ioff[rec][:, None] + 3 * np.asarray(prim, np.int64)[:, None] + np.arange(3)
        return self.indices[i] + self.rec_voff[rec][:, None]

    def interpolate_normal(self, rec, prim, u, v, dt):
        """interpolateVertexAttributes (S/RaytracingCommon.hlsli:53-82), normal only, in dtype dt."""
        vi = self.triangle(rec, prim)
        n = self.normals[vi].astype(dt)
        u, v = np.asarray(u, np.float32).astype(dt), np.asarray(v, np.float32).astype(dt)
        b0 = (dt(1) - u) - v
        return (n[:, 0] * b0[:, None] + n[:, 1] * u[:, None]) + n[:, 2] * v[:, None]


class Frame:
    """The float32 per-frame constants as arrays."""

    def __init__(self, f):
        cam = f.cameraParams
        self.eye, self.U, self.V, self.W = (np.array(list(a)[:3], np.float32) for a in (cam.worldEyePos, cam.U, cam.V, cam.W))
        self.jitter = np.array(list(cam.jitters), np.float32)
        self.frame_count, self.accum_count = int(cam.frameCount), int(cam.accumCount)
        self.dl_fwd = np.array(list(f.directionalLight.forwardDir)[:3], np.float32)
        self.dl_color = np.array(list(f.directionalLight.color), np.float32)
        self.pl_pos = np.array(list(f.pointLight.worldPos)[:3], np.float32)
        self.pl_color = np.array(list(f.pointLight.color), np.float32)
        o = f.options
        self.cosine = bool(o.cosineHemisphereSampling)
        self.no_indirect_diffuse = bool(o.noIndirectDiffuse)
        self.ao = bool(o.showAmbientOcclusionOnly)
        self.view = ("indirect_diffuse" if o.showIndirectDiffuseOnly else "indirect_specular" if o.showIndirectSpecularOnly else
                     "fresnel" if o.showFresnelTerm else "albedo" if o.showGBufferAlbedoOnly else
                     "direct" if o.showDirectLightingOnly else None)
        self.debug = int(o.debug)
        self.env_strength = float(F32(o.environmentStrength))


# ---------------------------------------------------------------------------------------------- shader library
def primary_ray(fr, w, h, x, y, jitter_scale, dt):
    """RayGen's camera ray (S/ProgressiveRaytracing.hlsl:17-31, S/RealtimeRaytracing.hlsl:25-40) in dtype dt."""
    c = lambda a: np.asarray(a, np.float32).astype(dt)
    dx = ((np.asarray(x).astype(dt) + dt(0.5)) / dt(w)) * dt(2) - dt(1)
    dy = ((np.asarray(y).astype(dt) + dt(0.5)) / dt(h)) * dt(2) - dt(1)
    j = c(fr.jitter) * dt(jitter_scale)
    o = c(fr.eye) + np.array([j[0], j[1], dt(0)], dt)
    d = normalize((dx[:, None] * c(fr.U) + (-dy)[:, None] * c(fr.V)) + c(fr.W))
    return np.broadcast_to(o, d.shape), d


def perpendicular_axis(u32):
    """getPerpendicularVector's axis choice (S/RaytracingUtils.hlsli:49-56) on the kernel's float32 vector."""
    a = np.abs(u32)
    xm = ((a[:, 0] - a[:, 1]) < 0) & ((a[:, 0] - a[:, 2]) < 0)
    ym = ~xm & ((a[:, 1] - a[:, 2]) < 0)
    zm = ~(xm | ym)
    return np.stack([xm, ym, zm], axis=-1).astype(np.float64)


def _frame_dir(n, axis, x, y, z):
    bitangent = cross(n, axis.astype(n.dtype))
    tangent = cross(bitangent, n)
    return (x[:, None] * tangent + y[:, None] * n) + z[:, None] * bitangent


def cos_hemisphere(u1, u2, n, axis):
    """getCosHemisphereSample (S/RaytracingUtils.hlsli:59-79).  Returns (direction, sin of the polar angle)."""
    r, phi = np.sqrt(u1), 2.0 * SAMPLER_PI * u2
    return _frame_dir(n, axis, r * np.cos(phi), np.sqrt(1.0 - u1), r * np.sin(phi)), r


def uniform_hemisphere(u1, u2, n, axis):
    """getUniformHemisphereSample (:82-98)."""
    sin_t, phi = np.sqrt(1.0 - u1 * u1), 2.0 * SAMPLER_PI * u2
    return _frame_dir(n, axis, sin_t * np.cos(phi), u1, sin_t * np.sin(phi)), sin_t


def phong_lobe(u1, u2, mirror, axis, exponent):
    """samplePhongLobe (:101-123).  Returns (direction, pdf, brdf, sin of the polar angle)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        cos_t = u1 ** (1.0 / (exponent + 1.0))
        sin_t = np.sqrt(1.0 - cos_t * cos_t)
        pc = cos_t ** exponent
    phi = 2.0 * SAMPLER_PI * u2
    pdf = (exponent + 1.0) / (2.0 * SAMPLER_PI) * pc
    brdf = (exponent + 2.0) / (2.0 * SAMPLER_PI) * pc
    return _frame_dir(mirror, axis, sin_t * np.cos(phi), cos_t, sin_t * np.sin(phi)), pdf, brdf, sin_t


def fresnel_schlick(i, n, f0):
    """FresnelReflectanceSchlick (:126-130)."""
    p = (1.0 - saturate(dot(-i, n))) ** 5.0
    return f0 + (1.0 - f0) * p[:, None]


def phong_exponent(roughness):
    return np.exp((1.0 - roughness.astype(np.float64)) * 12.0)


def env_face_ill_conditioned(d):
    """Directions whose cube face the float64 reference cannot decide for the kernel."""
    a = np.sort(np.abs(d), axis=-1)
    return (a[:, 2] - a[:, 1]) <= ENV_FACE_REL * a[:, 2]


def sample_env(env, d, d_face=None):
    """sampleEnvironment's cube lookup (S/RaytracingCommon.hlsli:149-159; pipeline.cu's sample_env): D3D face order, bilinear
    inside the face, clamped at its borders.  The face is chosen on d_face (the kernel's float32 direction) when given."""
    out = np.zeros(d.shape, np.float64)
    if env is None or d.shape[0] == 0:
        return out
    n = env.shape[1]
    df = d if d_face is None else d_face
    a = np.abs(df)
    xmaj = (a[:, 0] >= a[:, 1]) & (a[:, 0] >= a[:, 2])
    ymaj = ~xmaj & (a[:, 1] >= a[:, 2])
    zmaj = ~xmaj & ~ymaj
    pos = df > 0
    face = np.where(xmaj, np.where(pos[:, 0], 0, 1), np.where(ymaj, np.where(pos[:, 1], 2, 3), np.where(pos[:, 2], 4, 5)))
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    u = np.select([face == 0, face == 1, face == 2, face == 3, face == 4], [-z, z, x, x, x], -x)
    v = np.select([face == 0, face == 1, face == 2, face == 3, face == 4], [-y, -y, z, -z, -y], -y)
    ma = np.abs(np.select([xmaj, ymaj], [x, y], z))
    s, t = (u / ma + 1.0) * 0.5, (v / ma + 1.0) * 0.5
    fx, fy = s * n - 0.5, t * n - 0.5
    x0f, y0f = np.floor(fx), np.floor(fy)
    wx, wy = (fx - x0f)[:, None], (fy - y0f)[:, None]
    x0, y0 = x0f.astype(np.int64), y0f.astype(np.int64)
    cl = lambda k: np.clip(k, 0, n - 1)
    x1, y1, x0, y0 = cl(x0 + 1), cl(y0 + 1), cl(x0), cl(y0)
    tex = env.astype(np.float64)[..., :3]
    t00, t10, t01, t11 = tex[face, y0, x0], tex[face, y0, x1], tex[face, y1, x0], tex[face, y1, x1]
    top, bot = t00 + (t10 - t00) * wx, t01 + (t11 - t01) * wx
    return top + (bot - top) * wy


def eval_lights(fr, p, n):
    """evaluateDirectionalLight / evaluatePointLight without the visibility factor (S/RaytracingCommon.hlsli:126-147)."""
    dl_l = normalize(-fr.dl_fwd.astype(np.float64))
    nol = saturate(dot(n, dl_l[None, :]))
    dir_pre = fr.dl_color[:3].astype(np.float64) * float(fr.dl_color[3]) * nol[:, None]
    path = fr.pl_pos.astype(np.float64) - p
    dist = np.sqrt(dot(path, path))
    pl_l = path / dist[:, None]
    nolp = saturate(dot(n, pl_l))
    falloff = 1.0 / (2 * M_PI * dist * dist)
    point_pre = fr.pl_color[:3].astype(np.float64) * float(fr.pl_color[3]) * nolp[:, None]
    # the same terms at NoL = 1: what a float32 error of ~1 ulp of 1 in the saturated cosine is multiplied by
    dir_unit = np.broadcast_to(fr.dl_color[:3].astype(np.float64) * float(fr.dl_color[3]), p.shape)
    point_unit = np.broadcast_to(fr.pl_color[:3].astype(np.float64) * float(fr.pl_color[3]), p.shape)
    return NS(dir_l=np.broadcast_to(dl_l, p.shape), dir_pre=dir_pre, point_l=pl_l, point_dist=dist, falloff=falloff,
              point_pre=point_pre, dir_unit=dir_unit, point_unit=point_unit)


# ---------------------------------------------------------------------------------------------- k_shade_primary
def miss_colour(sc, fr, d, d_face=None):
    """PrimaryMiss (S/ProgressiveRaytracing.hlsl:160-164): the environment times environmentStrength."""
    return sample_env(sc.env, d, d_face) * fr.env_strength


def shade_primary(sc, fr, width, height, x, y, t, u, v, prim, rec, realtime):
    """Depth-0 shade() of hit slots (pipeline.cu k_shade_primary): the flags, the queued shadow-0 and secondary rays and the
    terms k_resolve reads.  x, y: image pixel; t, u, v, prim: the closest hit of the camera ray; rec: its hit-group record."""
    S = len(x)
    x, y = np.asarray(x, np.int64), np.asarray(y, np.int64)
    rec = sc.clamp_record(rec)
    js = 10.0 if realtime else 30.0
    # the camera ray is restated bit for bit in float32: the kernel's hit t belongs to that ray, so it is the input here
    o32, d32 = primary_ray(fr, width, height, x, y, js, np.float32)
    o, d = o32.astype(np.float64), d32.astype(np.float64)
    n32 = normalize(sc.interpolate_normal(rec, prim, u, v, np.float32))
    N = normalize(sc.interpolate_normal(rec, prim, u, v, np.float64))
    # HitWorldPosition: the kernel's float32 o + t * d is restated bit for bit (-fmad=false) and the lights are evaluated at
    # that point, so the rounding of the position (~1 ulp of |o| + t, large next to a close light) is not charged to them
    t32 = np.asarray(t, np.float32)
    pos32 = o32 + t32[:, None] * d32
    pos = pos32.astype(np.float64)
    rng = Rng((x + y * width).astype(np.uint32), fr.frame_count)
    flags = np.zeros(S, np.uint32)
    nplanes = 4 if (fr.ao and not realtime) else 2
    sh_dir = np.zeros((4, S, 3))
    sh_dir[..., 2] = 1.0
    sh_tmax = np.full((4, S), -1.0)
    sec_dir = np.zeros((2, S, 3))
    sec_dir[..., 2] = 1.0
    # the same samples evaluated in float32 (numpy's sin / cos / pow in place of CUDA's): rays that follow the kernel's own
    # to within its rounding, for tracing where the kernel's rays are not at hand (tests/test_shade_reference.py)
    sh_dir32, sec_dir32 = sh_dir.astype(F32), sec_dir.astype(F32)
    sec_tmax = np.full((2, S), -1.0)
    sin_sampled = np.full((2 if nplanes == 2 else 4, S), np.inf)  # sin(polar angle) of each sampled direction, per plane
    P = NS(S=S, x=x, y=y, rec=rec, o=o, d=d, d32=d32, N=N, pos=pos, pos32=pos32, pos64=o + t32.astype(np.float64)[:, None] * d,
           pos_mag=np.abs(o) + np.abs(t32.astype(np.float64)[:, None] * d),
           flags=flags, nplanes=nplanes, realtime=realtime)
    if nplanes == 4:
        # evaluateAO: S/RaytracingCommon.hlsli:98-124 — 4 shadow rays, tMax 10
        flags[:] = SLOT_AO
        axis = perpendicular_axis(n32)
        nol, pdf = np.zeros((4, S)), np.zeros((4, S))
        for i in range(4):
            u1, u2 = rng.draw(), rng.draw()
            sampler = cos_hemisphere if fr.cosine else uniform_hemisphere
            sh_dir32[i] = sampler(u1.astype(F32), u2.astype(F32), n32, axis)[0]
            if fr.cosine:
                sh_dir[i], sin_sampled[i] = cos_hemisphere(u1, u2, N, axis)
                nol[i] = saturate(dot(N, sh_dir[i]))
                pdf[i] = nol[i] / M_PI
            else:
                sh_dir[i], sin_sampled[i] = uniform_hemisphere(u1, u2, N, axis)
                nol[i] = saturate(dot(N, sh_dir[i]))
                pdf[i] = 1.0 / (2.0 * M_PI)
            sh_tmax[i] = 10.0
        P.ao_nol, P.ao_pdf = nol, pdf
        # a zero float32 NoL makes the kernel's NoL / pdf a NaN (the pixel clamps to 0); which side of zero a tangential
        # sample falls on is a rounding decision
        P.ill = (nol < 1e-5).any(axis=0)
        P.n_shadow = np.full(S, 4)
        P.n_secondary = np.zeros(S, np.int64)
    else:
        le = eval_lights(fr, pos, N)
        use_dir, use_point = np.ones(S, bool), np.ones(S, bool)
        if not realtime and fr.debug == 2:
            first = rng.draw() < 0.5
            use_point, use_dir = ~first, first
            flags |= np.where(first, SLOT_DEBUG2_DIR, SLOT_DEBUG2_POINT).astype(np.uint32)
        sh_dir[0], sh_tmax[0] = le.dir_l, np.where(use_dir, RAY_MAX_T, -1.0)
        sh_dir[1], sh_tmax[1] = le.point_l, np.where(use_point, le.point_dist - RAY_EPSILON, -1.0)
        sh_dir32[:2] = sh_dir[:2]
        has_diffuse = not realtime and not fr.no_indirect_diffuse
        uniform_nol = np.zeros(S)
        if has_diffuse:
            axis = perpendicular_axis(n32)
            u1, u2 = rng.draw(), rng.draw()
            sec_dir32[0] = (cos_hemisphere if fr.cosine else uniform_hemisphere)(u1.astype(F32), u2.astype(F32), n32, axis)[0]
            if fr.cosine:
                sec_dir[0], sin_sampled[0] = cos_hemisphere(u1, u2, N, axis)
            else:
                sec_dir[0], sin_sampled[0] = uniform_hemisphere(u1, u2, N, axis)
                uniform_nol = saturate(dot(N, sec_dir[0]))
                flags |= np.uint32(SLOT_UNIFORM)
            flags |= np.uint32(SLOT_HAS_DIFFUSE)
            sec_tmax[0] = RAY_MAX_T
        hs = sc.has_spec(rec)
        fres = np.zeros((S, 3))
        pdf, brdf = np.ones(S), np.zeros(S)
        if hs.any():
            mirror32 = reflect(d32, n32)
            mirror = reflect(d, N)
            u1, u2 = rng.draw(hs), rng.draw(hs)
            axis = perpendicular_axis(mirror32)
            ldir, lpdf, lbrdf, lsin = phong_lobe(u1, u2, mirror, axis, phong_exponent(sc.roughness[rec]))
            e32 = np.exp((F32(1) - sc.roughness[rec]) * F32(12))
            ldir32 = phong_lobe(u1.astype(F32), u2.astype(F32), mirror32, axis, e32)[0]
            sec_dir[1] = np.where(hs[:, None], ldir, sec_dir[1])
            sec_dir32[1] = np.where(hs[:, None], ldir32, sec_dir32[1])
            pdf, brdf = np.where(hs, lpdf, pdf), np.where(hs, lbrdf, brdf)
            sin_sampled[1] = np.where(hs, lsin, np.inf)
            fres = np.where(hs[:, None], fresnel_schlick(d, N, sc.specular[rec].astype(np.float64)), 0.0)
            flags |= np.where(hs, SLOT_HAS_SPEC, 0).astype(np.uint32)
            sec_tmax[1] = np.where(hs, RAY_MAX_T, -1.0)
        P.dir_pre, P.point_pre, P.falloff, P.dir_unit, P.point_unit = le.dir_pre, le.point_pre, le.falloff, le.dir_unit, le.point_unit
        P.pdf, P.brdf, P.fres, P.uniform_nol = pdf, brdf, fres, uniform_nol
        P.n_shadow = use_dir.astype(np.int64) + use_point
        P.n_secondary = (sec_tmax >= 0).sum(axis=0)
        P.ill = np.zeros(S, bool)
    P.sh_dir, P.sh_tmax, P.sh_tmin = sh_dir[:nplanes], sh_tmax[:nplanes], np.full(nplanes, RAY_EPSILON)
    P.sec_dir, P.sec_tmax, P.sec_tmin = sec_dir, sec_tmax, RAY_EPSILON
    P.sh_dir32, P.sec_dir32 = sh_dir32[:nplanes], sec_dir32
    P.sin_sampled = sin_sampled
    return P


# ---------------------------------------------------------------------------------------------- k_shade_secondary
def shade_secondary(sc, fr, width, x, y, o32, d32, tmax, t, u, v, prim, rec, realtime):
    """Depth-1 shade() of the secondary rays of one plane (pipeline.cu k_shade_secondary).  o32, d32, tmax: the queued ray
    (float32, as the kernel reads it); t, u, v, prim, rec: its closest hit; x, y: the image pixel of the ray's hit slot.
    kind: 0 inactive, 1 miss, 2 hit.  For hits: the two shadow-1 rays and the radiance terms secondary_radiance reads."""
    S = len(x)
    x, y = np.asarray(x, np.int64), np.asarray(y, np.int64)
    o32, d32 = np.asarray(o32, np.float32).reshape(S, 3), np.asarray(d32, np.float32).reshape(S, 3)
    active = np.asarray(tmax) >= 0
    hit = active & (np.asarray(prim, np.uint32) != NO_HIT)
    kind = np.where(hit, 2, np.where(active, 1, 0))
    Q = NS(S=S, kind=kind, hit=hit, env=np.zeros((S, 3)))
    miss = active & ~hit
    Q.env[miss] = miss_colour(sc, fr, d32[miss].astype(np.float64), d32[miss])
    hi = np.flatnonzero(hit)
    Q.hi = hi
    rec = sc.clamp_record(np.asarray(rec)[hi]) if hi.size else np.zeros(0, np.int64)
    Q.rec = rec
    o, d = o32[hi].astype(np.float64), d32[hi].astype(np.float64)
    tt = np.asarray(t, np.float32)[hi]
    pp, uu, vv = np.asarray(prim)[hi], np.asarray(u)[hi], np.asarray(v)[hi]
    Q.pos32 = o32[hi] + tt[:, None] * d32[hi]  # the kernel's float32 pos (-fmad=false), the origin of its shadow-1 rays
    Q.pos = Q.pos32.astype(np.float64)
    Q.pos64 = o + tt.astype(np.float64)[:, None] * d
    Q.pos_mag = np.abs(o) + np.abs(tt.astype(np.float64)[:, None] * d)  # the size of the terms the float32 sum rounds
    n32 = normalize(sc.interpolate_normal(rec, pp, uu, vv, np.float32))
    N = normalize(sc.interpolate_normal(rec, pp, uu, vv, np.float64))
    rng = Rng((x[hi] + y[hi] * width).astype(np.uint32), fr.frame_count)  # depth 1 re-seeds with the pixel's seed
    le = eval_lights(fr, Q.pos, N)
    H = hi.size
    use_dir, use_point = np.ones(H, bool), np.ones(H, bool)
    dbg = np.zeros(H, np.uint32)
    if not realtime and fr.debug == 2:
        first = rng.draw() < 0.5
        use_point, use_dir = ~first, first
        dbg = np.where(first, 16, 32).astype(np.uint32)
    hs = sc.has_spec(rec)
    spec, fres = np.zeros((H, 3)), np.zeros((H, 3))
    if hs.any():
        mirror32 = reflect(d32[hi], n32)
        u1, u2 = rng.draw(hs), rng.draw(hs)
        _, pdf, brdf, _ = phong_lobe(u1, u2, reflect(d, N), perpendicular_axis(mirror32), phong_exponent(sc.roughness[rec]))
        with np.errstate(divide="ignore", invalid="ignore"):
            spec = np.where(hs[:, None], 0.0 * brdf[:, None] / pdf[:, None], 0.0)  # shootSecondaryRay returns 0 at depth 1
        fres = np.where(hs[:, None], fresnel_schlick(d, N, sc.specular[rec].astype(np.float64)), 0.0)
    Q.dbg = dbg
    Q.sh_dir = np.stack([le.dir_l, le.point_l])
    Q.sh_tmax = np.stack([np.where(use_dir, RAY_MAX_T, -1.0), np.where(use_point, le.point_dist - RAY_EPSILON, -1.0)])
    Q.sh_tmin = RAY_EPSILON
    Q.dir_pre, Q.point_pre, Q.falloff, Q.dir_unit, Q.point_unit = le.dir_pre, le.point_pre, le.falloff, le.dir_unit, le.point_unit
    Q.spec_term = sc.reflectivity[rec].astype(np.float64)[:, None] * spec * fres
    Q.n_shadow = use_dir.astype(np.int64) + use_point
    return Q


def secondary_radiance(sc, fr, Q, vis_dir, vis_point, realtime):
    """pipeline.cu secondary_radiance: the radiance a secondary ray returns.  vis_dir / vis_point: the shadow-1 visibility of
    each HIT (in Q.hi order)."""
    rad = np.zeros((Q.S, 3))
    miss = Q.kind == 1
    rad[miss] = Q.env[miss]
    if Q.hi.size == 0:
        return rad
    v0, v1 = np.asarray(vis_dir, np.float64)[:, None], np.asarray(vis_point, np.float64)[:, None]
    dir_c = Q.dir_pre * v0
    point_c = Q.point_pre * v1 * Q.falloff[:, None]
    direct = np.where((Q.dbg == 16)[:, None], dir_c * 2.0, np.where((Q.dbg == 32)[:, None], point_c * 2.0, dir_c + point_c))
    albedo = sc.albedo[Q.rec].astype(np.float64)
    if realtime:
        r = albedo * direct / M_PI + Q.spec_term
    else:
        em = sc.emissive[Q.rec].astype(np.float64)
        r = (em[:, :3] * em[:, 3:4] + albedo * ((direct + 0.0) / M_PI)) + Q.spec_term
    rad[Q.hi] = r
    return rad


def _direct(dbg_dir, dbg_point, dir_pre, point_pre, falloff, v0, v1):
    dir_c = dir_pre * v0[:, None]
    point_c = point_pre * v1[:, None] * falloff[:, None]
    return np.where(dbg_dir[:, None], dir_c * 2.0, np.where(dbg_point[:, None], point_c * 2.0, dir_c + point_c))


def secondary_radiance_unit(sc, Q, vis_dir, vis_point):
    """What a cosine error of 1 at the secondary hit is multiplied by in secondary_radiance (0 for misses)."""
    u = np.zeros((Q.S, 3))
    if Q.hi.size:
        v0, v1 = np.asarray(vis_dir, np.float64), np.asarray(vis_point, np.float64)
        direct = _direct(Q.dbg == 16, Q.dbg == 32, Q.dir_unit, Q.point_unit, Q.falloff, v0, v1)
        u[Q.hi] = sc.albedo[Q.rec].astype(np.float64) * direct / M_PI
    return u


# ---------------------------------------------------------------------------------------------- k_resolve
def resolve_unit(sc, fr, P, vis0, rad_diffuse, rad_spec, unit_diffuse, unit_spec):
    """What an error of 1 in every saturated cosine of a slot (NoL of each light at depth 0 and at the secondary hits, the
    uniform sample's NoL, the AO samples' NoL, Fresnel's cos i) is multiplied by in each output of resolve(), summed in
    absolute value: the conditioning of the pixel on the cosines, whose float32 error is a few ulp of 1 however small the
    cosine.  Same keys as resolve()'s outputs."""
    v = np.asarray(vis0, np.float64)
    albedo = sc.albedo[P.rec].astype(np.float64)
    out = NS()
    with np.errstate(divide="ignore", invalid="ignore"):
        if P.nplanes == 4:
            u = np.zeros(P.S)
            for k in range(4):
                u = u + np.where(fr.cosine, 0.0, v[k] / P.ao_pdf[k])  # cosine sampling: NoL / (NoL / pi) does not depend on NoL
            out.color = np.repeat((u / 4.0)[:, None], 3, axis=1)
            return out
        d2d, d2p = (P.flags & SLOT_DEBUG2_DIR) != 0, (P.flags & SLOT_DEBUG2_POINT) != 0
        direct = _direct(d2d, d2p, P.dir_unit, P.point_unit, P.falloff, v[0], v[1])
        hd, uni, hs = [(P.flags & f) != 0 for f in (SLOT_HAS_DIFFUSE, SLOT_UNIFORM, SLOT_HAS_SPEC)]
        pdf_u = 1.0 / (2.0 * M_PI)
        ind = np.where(uni[:, None], (np.abs(rad_diffuse) + unit_diffuse * P.uniform_nol[:, None]) / pdf_u, unit_diffuse * M_PI)
        ind = np.where(hd[:, None], ind, 0.0)
        refl = sc.reflectivity[P.rec].astype(np.float64)[:, None]
        ratio = np.where(hs, P.brdf / P.pdf, 0.0)[:, None]
        f0 = sc.specular[P.rec].astype(np.float64)
        spec = np.nan_to_num(refl * ratio * (unit_spec * P.fres + np.abs(rad_spec) * 5.0 * (1.0 - f0)))
        fres = np.where(hs[:, None], 5.0 * (1.0 - f0), 0.0)
        direct_term = albedo * direct / M_PI
        if P.realtime:
            out.out0, out.out1 = direct_term, spec
            return out
        out.aovs = {"direct": direct_term, "indirect-diffuse": albedo * ind / M_PI, "indirect-specular": spec,
                    "albedo": np.zeros_like(albedo), "fresnel": fres}
        view = {"indirect_diffuse": out.aovs["indirect-diffuse"], "indirect_specular": spec, "fresnel": fres,
                "albedo": out.aovs["albedo"], "direct": direct_term}
        out.color = view[fr.view] if fr.view else albedo * (direct + ind) / M_PI + spec
    return out


def resolve(sc, fr, P, vis0, rad_diffuse, rad_spec):
    """k_resolve: the colour of every hit slot before write_pixel (NaN where the kernel's arithmetic makes one), the AOVs
    0-4 (progressive) or out0 / out1 (realtime).  vis0: (planes, S) shadow-0 visibility."""
    v = np.asarray(vis0, np.float64)
    albedo = sc.albedo[P.rec].astype(np.float64)
    out = NS()
    with np.errstate(divide="ignore", invalid="ignore"):
        if P.nplanes == 4:
            vis = np.zeros(P.S)
            for k in range(4):
                vis = vis + v[k] * P.ao_nol[k] / P.ao_pdf[k]
            ao = vis / 4.0
            out.color = np.repeat(ao[:, None], 3, axis=1)
            return out
        dir_c = P.dir_pre * v[0][:, None]
        point_c = P.point_pre * v[1][:, None] * P.falloff[:, None]
        d2d, d2p = (P.flags & SLOT_DEBUG2_DIR) != 0, (P.flags & SLOT_DEBUG2_POINT) != 0
        direct = np.where(d2d[:, None], dir_c * 2.0, np.where(d2p[:, None], point_c * 2.0, dir_c + point_c))
        indirect = np.zeros((P.S, 3))
        hd = (P.flags & SLOT_HAS_DIFFUSE) != 0
        uni = (P.flags & SLOT_UNIFORM) != 0
        c = np.where(uni[:, None], rad_diffuse * P.uniform_nol[:, None] / (1.0 / (2.0 * M_PI)), rad_diffuse * M_PI)
        indirect = np.where(hd[:, None], c / 1.0, indirect)
        spec = np.zeros((P.S, 3))
        hs = (P.flags & SLOT_HAS_SPEC) != 0
        spec = np.where(hs[:, None], rad_spec * P.brdf[:, None] / P.pdf[:, None], spec)
        refl = sc.reflectivity[P.rec].astype(np.float64)[:, None]
        spec_term = refl * spec * P.fres
        direct_term = albedo * direct / M_PI
        if P.realtime:
            out.out0, out.out1 = direct_term, spec_term
            return out
        out.aovs = {"direct": direct_term, "indirect-diffuse": albedo * indirect / M_PI, "indirect-specular": spec_term,
                    "albedo": albedo, "fresnel": P.fres}
        em = sc.emissive[P.rec].astype(np.float64)
        full = (em[:, :3] * em[:, 3:4] + albedo * ((direct + indirect) / M_PI)) + spec_term
        view = {"indirect_diffuse": out.aovs["indirect-diffuse"], "indirect_specular": spec_term, "fresnel": P.fres,
                "albedo": albedo, "direct": direct_term}
        out.color = view[fr.view] if fr.view else full
    return out


def clamp(c):
    """write_pixel's fmaxf(c, 0): a NaN becomes 0."""
    return np.fmax(c, 0.0)


def running_mean(prev32, cur, n, half=False):
    """write_pixel's accumulation (S/ProgressiveRaytracing.hlsl:36-38) of the clamped float64 colour cur into the float32
    value prev32 stored after n frames, in float64; half: the R16G16B16A16_FLOAT store."""
    r = (float(n) * np.asarray(prev32, np.float64) + clamp(cur)) / float(n + 1)
    return r.astype(np.float16).astype(np.float64) if half else r


# ---------------------------------------------------------------------------------------------- hit arithmetic
def intersect_own_triangle(sc, transforms, rec, prim, o32, d32):
    """float64 intersection of each ray with its own reported triangle in its instance's object space: (t, u, v, far, edge,
    cos), far = the distance of the triangle's farthest vertex from the ray origin, edge = its longest edge and cos = |cos| of
    the angle between the ray and the triangle's normal (together the conditioning of float32 edge functions)."""
    inst = np.asarray(rec, np.int64) // 2
    vi = sc.triangle(np.asarray(rec, np.int64), prim)
    p = sc.positions[vi].astype(np.float64)  # (S, 3, 3)
    xf = np.stack([np.asarray(transforms[i], np.float64).reshape(3, 4) for i in range(len(transforms))])[inst]
    A, b = xf[:, :, :3], xf[:, :, 3]
    Ainv = np.linalg.inv(A)
    o = np.einsum("sij,sj->si", Ainv, np.asarray(o32, np.float64) - b)
    d = np.einsum("sij,sj->si", Ainv, np.asarray(d32, np.float64))
    e1, e2 = p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]
    pv = np.cross(d, e2)
    det = np.sum(e1 * pv, axis=1)
    tv = o - p[:, 0]
    u = np.sum(tv * pv, axis=1) / det
    qv = np.cross(tv, e1)
    v = np.sum(d * qv, axis=1) / det
    t = np.sum(e2 * qv, axis=1) / det
    edge = np.max(np.linalg.norm(np.stack([e1, e2, p[:, 2] - p[:, 1]], 1), axis=2), axis=1)
    far = np.max(np.linalg.norm(p - o[:, None, :], axis=2), axis=1)
    nrm = np.cross(e1, e2)
    cos = np.abs(np.sum(nrm * d, axis=1)) / (np.linalg.norm(nrm, axis=1) * np.linalg.norm(d, axis=1))
    return t, u, v, far, edge, cos
