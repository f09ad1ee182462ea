"""The shading kernels of a dispatch, ray by ray and pixel by pixel, against the float64 reference of shade_reference.py.

A dispatch is captured (rt_enable_debug_capture) and the reference recomputes what k_shade_primary, k_shade_secondary and
k_resolve should have produced FROM THEIR OWN CAPTURED INPUTS: the GPU's primary and secondary hits and the visibility
bytes of its shadow waves feed the reference, so a hit that flips on an ulp cannot make a pixel disagree and what is left
to disagree is the shading arithmetic.  Every check names the kernel, the ray plane and the pixel, and prints its measured
worst case.  Traversal is held by test_gpu_stage_parity.py; only the arithmetic of each reported hit is checked here.
"""
import numpy as np
import pytest

import shade_reference as sr
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase, bunny_case, cornell_case, two_material_case

pytestmark = pytest.mark.gpu

# ---- bounds (each one is where it is checked; the measured worst cases are printed by every test)
# Ray origins: bit for bit the float32 o + t * d restated in numpy (-fmad=false), and per component within
# ORIGIN_ABS * (1 + |o| + |t d|) of the float64 value of the same inputs (two roundings of terms of that size: ~1.2e-7).
ORIGIN_ABS = 1e-6
# Light directions and the point light's tmax = dist - 1e-4, evaluated from that float32 position: 1e-6 relative.
LIGHT_REL = 1e-6
# Sampled directions: sinf / cosf / powf are a few ulp; 2e-6 on MIN_SAMPLED_FRACTION of the rays.  sin(theta) =
# sqrt(1 - cos^2) amplifies an absolute error e of cos(theta) to e / sin(theta) (phong_lobe near cos -> 1,
# uniform_hemisphere near u1 -> 1), so a ray's bound also allows SAMPLED_COND_ULPS float32 ulps of 1 over its sin(theta),
# and every ray is within SAMPLED_ALL.
SAMPLED_DIR = 2e-6
SAMPLED_COND_ULPS = 8.0 * 2.0 ** -24
MIN_SAMPLED_FRACTION = 0.999
SAMPLED_ALL = 1e-3
# Pixel colours: a float32 chain of a few dozen correctly rounded operations and a few transcendental calls stays within
# ~1e-6 relative of the float64 value; 1e-5 leaves a factor 10 and still fails a 1e-4 relative change of one term in one
# pixel.  The floor 1e-3 * mean|r| covers sums that cancel to near zero.
PIXEL_REL = 1e-5
PIXEL_FLOOR = 1e-3
# A saturated cosine (NoL, the uniform sample's NoL, an AO sample's NoL, Fresnel's cos i) is a dot product of float32 unit
# vectors: its error is a few ulp of 1 however small the cosine, so a grazing pixel is not held to PIXEL_REL of its own small
# value.  The bound adds COS_ULPS ulps of 1 times what the cosines are multiplied by (shade_reference.resolve_unit).  Before
# this term the first GPU runs measured 1.1e-5 - 2.3e-5 relative on single grazing pixels of the bunny and the sweep.
COS_ULPS = 8.0 * 2.0 ** -24
MAX_ILL_FRACTION = 1e-4
# Hit arithmetic: float32 edge functions of a triangle translated to the ray origin and sheared along the ray carry an
# absolute error ~ulp * distance in coordinates of size ~edge, and their sum (the determinant) shrinks with |cos| of the
# angle to the normal: u, v lose ~ulp * (1 + distance / edge) / |cos|, and t as much relative to t + distance (absolute, not
# relative to t: a short secondary ray to a large ground triangle keeps the error of its vertices' distance).  HIT_REL is ~32
# ulp of that: the first GPU run measured t at up to 2.03 x a bound of 1e-6 (secondary hits of the bunny and the sweep).
HIT_REL = 4e-6

SHADOW_FLAGS = T.RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH | T.RAY_FLAG_SKIP_CLOSEST_HIT_SHADER


# ---------------------------------------------------------------------------------------------- scenes
def material_sweep_case(env=True):
    """27 spheres over a ground plane: type in {0, 1, 2} x reflectivity in {0.001 exactly (no lobe: `> 0.001f`), 0.0011,
    1} x roughness in {0 (exponent e^12 ~ 1.6e5), 0.5, 1}, specular f0 alternating 0.04 / 0.9."""
    ball = scenes.icosphere(2)
    meshes, transforms, mats = [], [], []
    k = 0
    for ty in (0, 1, 2):
        for refl in (0.001, 0.0011, 1.0):
            for rough in (0.0, 0.5, 1.0):
                ix, iz = k % 9, k // 9
                meshes.append(ball)
                transforms.append(np.array([0.9, 0, 0, 2.2 * ix - 8.8, 0, 0.9, 0, 1.0, 0, 0, 0.9, 2.2 * iz - 2.2], np.float32))
                f0 = 0.04 if k % 2 == 0 else 0.9
                mats.append(scenes.make_material(type=ty, reflectivity=refl, roughness=rough, specular=(f0, f0, f0, 1.0),
                                                 albedo=(0.3 + 0.02 * k, 0.5, 0.7 - 0.02 * k, 1.0)))
                k += 1
    meshes.append(scenes.quad((-30, 0, 30), (30, 0, 30), (30, 0, -30), (-30, 0, -30)))
    transforms.append(scenes.IDENTITY_3X4)
    mats.append(scenes.make_material(type=2, reflectivity=0.4, roughness=0.2, emissive=(0.05, 0.02, 0.0, 2.0)))
    setup = scenes.FrameSetup(camera=scenes.Camera(eye=(0.0, 9.0, 14.0), at=(0.0, 0.0, 0.0)), point_light_pos=(2.0, 6.0, 3.0, 1.0))
    return SceneCase(meshes, transforms=transforms, materials=mats, setup=setup, env_size=16 if env else 0)


CASES = {"cornell": cornell_case, "bunny": lambda: bunny_case(4), "two": two_material_case, "sweep": material_sweep_case,
         "sweep_no_env": lambda: material_sweep_case(env=False)}

OPTION_CASES = {"default": {}, "uniform_hemisphere": dict(cosineHemisphereSampling=0), "no_indirect_diffuse": dict(noIndirectDiffuse=1),
                "indirect_diffuse_only": dict(showIndirectDiffuseOnly=1), "indirect_specular_only": dict(showIndirectSpecularOnly=1),
                "ambient_occlusion_only": dict(showAmbientOcclusionOnly=1),
                "ambient_occlusion_uniform": dict(showAmbientOcclusionOnly=1, cosineHemisphereSampling=0),
                "albedo_only": dict(showGBufferAlbedoOnly=1), "direct_only": dict(showDirectLightingOnly=1),
                "fresnel_only": dict(showFresnelTerm=1), "one_light_sampling": dict(debug=2),
                "environment_strength": dict(environmentStrength=2.5)}


def options(overrides):
    o = scenes.default_options()
    for k, v in overrides.items():
        setattr(o, k, v)
    return o


def ref_scene(case, n_instances_bound=None):
    return sr.Scene(case.meshes, case.materials, case.env, n_instances_bound=n_instances_bound)


# ---------------------------------------------------------------------------------------------- capture
def image_row(ly, y0, strips):
    """pipeline.cu image_row: virtual row -> image row of a region or strip-interleaved dispatch."""
    if strips is None or strips[1] <= 1:
        return y0 + ly
    rows, groups, group = strips
    shift = rows.bit_length() - 1
    return (((ly >> shift) * groups + group) << shift) + (ly & (rows - 1))


def capture(ctx, r, frame, region=None, strips=None):
    ctx.ray_counts(reset=True)
    ctx.enable_debug_capture(True)
    try:
        r.dispatch(frame, region=region, strips=strips)
        c = ctx.debug_counts()
        a = NSd(counts=c, ph=ctx.debug_array("primary_hits"), pr=ctx.debug_array("primary_records"),
                info=ctx.debug_array("slot_info"), rays=ctx.ray_counts())
        a.sec = [ctx.debug_array("secondary_rays", k) for k in range(2)]
        a.sec_hits = [ctx.debug_array("secondary_hits", k) for k in range(2)]
        a.sec_rec = [ctx.debug_array("secondary_records", k) for k in range(2)]
        a.sh0 = [ctx.debug_array("shadow0_rays", k) for k in range(4)]
        a.vis0 = [ctx.debug_array("shadow0_visibility", k) for k in range(4)]
        a.sh1 = [ctx.debug_array("shadow1_rays", k) for k in range(2)]
        a.vis1 = [ctx.debug_array("shadow1_visibility", k) for k in range(2)]
        return a
    finally:
        ctx.enable_debug_capture(False)


class NSd(sr.NS):
    pass


class Worst:
    """Measured worst case of every check of one test, printed at the end."""

    def __init__(self):
        self.v = {}

    def add(self, name, value):
        self.v[name] = max(self.v.get(name, 0.0), float(value))

    def print(self, title):
        print(f"\n{title}: " + ", ".join(f"{k} {v:.2e}" for k, v in sorted(self.v.items())))


def _where(mask):
    i = np.flatnonzero(mask)
    return i[:5].tolist()


def check_origin(name, got, want32, want64, mag, worst):
    same = (np.asarray(got, np.float32) == want32).all(axis=-1)
    assert same.all(), f"{name}: origin is not the float32 o + t * d at slots {_where(~same)}"
    err = np.abs(np.asarray(got, np.float64) - want64) / (1.0 + mag)
    worst.add("origin", err.max(initial=0))
    assert (err <= ORIGIN_ABS).all(), f"{name}: origin off by {err.max():.3e} at slots {_where((err > ORIGIN_ABS).any(-1))}"


def check_light_dir(name, got, want, worst):
    err = np.abs(np.asarray(got, np.float64) - want).max(axis=-1) / np.abs(want).max(axis=-1)
    worst.add("light direction", err.max(initial=0))
    assert (err <= LIGHT_REL).all(), f"{name}: light direction off by {err.max():.3e} at slots {_where(err > LIGHT_REL)}"


def check_sampled_dir(name, got, want, sin_t, worst):
    if len(want) == 0:
        return
    err = np.abs(np.asarray(got, np.float64) - want).max(axis=-1)
    bound = SAMPLED_DIR + SAMPLED_COND_ULPS / np.maximum(sin_t, 1e-30)
    i = int(np.argmax(err / bound))
    print(f"  {name}: worst ray slot {i}: |dd| {err[i]:.3e} (sin theta {sin_t[i]:.3e}); largest |dd| {err.max():.3e}")
    worst.add("sampled direction / bound", (err / bound).max())
    frac = float((err <= bound).mean())
    assert frac >= MIN_SAMPLED_FRACTION, f"{name}: only {frac:.5f} of the sampled directions within the bound"
    assert (err <= SAMPLED_ALL).all(), f"{name}: sampled direction off by {err.max():.3e} at slots {_where(err > SAMPLED_ALL)}"


def check_tmax(name, got, want, worst):
    got = np.asarray(got, np.float64)
    inactive = want < 0
    assert np.array_equal(got < 0, inactive), f"{name}: active planes differ at slots {_where((got < 0) != inactive)}"
    assert (got[inactive] == -1.0).all(), f"{name}: inactive tmax is not -1"
    big = want >= sr.RAY_MAX_T
    assert (got[big] == np.float32(1e38)).all(), f"{name}: tmax of an unbounded ray is not 1e38"
    fin = ~inactive & ~big
    if fin.any():
        err = np.abs(got[fin] - want[fin]) / np.abs(want[fin])
        worst.add("light tmax", err.max())
        assert (err <= LIGHT_REL).all(), f"{name}: tmax off by {err.max():.3e} at slots {_where(err > LIGHT_REL)}"


def pixel_check(name, got, ref, ill, worst, half=False, where=None, unit=None):
    """|g - r| <= PIXEL_REL (|r| + PIXEL_FLOOR mean|r|) + COS_ULPS * unit per pixel, or one fp16 ulp of an fp16-representable
    value."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert np.isfinite(got).all() and (got >= 0).all(), f"{name}: non-finite or negative pixels"
    if half:
        assert np.array_equal(got.astype(np.float16).astype(np.float64), got), f"{name}: not fp16-representable"
        r16 = ref.astype(np.float16)
        ulp = np.abs(np.spacing(np.abs(r16))).astype(np.float64)
        err = np.abs(got - ref) / np.maximum(ulp, 1e-30)
        bad = (err > 1.0).any(-1) & ~ill
        worst.add("pixel fp16 ulps", err[~ill].max(initial=0))
        assert not bad.any(), f"{name}: {int(bad.sum())} pixels more than one fp16 ulp away, first {np.argwhere(bad)[:5].tolist()}"
        return
    scale = np.abs(ref) + PIXEL_FLOOR * max(float(np.abs(ref).mean()), 1e-30)
    bound = PIXEL_REL * scale + (0.0 if unit is None else COS_ULPS * np.abs(np.asarray(unit, np.float64)))
    rel = (np.abs(got - ref) / scale).max(axis=-1)
    err = (np.abs(got - ref) / bound).max(axis=-1)
    worst.add("pixel relative", rel[~ill].max(initial=0))
    worst.add("pixel / bound", err[~ill].max(initial=0))
    bad = (err > 1.0) & ~ill
    if bad.any():
        for i in np.flatnonzero(bad)[:10]:
            at = f"x={where[1][i]} y={where[0][i]}" if where is not None else f"#{i}"
            print(f"  {name} pixel {at}: got {got[i]} want {ref[i]} ({rel[i]:.2e} relative, {err[i]:.2f} x the bound)")
    assert not bad.any(), f"{name}: {int(bad.sum())} pixels outside the bound (worst {err[bad].max():.2f} x the bound)"
    assert ill.mean() <= MAX_ILL_FRACTION or ill.sum() <= 1, f"{name}: {int(ill.sum())} ill-conditioned pixels"
    if ill.any():
        print(f"  {name}: {int(ill.sum())} ill-conditioned pixels")


# ---------------------------------------------------------------------------------------------- the check of one dispatch
def check_dispatch(a, sc, frame, w, h, realtime, region=None, strips=None, worst=None, transforms=None):
    """Check a captured dispatch kernel by kernel; return the reference's (per-pixel colour terms) for its pixels as
    (ys, xs, colour or (out0, out1), ill, aovs)."""
    fr = sr.Frame(frame)
    x0, y0 = (region[0], region[1]) if region else (0, 0)
    if strips is not None:
        rw = w
    else:
        rw = (region[2] - region[0]) if region else w
    P_count = a.counts["pixels"]
    rh = P_count // rw
    assert rw * rh == P_count
    pix = np.arange(P_count)
    xs, ys = x0 + pix % rw, image_row(pix // rw, y0, strips)
    hit = a.ph["prim"] != T.NO_HIT
    info = a.info
    # ---- exact: hit pixels, records, flags
    assert np.array_equal(np.sort(info["pixel"]), np.flatnonzero(hit)), "k_shade_primary: hit slots are not the hit pixels"
    p = info["pixel"].astype(np.int64)
    rec = sc.clamp_record(a.pr[p])
    assert np.array_equal(info["record"], rec), f"k_shade_primary: slot records differ at slots {_where(info['record'] != rec)}"
    ph = a.ph[p]
    P = sr.shade_primary(sc, fr, w, h, xs[p], ys[p], ph["t"], ph["u"], ph["v"], ph["prim"], a.pr[p], realtime)
    bad = info["flags"] != P.flags
    assert not bad.any(), f"k_shade_primary: slot flags differ at slots {_where(bad)} (got {info['flags'][bad][:5]}, want {P.flags[bad][:5]})"
    # ---- k_shade_primary: shadow-0 rays
    for k in range(P.nplanes):
        q, nm = a.sh0[k], f"k_shade_primary shadow0 plane {k}"
        check_origin(nm, q["origin"], P.pos32, P.pos64, P.pos_mag, worst)
        assert (q["tmin"] == np.float32(sr.RAY_EPSILON)).all(), f"{nm}: tmin is not RT_RAY_EPSILON at slots {_where(q['tmin'] != np.float32(sr.RAY_EPSILON))}"
        if P.nplanes == 4:
            check_tmax(nm, q["tmax"], P.sh_tmax[k], worst)
            check_sampled_dir(nm, q["direction"], P.sh_dir[k], P.sin_sampled[k], worst)
        else:
            check_tmax(nm, q["tmax"], P.sh_tmax[k], worst)
            check_light_dir(nm, q["direction"], P.sh_dir[k], worst)
    # ---- k_shade_primary: secondary rays (plane 0 indirect diffuse, plane 1 Phong lobe)
    for k in range(2):
        q, nm = a.sec[k], f"k_shade_primary secondary plane {k}"
        check_origin(nm, q["origin"], P.pos32, P.pos64, P.pos_mag, worst)
        assert (q["tmin"] == np.float32(sr.RAY_EPSILON)).all(), f"{nm}: tmin is not RT_RAY_EPSILON at slots {_where(q['tmin'] != np.float32(sr.RAY_EPSILON))}"
        check_tmax(nm, q["tmax"], P.sec_tmax[k], worst)
        act = P.sec_tmax[k] >= 0
        assert (q["direction"][~act] == np.float32([0, 0, 1])).all(), f"{nm}: inactive direction"
        if P.nplanes == 2:
            check_sampled_dir(nm, q["direction"][act], P.sec_dir[k][act], P.sin_sampled[k][act], worst)
    # ---- k_shade_secondary: shadow-1 rays, matched to their secondary ray by the exact bits of the origin
    pairs = a.counts["pairs"]
    origin_bits = np.ascontiguousarray(a.sh1[0]["origin"]).view(np.uint32).reshape(-1, 3)
    lookup = {tuple(b): i for i, b in enumerate(origin_bits.tolist())}
    rad = [np.zeros((P.S, 3)), np.zeros((P.S, 3))]
    rad_unit = [np.zeros((P.S, 3)), np.zeros((P.S, 3))]
    n_sh1 = matched = 0
    ill = P.ill.copy()
    for k in range(2):
        q, sh, srec = a.sec[k], a.sec_hits[k], a.sec_rec[k]
        Q = sr.shade_secondary(sc, fr, w, xs[p], ys[p], q["origin"], q["direction"], q["tmax"], sh["t"], sh["u"], sh["v"],
                               sh["prim"], srec, realtime)
        nm = f"k_shade_secondary plane {k}"
        idx = np.array([lookup.get(tuple(b), -1) for b in Q.pos32.view(np.uint32).reshape(-1, 3).tolist()], np.int64)
        assert (idx >= 0).all(), f"{nm}: no shadow-1 pair starts at the hit of slots {Q.hi[idx < 0][:5].tolist()}"
        matched += idx.size
        r0, r1 = a.sh1[0][idx], a.sh1[1][idx]
        for j, rr in enumerate((r0, r1)):
            check_origin(f"{nm} shadow1 plane {j}", rr["origin"], Q.pos32, Q.pos64, Q.pos_mag, worst)
            assert (rr["tmin"] == np.float32(sr.RAY_EPSILON)).all(), f"{nm} shadow1 plane {j}: tmin"
            check_light_dir(f"{nm} shadow1 plane {j}", rr["direction"], Q.sh_dir[j], worst)
            check_tmax(f"{nm} shadow1 plane {j}", rr["tmax"], Q.sh_tmax[j], worst)
        n_sh1 += int(Q.n_shadow.sum())
        rad[k] = sr.secondary_radiance(sc, fr, Q, a.vis1[0][idx], a.vis1[1][idx], realtime)
        rad_unit[k] = sr.secondary_radiance_unit(sc, Q, a.vis1[0][idx], a.vis1[1][idx])
        if transforms is not None and Q.hi.size:
            check_hits(f"{nm} hits", sc, transforms, srec[Q.hi], sh[Q.hi], q["origin"][Q.hi], q["direction"][Q.hi], worst)
    assert matched == pairs, f"k_shade_secondary: {pairs} shadow-1 pairs for {matched} secondary hits"
    if transforms is not None and P.S:
        o32, d32 = sr.primary_ray(fr, w, h, xs[p], ys[p], 10.0 if realtime else 30.0, np.float32)
        check_hits("k_primary hits", sc, transforms, a.pr[p], ph, o32, d32, worst)
    # ---- rt_get_ray_counts
    assert a.rays.primary == P_count, "primary ray count"
    assert a.rays.secondary == int(P.n_secondary.sum()), f"secondary ray count {a.rays.secondary} != {int(P.n_secondary.sum())}"
    assert a.rays.shadow == int(P.n_shadow.sum()) + n_sh1, f"shadow ray count {a.rays.shadow} != {int(P.n_shadow.sum()) + n_sh1}"
    # ---- k_resolve
    vis0 = np.stack([a.vis0[k] for k in range(P.nplanes)])
    out = sr.resolve(sc, fr, P, vis0, rad[0], rad[1])
    unit = sr.resolve_unit(sc, fr, P, vis0, rad[0], rad[1], rad_unit[0], rad_unit[1])
    miss = np.flatnonzero(~hit)
    d64 = sr.primary_ray(fr, w, h, xs[miss], ys[miss], 10.0 if realtime else 30.0, np.float64)[1]
    d32 = sr.primary_ray(fr, w, h, xs[miss], ys[miss], 10.0 if realtime else 30.0, np.float32)[1]
    mc = sr.miss_colour(sc, fr, d64, d32)
    ill_px = np.zeros(P_count, bool)
    ill_px[p] = ill

    def scatter(hit_vals, miss_vals):
        img = np.zeros((P_count, 3))
        img[p] = hit_vals
        img[miss] = miss_vals
        return img

    if realtime:
        cols = (scatter(out.out0, mc), scatter(out.out1, 0.0))
        units = (scatter(unit.out0, 0.0), scatter(unit.out1, 0.0))
        aovs = None
    else:
        cols, units = scatter(out.color, mc), scatter(unit.color, 0.0)
        aovs = {k: (scatter(v, mc), scatter(unit.aovs[k], 0.0)) for k, v in out.aovs.items()} if P.nplanes == 2 else None
    return ys, xs, cols, ill_px, aovs, units


def check_hits(name, sc, transforms, rec, hits, o32, d32, worst):
    """Each reported closest hit against the float64 intersection of ITS OWN ray with ITS OWN triangle."""
    t, u, v, far, edge, cos = sr.intersect_own_triangle(sc, transforms, rec, hits["prim"], o32, d32)
    tg = hits["t"].astype(np.float64)
    cond = (1.0 + far / edge) / np.maximum(cos, 1e-12)
    du = np.maximum(np.abs(hits["u"] - u), np.abs(hits["v"] - v)) / (HIT_REL * cond)
    dt = np.abs(tg - t) / (HIT_REL * cond * (np.abs(t) + far))
    worst.add("hit uv / bound", du.max(initial=0))
    worst.add("hit t / bound", dt.max(initial=0))
    assert (du <= 1).all(), f"{name}: barycentrics off at {_where(du > 1)} ({du.max():.2f} x the bound)"
    assert (dt <= 1).all(), f"{name}: t off at {_where(dt > 1)} ({dt.max():.2f} x the bound)"


def stored(img, ys, xs):
    return np.asarray(img, np.float64)[ys, xs, :3]


def run_one(ctx, rt, case, w, h, frame, realtime=False, region=None, strips=None, name="", worst=None, sc=None,
            renderer=None, hits=True):
    r = renderer or case.renderer(rt, ctx, rt.REALTIME if realtime else rt.PROGRESSIVE, w, h)
    a = capture(ctx, r, frame, region, strips)
    ys, xs, cols, ill, aovs, units = check_dispatch(a, sc or ref_scene(case), frame, w, h, realtime, region, strips, worst,
                                                    transforms=case.transforms if hits else None)
    if realtime:
        pixel_check(f"{name} k_resolve out0", stored(r.image(0), ys, xs), sr.clamp(cols[0]), ill, worst, where=(ys, xs), unit=units[0])
        pixel_check(f"{name} k_resolve out1", stored(r.image(1), ys, xs), sr.clamp(cols[1]), ill, worst, where=(ys, xs), unit=units[1])
    else:
        pixel_check(f"{name} k_resolve", stored(r.image(0), ys, xs), sr.clamp(cols), ill, worst, where=(ys, xs), unit=units)
    return r, ys, xs, cols, ill, aovs, units


# ---------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("opt", sorted(OPTION_CASES))
@pytest.mark.parametrize("scene", sorted(CASES))
def test_shading_kernels_match_reference(scene, opt, ctx, rt):
    case = CASES[scene]()
    w, h = 72, 52
    frame = scenes.make_frame(case.setup, w, h, 3, 0, jitter=(0.2 / w, -0.3 / h), options=options(OPTION_CASES[opt]))
    worst = Worst()
    run_one(ctx, rt, case, w, h, frame, name=f"{scene}/{opt}", worst=worst, hits=(opt == "default"))
    worst.print(f"{scene}/{opt}")
    ctx.status()


@pytest.mark.parametrize("scene", ["cornell", "two", "sweep"])
def test_realtime_shading_matches_reference(scene, ctx, rt):
    case = CASES[scene]()
    w, h = 80, 45
    frame = scenes.make_frame(case.setup, w, h, 1, 0, jitter=(0.1 / w, 0.2 / h))
    worst = Worst()
    run_one(ctx, rt, case, w, h, frame, realtime=True, name=f"{scene}/realtime", worst=worst)
    worst.print(f"{scene}/realtime")
    ctx.status()


@pytest.mark.parametrize("w,h", [(1, 1), (33, 17), (17, 300), (200, 200)])
@pytest.mark.parametrize("scene", ["cornell", "sweep"])
def test_shapes_ragged_against_the_shading_tile(scene, w, h, ctx, rt):
    case = CASES[scene]()
    frame = scenes.make_frame(case.setup, w, h, 7, 0, jitter=(0.0, 0.1 / h))
    worst = Worst()
    run_one(ctx, rt, case, w, h, frame, name=f"{scene} {w}x{h}", worst=worst)
    worst.print(f"{scene} {w}x{h}")


@pytest.mark.parametrize("region", [(13, 9, 77, 50), (40, 31, 41, 76), (0, 5, 100, 6)])
def test_region_dispatch(region, ctx, rt):
    case = cornell_case()
    w, h = 100, 76
    frame = scenes.make_frame(case.setup, w, h, 2, 0, options=options(dict(debug=2)))
    worst = Worst()
    run_one(ctx, rt, case, w, h, frame, region=region, name=f"region {region}", worst=worst)
    worst.print(f"region {region}")


@pytest.mark.parametrize("strips", [(4, 3, 0), (4, 3, 1), (4, 3, 2), (8, 2, 0), (8, 2, 1)])
def test_strip_dispatch(strips, ctx, rt):
    case = two_material_case()
    w, h = 90, 70
    frame = scenes.make_frame(case.setup, w, h, 4, 0)
    worst = Worst()
    run_one(ctx, rt, case, w, h, frame, strips=strips, name=f"strips {strips}", worst=worst)
    worst.print(f"strips {strips}")


@pytest.mark.parametrize("half", [False, True])
def test_accumulation_is_the_running_mean_of_the_reference_frames(half, ctx, rt):
    case = material_sweep_case()
    w, h, n = 48, 40, 3
    ctx.set_render_options(1, half)
    try:
        r = case.renderer(rt, ctx, rt.PROGRESSIVE, w, h)
        sc, worst = ref_scene(case), Worst()
        mean = np.zeros((h, w, 3))
        jit = scenes.jitter_sequence(5, n, w, h)
        for s in range(n):
            frame = scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s])
            a = capture(ctx, r, frame)
            ys, xs, cols, ill, _, units = check_dispatch(a, sc, frame, w, h, False, worst=worst)
            prev = mean[ys, xs].astype(np.float32)
            mean[ys, xs] = sr.running_mean(prev, cols, s, half)
            pixel_check(f"frame {s}{' fp16' if half else ''}", stored(r.image(0), ys, xs), mean[ys, xs], ill, worst, half=half,
                        where=(ys, xs), unit=units / (s + 1))
            mean[ys, xs] = stored(r.image(0), ys, xs)  # the next frame accumulates onto what the target holds
        worst.print(f"accumulation half={half}")
    finally:
        ctx.set_render_options(1, False)


def test_aovs_match_reference(ctx, rt):
    case = material_sweep_case()
    w, h = 64, 48
    r = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h,
                    aovs=("direct", "indirect-diffuse", "indirect-specular", "albedo", "fresnel"))
    frame = scenes.make_frame(case.setup, w, h, 1, 0)
    worst = Worst()
    _, ys, xs, _, ill, aovs, _ = run_one(ctx, rt, case, w, h, frame, name="aovs", worst=worst, renderer=r)
    for name, (ref, unit) in aovs.items():
        pixel_check(f"AOV {name}", stored(r.aov(name), ys, xs), sr.clamp(ref), ill, worst, where=(ys, xs), unit=unit)
    worst.print("aovs")


def test_two_band_dispatch_matches_reference(ctx, rt):
    """At 640 x 512 an uncaptured dispatch runs as two pixel bands on two streams (pipeline.cu:921); a captured one runs as
    one band with the same image (test_gpu_stage_parity.py::test_capture_does_not_change_the_image).  The uncaptured image
    is held to the reference built from the captured dispatch of the same frame."""
    case = bunny_case(4)
    w, h = 640, 512
    frame = scenes.make_frame(case.setup, w, h, 0, 0)
    worst = Worst()
    _, ys, xs, cols, ill, _, units = run_one(ctx, rt, case, w, h, frame, name="captured 640x512", worst=worst, hits=False)
    r2 = case.renderer(rt, ctx, rt.PROGRESSIVE, w, h)
    r2.dispatch(frame)
    pixel_check("two-band k_resolve", stored(r2.image(0), ys, xs), sr.clamp(cols), ill, worst, where=(ys, xs), unit=units)
    worst.print("two-band")


def test_missing_hit_record_shades_with_record_zero(ctx, rt):
    """An instance without a hit record: the kernels shade its hits with record 0 and rt_get_status reports the error."""
    case = two_material_case()
    w, h = 64, 48
    r = case.renderer(rt, ctx, rt.PROGRESSIVE, w, h)
    prog = rt.Program(ctx, rt.PROGRESSIVE)
    for ray_type in range(2):  # instance 0 only: the ground (instance 1) hits record 2 >= n_recs
        prog.set_hit_record(ray_type, 0, r.blases[0].vb, r.blases[0].ib, case.materials[0])
    prog.set_env(case.env)
    r.program = prog
    frame = scenes.make_frame(case.setup, w, h, 1, 0)
    worst = Worst()
    a = capture(ctx, r, frame)
    assert (a.pr[a.ph["prim"] != T.NO_HIT] >= 2).any(), "no hit on the instance without a record"
    with pytest.raises(rt.RtError):
        ctx.status()
    ctx.status()  # reading the status clears it
    sc = ref_scene(case, n_instances_bound=1)
    ys, xs, cols, ill, _, units = check_dispatch(a, sc, frame, w, h, False, worst=worst)
    pixel_check("missing record k_resolve", stored(r.image(0), ys, xs), sr.clamp(cols), ill, worst, where=(ys, xs), unit=units)
    worst.print("missing record")
