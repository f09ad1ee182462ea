"""The float64 shading reference (shade_reference.py) checked on its own, without a GPU: against the closed-form answers of
closed_form.py, and pixel by pixel against the oracle's renders when driven by the oracle's traversal.

The reference's rays are traced by the oracle with the flags of each ray kind.  Sampled directions are traced as the
reference evaluates them in float32 (numpy's sin / cos / pow in place of the oracle's), so that a secondary hit lies where
the oracle's own ray hit to within rounding; the shading along those rays is float64.  A rare pixel may still differ because
such a ray hit another triangle than the oracle's;
at least MIN_PIXELS_AGREE of the pixels must meet the per-pixel bound of the GPU check, and the rest are printed.
"""
import numpy as np
import pytest

import closed_form as cf
import shade_reference as sr
from dxrexperiments_b200 import scenes, types as T
from helpers import bunny_case, cornell_case, two_material_case

SHADOW_FLAGS = T.RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH | T.RAY_FLAG_SKIP_CLOSEST_HIT_SHADER
# The per-pixel bound of tests/test_gpu_shade_parity.py: a float32 chain of a few dozen correctly rounded operations and a
# few transcendental calls (a few ulp each) stays within ~1e-6 relative of the float64 value; 1e-5 leaves a factor 10 and
# still fails a 1e-4 relative change of one term.  The 1e-3 * mean|r| floor covers terms that cancel to near zero.
PIXEL_REL = 1e-5
PIXEL_FLOOR = 1e-3
# The oracle traces its own float32 samples (glibc's sinf / cosf / powf), the reference its float32 evaluation with numpy's:
# the two directions differ by a few ulp.  A uniform-hemisphere AO ray that grazes the surface, or a shadow ray that grazes a
# silhouette, can change its visibility on that, and a secondary hit near a light moves with the direction.  Measured on
# these scenes at 64 x 48: up to 0.75 % of the pixels in the uniform AO view, 0.3 % or fewer elsewhere, so 99 % rather than
# 99.9 %; the kernels themselves are held at the per-pixel bound on their own rays by tests/test_gpu_shade_parity.py.
MIN_PIXELS_AGREE = 0.99
CLOSED_FORM_REL = 1e-6


def rays32(origin, tmin, direction, tmax):
    r = np.zeros(len(tmax), T.RAY_DTYPE)
    r["origin"], r["tmin"], r["direction"], r["tmax"] = origin, tmin, direction, tmax
    return r


def oracle_frame(sc, fr, otlas, frame, w, h, realtime, threads=8):
    """Shade a whole frame with the reference, every ray traced by the oracle.  Returns (colour (h, w, 3) before the clamp,
    ill-conditioned mask (h, w)) — for realtime, colour is (out0, out1)."""
    js = 10.0 if realtime else 30.0
    import oracle
    prim_rays = oracle.primary_rays(frame, w, h, js)
    ho = otlas.trace(prim_rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES, threads=threads)
    hit = ho["primitive_index"] != T.NO_HIT
    pix = np.flatnonzero(hit)
    px, py = pix % w, pix // w
    ill = np.zeros(h * w, bool)
    # primary misses: the camera direction is the kernel's bit for bit (primary_ray in float32)
    miss = np.flatnonzero(~hit)
    _, dm = sr.primary_ray(fr, w, h, miss % w, miss // w, js, np.float64)
    _, dm32 = sr.primary_ray(fr, w, h, miss % w, miss // w, js, np.float32)
    miss_c = sr.miss_colour(sc, fr, dm, dm32)
    hh = ho[pix]
    P = sr.shade_primary(sc, fr, w, h, px, py, hh["t"], hh["bary"][:, 0], hh["bary"][:, 1], hh["primitive_index"],
                         2 * hh["instance_index"], realtime)
    ill[pix] |= P.ill
    pos32 = P.pos.astype(np.float32)
    vis0 = np.ones((P.nplanes, P.S), np.uint8)
    for k in range(P.nplanes):
        act = P.sh_tmax[k] >= 0
        if act.any():
            q = rays32(pos32[act], P.sh_tmin[k], P.sh_dir32[k][act], P.sh_tmax[k][act])
            vis0[k, act] = otlas.trace(q, SHADOW_FLAGS, threads=threads)["primitive_index"] == T.NO_HIT
    rad = [np.zeros((P.S, 3)), np.zeros((P.S, 3))]
    if P.nplanes == 2:
        for k in range(2):
            act = P.sec_tmax[k] >= 0
            if not act.any():
                continue
            q = rays32(pos32, P.sec_tmin, P.sec_dir32[k], np.where(act, P.sec_tmax[k], -1.0))
            sh = np.zeros(P.S, T.HIT_DTYPE)
            sh["primitive_index"] = T.NO_HIT
            sh[act] = otlas.trace(q[act], 0, threads=threads)
            Q = sr.shade_secondary(sc, fr, w, px, py, q["origin"], q["direction"], q["tmax"], sh["t"], sh["bary"][:, 0],
                                   sh["bary"][:, 1], sh["primitive_index"], 2 * sh["instance_index"], realtime)
            # the environment face of a direction the reference sampled itself is not the kernel's decision
            ill[pix[Q.kind == 1]] |= sr.env_face_ill_conditioned(q["direction"][Q.kind == 1].astype(np.float64))
            vis1 = np.ones((2, Q.hi.size), np.uint8)
            for j in range(2):
                a1 = Q.sh_tmax[j] >= 0
                if a1.any():
                    r1 = rays32(Q.pos32[a1], Q.sh_tmin, Q.sh_dir[j][a1], Q.sh_tmax[j][a1])
                    vis1[j, a1] = otlas.trace(r1, SHADOW_FLAGS, threads=threads)["primitive_index"] == T.NO_HIT
            rad[k] = sr.secondary_radiance(sc, fr, Q, vis1[0], vis1[1], realtime)
    out = sr.resolve(sc, fr, P, vis0, rad[0], rad[1])
    if realtime:
        imgs = []
        for c in (out.out0, out.out1):
            img = np.zeros((h * w, 3))
            img[pix] = c
            imgs.append(img)
        imgs[0][miss] = miss_c
        return (imgs[0].reshape(h, w, 3), imgs[1].reshape(h, w, 3)), ill.reshape(h, w)
    img = np.zeros((h * w, 3))
    img[pix] = out.color
    img[miss] = miss_c
    return img.reshape(h, w, 3), ill.reshape(h, w)


def pixel_errors(got, ref):
    """|g - r| / (|r| + PIXEL_FLOOR * mean|r|) per pixel (largest channel)."""
    ref = np.asarray(ref, np.float64)
    scale = np.abs(ref) + PIXEL_FLOOR * max(float(np.abs(ref).mean()), 1e-30)
    return (np.abs(np.asarray(got, np.float64) - ref) / scale).max(axis=-1)


def report(name, err, ok, limit):
    bad = np.argwhere(~ok)
    worst = float(err[ok].max()) if ok.any() else 0.0
    print(f"{name}: worst within-bound deviation {worst:.3e} (bound {limit:.0e}); {len(bad)} of {err.size} pixels outside")
    for yx in bad[:20]:
        print(f"  pixel x={yx[1]} y={yx[0]}: {err[tuple(yx)]:.3e}")


# ---------------------------------------------------------------------------------------------- closed forms
def _closed_form_scene(case):
    return sr.Scene(case.meshes, case.materials, case.env)


@pytest.mark.parametrize("make", cf.CASES, ids=lambda f: f.__name__)
def test_reference_reproduces_closed_form_radiance(make, orc):
    case = make()
    blases = [orc.Blas.from_mesh(m) for m in case.meshes]
    otlas = orc.Tlas(blases, [scenes.IDENTITY_3X4] * len(blases))
    frame = case.frame(0)
    img, ill = oracle_frame(_closed_form_scene(case), sr.Frame(frame), otlas, frame, case.w, case.h, case.realtime)
    if case.realtime:
        img, spec = img
        assert not sr.clamp(spec).any()
    got = sr.clamp(img)[case.mask]
    want = case.expected[case.mask]
    err = np.abs(got - want).max() / np.abs(want).max()
    print(f"{case.name}: max deviation {err:.3e} relative to the largest expected value")
    assert err <= CLOSED_FORM_REL, f"{case.name}: {err:.3e}"


def test_reference_uniform_furnace_converges(orc):
    """Uniform hemisphere sampling is not a constant of the random numbers: its 48-spp mean lands on the closed form."""
    c = cf.furnace(w=48, h=36, spp=48, uniform=True)
    blases = [orc.Blas.from_mesh(m) for m in c.meshes]
    otlas = orc.Tlas(blases, [scenes.IDENTITY_3X4])
    sc = _closed_form_scene(c)
    acc = np.zeros((c.h, c.w, 3))
    for s in range(c.spp):
        frame = c.frame(s)
        img, _ = oracle_frame(sc, sr.Frame(frame), otlas, frame, c.w, c.h, False)
        acc += sr.clamp(img)
    ratio = (acc / c.spp)[c.mask].mean(axis=0) / c.expected[c.mask].mean(axis=0)
    np.testing.assert_allclose(ratio, 1.0, atol=5e-3)


# ---------------------------------------------------------------------------------------------- the oracle's renders
OPTION_CASES = {"default": {}, "uniform_hemisphere": dict(cosineHemisphereSampling=0), "no_indirect_diffuse": dict(noIndirectDiffuse=1),
                "indirect_diffuse_only": dict(showIndirectDiffuseOnly=1), "indirect_specular_only": dict(showIndirectSpecularOnly=1),
                "ambient_occlusion_only": dict(showAmbientOcclusionOnly=1),
                "ambient_occlusion_uniform": dict(showAmbientOcclusionOnly=1, cosineHemisphereSampling=0),
                "albedo_only": dict(showGBufferAlbedoOnly=1), "direct_only": dict(showDirectLightingOnly=1),
                "fresnel_only": dict(showFresnelTerm=1), "one_light_sampling": dict(debug=2),
                "environment_strength": dict(environmentStrength=2.5)}
SCENES = {"cornell": (cornell_case, 64, 48), "bunny": (lambda: bunny_case(3), 64, 40), "two": (two_material_case, 60, 44)}


def options(overrides):
    o = scenes.default_options()
    for k, v in overrides.items():
        setattr(o, k, v)
    return o


def check_against_oracle(case, orc, frame, w, h, realtime, name):
    otlas, recs = case.oracle(orc)
    sc = sr.Scene(case.meshes, case.materials, case.env)
    img, ill = oracle_frame(sc, sr.Frame(frame), otlas, frame, w, h, realtime)
    if realtime:
        want = orc.render_realtime(otlas, recs, case.env, frame, w, h, threads=8)
        pairs = [(f"{name} out0", img[0], want[0]), (f"{name} out1", img[1], want[1])]
    else:
        acc = np.zeros((h, w, 4), np.float32)
        orc.render_progressive(otlas, recs, case.env, frame, w, h, acc, threads=8)
        pairs = [(name, img, acc)]
    for label, ref, got in pairs:
        err = pixel_errors(got[..., :3], sr.clamp(ref))
        ok = (err <= PIXEL_REL) | ill
        report(label, err, ok, PIXEL_REL)
        assert ok.mean() >= MIN_PIXELS_AGREE, f"{label}: {int((~ok).sum())} pixels outside the bound"


@pytest.mark.parametrize("scene", sorted(SCENES))
@pytest.mark.parametrize("opt", sorted(OPTION_CASES))
def test_reference_matches_oracle_progressive(scene, opt, orc):
    make, w, h = SCENES[scene]
    case = make()
    frame = scenes.make_frame(case.setup, w, h, 5, 0, jitter=(0.3 / w, -0.2 / h), options=options(OPTION_CASES[opt]))
    check_against_oracle(case, orc, frame, w, h, False, f"{scene}/{opt}")


@pytest.mark.parametrize("scene", sorted(SCENES))
def test_reference_matches_oracle_realtime(scene, orc):
    make, w, h = SCENES[scene]
    case = make()
    frame = scenes.make_frame(case.setup, w, h, 2, 0, jitter=(0.1 / w, 0.2 / h))
    check_against_oracle(case, orc, frame, w, h, True, f"{scene}/realtime")


def test_rng_stream_matches_oracle(orc):
    """The vectorised LCG of the reference draws the oracle's numbers in the oracle's order."""
    rng = sr.Rng(np.array([0, 1, 77, 4095], np.uint32), 9)
    seeds = [orc.init_rand(p, 9) for p in (0, 1, 77, 4095)]
    for _ in range(5):
        got = rng.draw()
        for i in range(4):
            v, seeds[i] = orc.next_rand(seeds[i])
            assert got[i] == v
