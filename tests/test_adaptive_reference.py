"""CPU: the restatement of adaptive sampling (tests/adaptive_reference.py) that the GPU is held to has the update rule's
exact properties, and at the same total number of samples an adaptive render is closer to 1024 spp than a uniform one."""
import numpy as np
import pytest

import adaptive_reference as ar
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from helpers import cornell_case, two_material_case

F = np.float32

# Adaptive (threshold 0.1, floor 0.1, min 8, update every 4 dispatches, at most 256 samples) against a uniform frame with
# the same total samples (sum of n_p, rounded to whole spp), both against 1024 spp, jitter-free 96 x 96.  Measured with
# this restatement: rel RMSE ratio 0.948 on Cornell and 0.814 on two-material; the luminance relMSE ratio (the measure
# the relative-error rule targets) 0.834 and 0.632.
QUALITY = {"cornell": dict(rmse=0.948, rmse_bound=1.0, relmse=0.834, relmse_bound=0.9),
           "two-material": dict(rmse=0.814, rmse_bound=0.9, relmse=0.632, relmse_bound=0.72)}


def state(counts, m1, m2):
    counts = np.asarray(counts, np.uint32)
    return counts, np.stack([np.asarray(m1, F), np.asarray(m2, F)], axis=-1)


def test_defaults_match_the_header():
    d = T.adaptive_defaults()
    assert (round(d.threshold, 6), round(d.floor, 6), d.min_samples, d.max_samples) == (0.1, 0.1, 8, 1024)


def test_update_is_monotone_and_never_clears_the_bit():
    rng = np.random.default_rng(1)
    h, w = 23, 31
    counts = rng.integers(0, 40, (h, w)).astype(np.uint32)
    counts[rng.random((h, w)) < 0.2] |= ar.CONVERGED
    m1 = rng.random((h, w)).astype(F)
    m2 = (m1 * m1 + rng.random((h, w)).astype(F) * F(0.01)).astype(F)
    c, m = state(counts, m1, m2)
    prev = c
    for thr in (0.0, 0.02, 0.05, 0.2, 10.0):
        out, active = ar.update(prev, m, thr, 0.1, 4, 1000)
        assert np.all(out[(prev & ar.CONVERGED) != 0] & ar.CONVERGED), "a converged pixel was reopened"
        assert np.array_equal(out & ar.COUNT_MASK, prev & ar.COUNT_MASK), "the update changed a count"
        assert active == int(((out & ar.CONVERGED) == 0).sum())
        prev = out


def test_max_samples_caps_whatever_the_error():
    counts, m = state(np.array([[9, 10, 11]]), [[1, 1, 1]], [[100, 100, 100]])
    out, active = ar.update(counts, m, 0.0, 0.1, 2, 10)
    assert ((out & ar.CONVERGED) != 0).tolist() == [[False, True, True]]
    assert active == 1


def test_min_samples_holds_a_zero_variance_pixel():
    counts, m = state(np.full((3, 3), 5), np.ones((3, 3)), np.ones((3, 3)))
    out, _ = ar.update(counts, m, 0.01, 0.1, 6, 100)
    assert not np.any(out & ar.CONVERGED)
    out, active = ar.update(counts, m, 0.01, 0.1, 5, 100)
    assert np.all(out & ar.CONVERGED) and active == 0, "zero variance at min_samples converges"


@pytest.mark.parametrize("n", [0, 1])
def test_fewer_than_two_samples_stay_active(n):
    counts, m = state(np.full((2, 2), n), np.zeros((2, 2)), np.zeros((2, 2)))
    out, active = ar.update(counts, m, 1e30, 0.1, 1, 100)
    assert active == 4 and not np.any(out & ar.CONVERGED)


def test_nan_moments_never_pass():
    counts, m = state(np.full((1, 1), 8), [[np.nan]], [[np.nan]])
    assert ar.update(counts, m, 1e30, 0.1, 1, 100)[1] == 1


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (6, 1), (5, 8), (9, 4)])
def test_one_pixel_dilation_at_edges_and_corners(shape):
    h, w = shape
    for y in range(h):
        for x in range(w):
            counts, m = state(np.full((h, w), 8), np.ones((h, w)), np.ones((h, w)))
            counts[y, x] = 1  # sigma = inf: this pixel and its 3 x 3 neighbours inside the image stay active
            out, active = ar.update(counts, m, 0.01, 0.1, 2, 100)
            want = np.zeros((h, w), bool)
            want[max(y - 1, 0):y + 2, max(x - 1, 0):x + 2] = True
            assert np.array_equal((out & ar.CONVERGED) == 0, want), (y, x)
            assert active == int(want.sum())


def test_relative_error_rule():
    # n = 5, m1 = 2, m2 = 4.04: sigma = sqrt(0.04 / 4) = 0.1, e = 0.1 / 2.1
    counts, m = state([[5]], [[2.0]], [[4.04]])
    e = ar.relative_error(counts, m, 0.1)[0, 0]
    want = np.sqrt(np.fmax(F(0), F(4.04) - F(2.0) * F(2.0)) / F(4)) / (F(2.0) + F(0.1))
    assert e == want
    assert ar.update(counts, m, float(want), 0.1, 2, 100)[1] == 0
    assert ar.update(counts, m, float(np.nextafter(want, F(0))), 0.1, 2, 100)[1] == 1


def test_compose_without_updates_is_the_running_mean():
    rng = np.random.default_rng(3)
    K, h, w = 7, 5, 6
    frames = rng.random((K, h, w, 4)).astype(F)
    frames[..., 3] = 1
    res = ar.compose(frames)
    acc = np.zeros((h, w, 4), F)
    for k in range(K):  # write_pixel's running mean with accumCount = k
        acc = (F(k) * acc + frames[k]) / F(k + 1)
    np.testing.assert_array_equal(res["beauty"], acc)
    assert np.all(res["counts"] == K)


def test_converged_pixels_stop_changing():
    rng = np.random.default_rng(4)
    K, h, w = 12, 6, 6
    frames = rng.random((K, h, w, 4)).astype(F)
    frames[:, :3, :] = frames[0, :3, :]  # the top half is constant: zero variance
    res = ar.compose(frames, schedule=ar.every(4, (0.01, 0.1, 4, 100), K))
    n = res["counts"] & ar.COUNT_MASK
    assert np.all(n[:2] == 4), "interior constant rows converge at the first update"
    assert np.all(n[3:] == K)
    assert res["active"][0] == 4 * w


def stack(case, w, h, first, count, orc):
    otlas, recs = case.oracle(orc)
    out = np.zeros((count, h, w, 4), F)
    for k in range(count):
        frame = scenes.make_frame(case.setup, w, h, first + k, 0, jitter=(0.0, 0.0))
        orc.render_progressive(otlas, recs, case.env, frame, w, h, out[k], threads=8)
    return out


def quality(case, orc, w=96, h=96, K=256):
    """(adaptive / uniform rel RMSE, adaptive / uniform relMSE, spp) at the same total samples, against 1024 spp."""
    ref = stack(case, w, h, 0, 1024, orc).mean(axis=0, dtype=np.float64).astype(F)
    frames = stack(case, w, h, 5000, K, orc)  # other random numbers than the reference's
    res = ar.run_until_converged(frames, (0.1, 0.1, 8, K), 4)
    spp = float((res["counts"] & ar.COUNT_MASK).sum()) / (w * h)
    uniform = frames[:max(1, int(round(spp)))].mean(axis=0, dtype=np.float64).astype(F)
    a = res["beauty"]
    return (rel_rmse(a[..., :3], ref[..., :3]) / rel_rmse(uniform[..., :3], ref[..., :3]),
            ar.rel_mse(a, ref) / ar.rel_mse(uniform, ref), spp)


@pytest.mark.parametrize("name", ["cornell", "two-material"])
def test_quality_on_the_oracle(orc, name):
    case = cornell_case() if name == "cornell" else two_material_case()
    r_rmse, r_relmse, spp = quality(case, orc)
    print(f"{name}: {spp:.1f} spp, adaptive / uniform rel RMSE {r_rmse:.3f}, relMSE {r_relmse:.3f}")
    q = QUALITY[name]
    assert r_rmse <= q["rmse_bound"], r_rmse
    assert r_relmse <= q["relmse_bound"], r_relmse
