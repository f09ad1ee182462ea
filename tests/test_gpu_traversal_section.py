"""The traversal section (BVH2 wide nodes, 4-wide nodes, the root box in rt_ext_header) derived on the CPU from the
reference blob of the same build and compared bit for bit, for every fit path of the build:

* PREFER_FAST_BUILD without update caches (hierarchy emission and fit in one bottom-up pass);
* the staged builds with treelet passes or ALLOW_UPDATE (block-local fit plus the global climb of its exits);
* PERFORM_UPDATE refits of a bottom-level build, and top-level builds and updates (the one-thread-per-leaf climb).

The 4-wide rule restated here: start from the node's two children; twice, open the internal child whose half extents
have the largest area (hx*hy + hy*hz) + hz*hx (float32, in that order; the library is built with -fmad=false), the
lower slot winning a tie; the opened child's left child takes its slot and its right child is appended.  Empty slots
are {0, 0, 0, RT_WIDE4_EMPTY}, {-1, -1, -1, 0}.
"""
import numpy as np
import pytest

from dxrexperiments_b200 import scenes, types as T

pytestmark = pytest.mark.gpu

UPD = T.BUILD_FLAG_ALLOW_UPDATE
FAST_BUILD = T.BUILD_FLAG_PREFER_FAST_BUILD
WIDE4_EMPTY = 0x7FFFFFFF
SIZES = [255, 256, 257, 511, 513, 4097, 300_000]


def _nodes(acc) -> np.ndarray:
    """The reference AABBNodes of the blob as (2n-1, 8) words: {center, flags}, {halfDim, right}."""
    return acc.blob()[16:16 + 32 * (2 * acc.n - 1)].view(np.uint32).reshape(-1, 8)


def _ref(node: np.ndarray, n_internal: int) -> np.ndarray:
    return np.where(node >= n_internal, T.LEAF_FLAG | (node - n_internal), node).astype(np.uint32)


def _expected_wide(nodes: np.ndarray, n: int) -> np.ndarray:
    """wide[p] = {left center, lref}, {left half, rref}, {right center, 0}, {right half, 0}."""
    n_int = n - 1
    left, right = nodes[:n_int, 3] & 0x00FFFFFF, nodes[:n_int, 7]
    out = np.zeros((n_int, 16), np.uint32)
    out[:, 0:3], out[:, 3] = nodes[left, 0:3], _ref(left, n_int)
    out[:, 4:7], out[:, 7] = nodes[left, 4:7], _ref(right, n_int)
    out[:, 8:11] = nodes[right, 0:3]
    out[:, 12:15] = nodes[right, 4:7]
    return out


def _expected_wide4(wide: np.ndarray) -> np.ndarray:
    m = wide.shape[0]
    rows = np.arange(m)
    ref = np.full((m, 4), WIDE4_EMPTY, np.uint32)
    ctr = np.zeros((m, 4, 3), np.uint32)
    half = np.zeros((m, 4, 3), np.uint32)
    ref[:, 0], ctr[:, 0], half[:, 0] = wide[:, 3], wide[:, 0:3], wide[:, 4:7]
    ref[:, 1], ctr[:, 1], half[:, 1] = wide[:, 7], wide[:, 8:11], wide[:, 12:15]
    cnt = np.full(m, 2)
    for _ in range(2):
        h = half.view(np.float32)
        area = (h[..., 0] * h[..., 1] + h[..., 1] * h[..., 2]) + h[..., 2] * h[..., 0]
        best, best_area = np.full(m, -1), np.full(m, np.float32(-1.0), np.float32)
        for k in range(4):
            take = (k < cnt) & ((ref[:, k] & T.LEAF_FLAG) == 0) & (area[:, k] > best_area)
            best = np.where(take, k, best)
            best_area = np.where(take, area[:, k], best_area)
        r = rows[best >= 0]
        if r.size == 0:
            break
        b, c = best[r], cnt[r]
        child = wide[ref[r, b]]
        ref[r, b], ctr[r, b], half[r, b] = child[:, 3], child[:, 0:3], child[:, 4:7]
        ref[r, c], ctr[r, c], half[r, c] = child[:, 7], child[:, 8:11], child[:, 12:15]
        cnt[r] += 1
    out = np.zeros((m, 4, 8), np.uint32)
    out[:, :, 0:3], out[:, :, 3], out[:, :, 4:7] = ctr, ref, half
    empty = np.arange(4)[None, :] >= cnt[:, None]
    out[empty] = np.array([0, 0, 0, WIDE4_EMPTY, *np.float32([-1, -1, -1]).view(np.uint32), 0], np.uint32)
    return out.reshape(m, 32)


def _check(acc):
    n = acc.n
    nodes = _nodes(acc)
    sec = acc.traversal_section()
    if n > 1:
        wide = _expected_wide(nodes, n)
        np.testing.assert_array_equal(sec["wide"], wide, err_msg="wide")
        np.testing.assert_array_equal(sec["wide4"], _expected_wide4(wide), err_msg="wide4")
    # the root box (rt_ext_header words 8-10 and 12-14): reference node 0 (the root, or the only leaf when n = 1)
    hdr = acc.ext_header()
    np.testing.assert_array_equal(hdr[8:11], nodes[0, 0:3], err_msg="root center")
    np.testing.assert_array_equal(hdr[12:15], nodes[0, 4:7], err_msg="root half")


def _soup(n):
    return scenes.triangle_soup(n, seed=7000 + n, extent=30.0, edge=1.0)


@pytest.mark.parametrize("n", [1, 2, 3] + SIZES)
@pytest.mark.parametrize("flags", [FAST_BUILD, 0, T.BUILD_FLAG_PREFER_FAST_TRACE, FAST_BUILD | UPD],
                         ids=["fused", "local_default", "local_fast_trace", "local_allow_update"])
def test_blas_build_traversal_section(n, flags, ctx):
    acc = ctx.build_blas_from_mesh(_soup(n), build_flags=flags)
    ctx.status()
    _check(acc)


@pytest.mark.parametrize("n", [1, 2] + SIZES)
def test_blas_refit_traversal_section(n, ctx):
    mesh = _soup(n)
    acc = ctx.build_blas_from_mesh(mesh, build_flags=UPD)
    rng = np.random.Generator(np.random.PCG64(n))
    moved = mesh.vertices.copy()
    moved["position"] += rng.uniform(-0.5, 0.5, size=moved["position"].shape).astype(np.float32)
    vb = ctx.upload(moved)
    ctx.update_blas(acc, [dict(vertices=vb, vertex_count=moved.shape[0], stride=24, indices=acc.ib, index_count=mesh.indices.size,
                               index_format=32)])
    ctx.status()
    _check(acc)


@pytest.fixture(scope="module")
def blases(ctx):
    return [ctx.build_blas_from_mesh(scenes.icosphere(1)), ctx.build_blas_from_mesh(_soup(500))]


@pytest.mark.parametrize("n", [1, 2, 50, 255, 256, 257, 1000, 4097])
def test_tlas_build_and_update_traversal_section(n, ctx, blases):
    inst = [blases[i % 2] for i in range(n)]
    acc = ctx.build_tlas(inst, scenes.random_rigid_transforms(n, seed=n), build_flags=UPD)
    ctx.status()
    _check(acc)
    ctx.update_tlas(acc, scenes.random_rigid_transforms(n, seed=n + 1))
    ctx.status()
    _check(acc)
