"""CPU: the AOV reference the GPU tests compare against (tests/aov_reference.py) agrees with closed-form answers and with
the oracle's own shading path, so that a GPU failure points at the GPU."""
import numpy as np

import aov_reference
from closed_form import const_env
from dxrexperiments_b200 import scenes
from helpers import bunny_case, cornell_case, two_material_case


def test_reference_normal_of_a_plane(orc):
    w, h = 96, 64
    case, on, off = aov_reference.plane_case(w, h)
    otlas, recs = case.oracle(orc)
    frames = [scenes.make_frame(case.setup, w, h, s, s) for s in range(3)]
    n = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, frames, w, h, names=("normal",))["normal"]
    aov_reference.check_plane_normals(n, on, off)


def test_reference_normal_coverage_matches_the_oracle_hits(orc):
    """Under an environment of a colour no material has, the oracle's albedo view shows that colour exactly on the primary
    misses: the normal reference must have coverage 0 there and 1 everywhere else, with unit normals on the hits."""
    for case in (cornell_case(), two_material_case(), bunny_case(3)):
        case.env = const_env((5.0, 5.0, 5.0))
        w, h = 64, 48
        otlas, recs = case.oracle(orc)
        f = scenes.make_frame(case.setup, w, h, 0, 0, jitter=(0.2 / w, -0.1 / h))
        ref = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, [f], w, h, names=("albedo", "normal"))
        miss = np.all(ref["albedo"][..., :3] == 5.0, axis=-1)
        assert miss.any() and not miss.all()
        np.testing.assert_array_equal(ref["normal"][..., 3], np.where(miss, 0.0, 1.0).astype(np.float32))
        hit = ~miss
        np.testing.assert_allclose(np.linalg.norm(ref["normal"][hit][:, :3], axis=-1), 1.0, atol=1e-6)
