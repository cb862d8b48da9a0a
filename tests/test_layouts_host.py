"""CPU-side checks of the models the layout tests derive from the synthetic one (other vertex counts, fewer output
joints): the packing logic reproduces the oracle on each of them when emulated in numpy, and the derived set covers
the blend-row layouts it is meant to cover (odd and even row-tile counts of the GEMMs, a mesh without a ragged last
vertex tile, a model without virtual joint rows).  `derive_model` is also what tests/test_gpu_layouts.py runs the
kernels on."""
import numpy as np
import pytest

from soccerplayershapepose_b200.engine import SMPLEngine
from soccerplayershapepose_b200.model_io import validate_model
from test_cabi_host import _check_packed_emulation

REGRESSORS = ("extra", "cocoplus", "h36m")
TILE_V = 32                  # vertices per skinning tile; the tile count is rounded up to a multiple of 4


def derive_model(base, V, regressors=REGRESSORS, picked=True):
    """A model with V vertices built from `base`: vertex i copies base vertex i % n0 (copies past the first n0 get a
    1 cm jitter of the template) with its shape directions, skinning weights and pose-corrective columns; the joint
    regressor and the chosen extra regressors keep the columns of those vertices and are renormalised (a row left
    empty gets a single 1.0); a regressor left out becomes a (0, V) array; the picked-vertex joints are the base ids
    mod V, or none.  Output joints: 24 + 21 * picked + the rows of the chosen regressors."""
    rng = np.random.default_rng(V)
    n0 = base["v_template"].shape[0]
    idx = np.arange(V) % n0
    jitter = (idx != np.arange(V))[:, None] * rng.standard_normal((V, 3)) * 0.01
    m = {"v_template": (base["v_template"][idx] + jitter).astype(np.float32),
         "shapedirs": np.ascontiguousarray(base["shapedirs"][idx]),
         "posedirs": np.ascontiguousarray(base["posedirs"].reshape(-1, n0, 3)[:, idx].reshape(-1, 3 * V)),
         "lbs_weights": np.ascontiguousarray(base["lbs_weights"][idx]),
         "parents": base["parents"],
         "faces": base["faces"][(base["faces"] < V).all(1)]}

    def restrict(R):
        R = R[:, idx].astype(np.float64)
        for r in np.nonzero(R.sum(1) == 0)[0]:
            R[r, r % V] = 1.0
        return (R / R.sum(1, keepdims=True)).astype(np.float32)

    m["J_regressor"] = restrict(base["J_regressor"])
    for k in REGRESSORS:
        key = "J_regressor_" + k
        m[key] = restrict(base[key]) if k in regressors else np.zeros((0, V), np.float32)
    m["extra_joints_idxs"] = (np.asarray(base["extra_joints_idxs"]) % V) if picked else np.zeros(0, np.int64)
    validate_model(m)
    return m


# (V, regressors, picked): output joints 90, 54, 45 or 24
DERIVED = [
    (1, REGRESSORS, True),
    (33, (), True),
    (33, (), False),
    (129, REGRESSORS, True),
    (1001, ("extra",), True),
    (6889, REGRESSORS, True),
    (6912, (), False),
    (10475, REGRESSORS, True),
]


@pytest.fixture(scope="module")
def derived(synthetic_model):
    return {spec: derive_model(synthetic_model, spec[0], spec[1], spec[2]) for spec in DERIVED}


def _njout(regressors, picked):
    return 24 + 21 * picked + sum({"extra": 9, "cocoplus": 19, "h36m": 17}[k] for k in regressors)


@pytest.mark.parametrize("spec", DERIVED, ids=lambda s: "V{}-{}j".format(s[0], _njout(s[1], s[2])))
def test_packed_emulation_on_derived_models(derived, spec):
    V, regressors, picked = spec
    model = derived[spec]
    eng = SMPLEngine(model, device=None)
    info = eng.info
    assert info.num_verts == V
    assert info.num_joints_out == 24 + len(model["extra_joints_idxs"]) + sum(
        model["J_regressor_" + k].shape[0] for k in REGRESSORS)
    assert info.num_joints_out == _njout(regressors, picked)
    _check_packed_emulation(eng, model)


def test_derived_set_covers_the_blend_row_layouts(derived):
    """The set must keep covering: odd and even row-tile counts of the CTA-pair GEMMs (an odd count leaves one tile
    of the last pair alone), a mesh whose vertex tiles have no ragged tail, odd vertex counts (the skinning kernels'
    element-wise row copies) and a model with no virtual joint rows (a joints-only GEMM over an empty row range)."""
    seen = {}
    for spec, model in derived.items():
        info = SMPLEngine(model, device=None).info
        V = spec[0]
        ntiles = -(-V // TILE_V)
        ntiles += (-ntiles) % 4
        row_tiles = info.num_blend_rows_padded // 128
        assert info.num_blend_rows_padded % 384 == 0
        assert info.num_blend_rows >= 3 * TILE_V * ntiles
        seen[spec] = (row_tiles, info.num_joints_out, info.num_blend_rows == 3 * TILE_V * ntiles)
    tiles = [t for t, _, _ in seen.values()]
    assert any(t % 2 for t in tiles) and any(t % 2 == 0 for t in tiles)
    assert any(s[0] % TILE_V == 0 for s in seen) and any(s[0] % TILE_V for s in seen)
    assert any(s[0] % 2 for s in seen)
    no_virtual = [s for s, (_, nj, empty) in seen.items() if empty]
    assert no_virtual and all(seen[s][1] == 24 for s in no_virtual)
    assert (6912, (), False) in no_virtual
    # the row-tile counts read off the packing (V, joints) -> tiles
    expect = {(1, 90): 12, (33, 45): 6, (33, 24): 3, (129, 90): 15, (1001, 54): 27, (6889, 90): 177,
              (6912, 24): 162, (10475, 90): 261}
    assert {(s[0], nj): t for s, (t, nj, _) in seen.items()} == expect
