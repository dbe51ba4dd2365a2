"""learn() from the reference's own input type (src/GraphicalModelLearning.jl:69-81): a column-major K x (N+1) matrix of
Float64 (readdlm, test/runtests.jl:71) or Int64 (`sample`, src/sampling.jl:54), through gml_b200_learn_pairwise_matrix /
gml_b200_learn_multibody_matrix: host-side threaded narrowing + validation, lambda computed by the library."""
import numpy as np
import pytest

import c_oracle as c
import gml_b200
from gml_b200 import B200, RISE, RPLE, logRISE, multiRISE

pytestmark = pytest.mark.gpu
FORMS = {"RISE": RISE, "logRISE": logRISE, "RPLE": RPLE}


@pytest.mark.parametrize("dtype", [np.float64, np.int64, np.float32, np.int32])
@pytest.mark.parametrize("name", ["a", "c", "mvt"])
def test_matrix_entry_equals_packed_entry_on_goldens(golden, name, dtype):
    # the histogram as the matrix entry receives it: exact in every dtype except float32, which rounds mvt's largest
    # count (35 712 921 > 2^24) by one -- the packed entry gets the same rounded count
    s = golden(f"{name}_samples.csv").astype(dtype).astype(np.float64)
    for form in FORMS.values():
        f = form(0.2, False) if name == "mvt" else form()
        packed = gml_b200.learn(s, f, B200(barrier_mu=1e-9))                      # row-major input -> packed entry
        mat, info = gml_b200.learn(np.asfortranarray(s.astype(dtype)), f, B200(barrier_mu=1e-9), return_info=True)
        assert np.array_equal(packed, mat)                                           # same bytes reach the same solver
        gold = golden(f"{name}_{type(f).__name__}_learned.csv")
        assert np.abs(mat - gold).max() <= (1e-4 if name == "mvt" else 2e-9)


def test_matrix_entry_row_range_of_a_taller_matrix_and_multibody(golden):
    s = golden("c_samples.csv")
    tall = np.asfortranarray(np.vstack([s, np.full((5, s.shape[1]), 7.0)]))      # ld = K + 5, junk rows below
    view = tall[:s.shape[0], :]
    assert not view.flags.f_contiguous
    a = gml_b200.learn_matrix(view, RISE(), B200())
    assert np.array_equal(a, gml_b200.learn(s, RISE(), B200()))
    m = gml_b200.learn_matrix(np.asfortranarray(s), multiRISE(0.2, True, 3), B200())
    ref = c.learn_multibody(s, 0.2, True, 3)
    assert m.terms.keys() == ref.keys() and max(abs(m[k] - ref[k]) for k in ref) <= 1e-9


def test_matrix_entry_validation():
    rng = np.random.default_rng(1)
    k, n = 3000, 5
    s = np.asfortranarray(np.concatenate([rng.integers(1, 9, size=(k, 1)), rng.choice([-1, 1], size=(k, n))], axis=1).astype(np.float64))
    gml_b200.learn_matrix(s, RISE(), B200())
    for bad_value in (0.0, 0.5, 2.0, -1.0000001, np.nan):
        bad = s.copy(order="F"); bad[1234, 3] = bad_value
        with pytest.raises(gml_b200.GMLB200Error) as e:
            gml_b200.learn_matrix(bad, RISE(), B200())
        assert e.value.code == 1
    badc = s.copy(order="F"); badc[7, 0] = 0.0
    with pytest.raises(gml_b200.GMLB200Error) as e:
        gml_b200.learn_matrix(badc, RISE(), B200())
    assert e.value.code == 1


def test_matrix_entry_large_multichunk_tensor_path():
    """N = 70 (tensor-core FISTA), K = 2.3e6 > one ingest chunk per column, Float64: equals the packed entry exactly and the
    oracle on two nodes; reports the ingest time."""
    rng = np.random.default_rng(3)
    n, k = 70, 2_300_001
    spins = rng.choice(np.array([-1, 1], dtype=np.int8), size=(n, k))
    spins[5] = spins[4] * np.where(rng.random(k) < 0.75, 1, -1).astype(np.int8)
    counts = np.ones(k)
    mat = np.empty((k, n + 1), dtype=np.float64, order="F")
    mat[:, 0] = counts
    mat[:, 1:] = spins.T
    m = B200(tol=1e-7)
    got, info = gml_b200.learn_matrix(mat, RISE(0.4, False), m, return_info=True)
    packed = gml_b200.learn_packed(counts, spins, RISE(0.4, False), B200(tol=1e-7))
    assert np.array_equal(got, packed)
    lam = gml_b200.regularizer_lambda(0.4, n, float(k))
    ref = c.learn_pairwise_packed(counts, spins, "RISE", lam, False, nodes=(4, 6))
    assert np.abs(got[4:6] - ref[4:6]).max() <= 1e-5
    print(f"ingest of {mat.nbytes / 1e9:.2f} GB float64: {info['h2d_ms']:.1f} ms ({mat.nbytes / 1e6 / info['h2d_ms']:.1f} GB/s of matrix)")
