"""Pins the CPU oracle against every fixture the reference's own tests/examples hold for the
hot path (SURVEY 8c).  No GPU, no product code."""
import numpy as np
import pytest

import fixtures as fx
from oracle import clipper_oracle as orc


def test_toy_affinity_matches_reference_literal():
    # reference test/affinity_test.cpp:55-107
    model, data = fx.toy_problem()
    o = orc.Oracle()
    o.score_euclidean(model, data)
    A = o.get_initial_associations()
    assert A.shape == (12, 2)
    for i in range(4):
        for j in range(3):
            assert A[i * 3 + j, 0] == i and A[i * 3 + j, 1] == j  # :66-72
    M, C = o.get_affinity_matrix(), o.get_constraint_matrix()
    assert np.array_equal(np.diag(M), np.ones(12))  # :83
    assert np.array_equal(M, M.T) and np.array_equal(C, C.T)  # :86-87
    assert np.array_equal(M, C)  # :91
    assert np.array_equal(M, fx.MTRUE_12)  # :94-107


# The reference test draws u0 from std::random_device.  CLIPPER is a local method: on this graph
# ~6 % of uniform random starts (e.g. numpy seeds 1, 25, 29) converge to one of the 2-cliques
# {1,3} / {3,10} instead of the maximum clique, i.e. the reference test itself is (rarely) flaky.
# The seeds below are starts for which the reference's expected answer is reached.
@pytest.mark.parametrize("seed", [0, 2, 3, 4, 5, 6, 7, 8])
def test_toy_inliers_for_seeded_u0(seed):
    # reference test/clipper_test.cpp:56-66 (random u0 there; seeded here)
    model, data = fx.toy_problem()
    o = orc.Oracle()
    o.score_euclidean(model, data)
    o.solve(np.random.default_rng(seed).random(12))
    Ain = o.get_selected_associations()
    assert Ain.shape[0] == 3
    assert sorted(map(tuple, Ain.tolist())) == [(0, 0), (1, 1), (2, 2)]


def test_get_set_roundtrip_dense_and_sparse():
    # reference test/clipper_test.cpp:115-124 and :181-196 (the getter/setter part)
    model, data = fx.toy_problem()
    o = orc.Oracle()
    o.score_euclidean(model, data)
    M, C = o.get_affinity_matrix(), o.get_constraint_matrix()
    o2 = orc.Oracle()
    o2.set_matrix_data(M, C)
    assert np.array_equal(o2.get_affinity_matrix(), M) and np.array_equal(o2.get_constraint_matrix(), C)
    cpM, riM, vM = o.get_csc(0)
    cpC, riC, vC = o.get_csc(1)
    o3 = orc.Oracle()
    o3.set_sparse_upper(12, cpM, riM, vM, cpC, riC, vC)
    assert np.array_equal(o3.get_affinity_matrix(), M)
    u0 = np.full(12, 0.5)
    assert o2.solve(u0).nodes.tolist() == o.solve(u0).nodes.tolist() == o3.solve(u0).nodes.tolist()


def test_m20_weighted_problem():
    # reference test/sdp_test.cpp:17-57: setMatrixData + solve() must run; the reference asserts
    # nothing, the strongest cluster of this matrix is the pair {5,12} (weight .9927) inside the
    # DSD answer {3,5,12,14,15} of test/dsd_test.cpp:15.
    M, C = fx.m20()
    o = orc.Oracle()
    o.set_matrix_data(M, C)
    s = o.solve(np.full(20, 1.0))
    assert set(s.nodes.tolist()) <= set(fx.DSD_NODES_20)
    u = s.u
    assert abs(u @ u - 1.0) < 1e-12 and (u >= 0).all()
    # objective equals u' Md u for the final u (clipper.cpp:220)
    y, F = o.gradf(u, s.d_final)
    assert abs(F - s.score) <= 1e-9 * max(1.0, abs(s.score)) or s.ifinal >= 0


def test_planecloud_pointnormal_known_answer():
    # reference examples/matlab/ex3_planecloud.m:18-33,79-91 -- Agt = [1 4; 2 3; 3 2] (1-based)
    D1, D2, Agt, pp = fx.planecloud()
    o = orc.Oracle()
    o.score_pointnormal(D1, D2, None, **pp)
    o.solve(np.full(16, 1.0))
    Ain = o.get_selected_associations()
    assert sorted(map(tuple, Ain.tolist())) == sorted(map(tuple, Agt.tolist()))


def test_k2ij_enumerates_upper_triangle():
    # reference src/utils.cpp:87-97
    n = 37
    k = 0
    for i in range(n):
        for j in range(i + 1, n):
            assert orc.k2ij(k, n) == (i, j)
            k += 1


def test_find_k_largest_tie_rule():
    # reference src/utils.cpp:33-55, SURVEY 8a K6: x=[5,5,5,7], k=2 -> [3,1]
    assert orc.find_k_largest(np.array([5.0, 5, 5, 7]), 2).tolist() == [3, 1]
    assert orc.find_k_largest(np.array([1.0, 3, 2]), 0).tolist() == []
    x = np.array([0.1, 0.9, 0.5, 0.7, 0.3])
    assert orc.find_k_largest(x, 3).tolist() == [1, 3, 2]
    assert orc.find_above(x, 0.4).tolist() == [1, 2, 3]


def test_pointnormal_nan_is_zero():
    # SURVEY H3: |dot| > 1 by rounding -> acos NaN -> score 0, not clamped
    a = np.array([0, 0, 0, 1.0, 0, 0]); b = np.array([1.0, 0, 0, 1.0 + 1e-12, 0, 0])
    assert orc.pointnormal(a, b, a, b) == 0.0


def test_mindist():
    # reference src/invariants/euclidean_distance.cpp:23-25
    ai, aj = np.array([0.0, 0, 0]), np.array([0.05, 0, 0])
    assert orc.euclidean(ai, aj, ai, aj, mindist=0.1) == 0.0
    assert orc.euclidean(ai, aj, ai, aj, mindist=0.0) == 1.0


# ------------------------------------------------------------------------------------------
# committed golden files (tests/golden/*.npz, written by tests/golden/make_golden.py)
# ------------------------------------------------------------------------------------------
def _golden_cases():
    import glob
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(here, "*.npz")) if not os.path.basename(p).startswith("bun10k"))


@pytest.mark.parametrize("name", _golden_cases())
def test_oracle_reproduces_golden_files(name):
    """the oracle is the pin for everything the reference's tests do not observe (solver trajectory, mat-vec):
    freeze it -- same inputs must give bit-identical scores, mat-vec, objective and iterate"""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden
    from oracle.clipper_oracle import Oracle
    g = make_golden.load(name)
    o = Oracle()
    if g["kind"] == "euclidean":
        o.score_euclidean(g["D1"], g["D2"], g["A"], **g["params"])
    else:
        o.score_pointnormal(g["D1"], g["D2"], g["A"], **g["params"])
    cp, ri, val = o.get_csc(0)
    assert np.array_equal(cp, g["M_colptr"]) and np.array_equal(ri, g["M_rowidx"]) and np.array_equal(val, g["M_val"])
    y, _ = o.gradf(g["v"], float(g["d"]))
    assert np.array_equal(y, g["gradf"]) and np.array_equal(o.matvec(g["v"], 0), g["Mv"]) and np.array_equal(o.matvec(g["v"], 1), g["Cv"])
    s = o.solve(g["u0"])
    assert s.nodes.tolist() == g["nodes"].tolist() and s.score == float(g["score"]) and np.array_equal(s.u, g["u"])
    assert (s.ifinal, s.n_evals, s.n_inner) == (int(g["ifinal"]), int(g["n_evals"]), int(g["n_inner"]))


def test_dsd_goldberg_known_answers():
    # reference test/dsd_test.cpp:15,38-43 (whole graph) and :49,72-79 (search restricted to S)
    M, _ = fx.m20()
    assert orc.dsd_solve(M) == fx.DSD_NODES_20
    assert orc.dsd_solve(M, [0, 1, 3, 5, 7, 12, 14, 15, 19]) == fx.DSD_NODES_20
    # a 2-node subset: the densest subgraph of an edge is the edge
    assert orc.dsd_solve(M, [5, 12]) == [5, 12]


def test_dsd_rounding_in_solve():
    # Rounding::DSD (clipper.cpp:294-300) = dsd::solve(M_, support(u)): the nodes are a subset of support(u) and,
    # on a seeded synthetic problem, exactly the densest subgraph of the support's sub-matrix
    from clipper_b200 import datagen
    prob = datagen.euclidean_problem(300, 0.85, 99)
    o = orc.Oracle(orc.default_params(rounding=orc.DSD))
    o.score_euclidean(prob["D1"], prob["D2"], prob["A"], sigma=0.015, epsilon=0.05)
    s = o.solve(prob["u0"])
    supp = orc.find_above(s.u, 0.0)
    assert set(s.nodes.tolist()) <= set(supp.tolist()) and len(s.nodes) >= 2
    assert s.nodes.tolist() == orc.dsd_solve(o.get_affinity_matrix(), supp)
    # the product's own host DSD (dense Dinic on the support sub-block, clp_host_utils.cpp) agrees with the restatement
    import clipper_b200 as clp
    assert clp.dsd.solve(o.get_affinity_matrix(), supp) == s.nodes.tolist()


# SHA-256 of the vertex payload of the reference's examples/data/bun10k.ply (the 119 904 bytes after its 235-byte
# header: 9992 x (float32 x, y, z), little-endian), taken from the reference tree at e514dc29
BUN10K_PLY_VERTEX_SHA256 = "0d41d0c866eb84790eb4e3943149fe8beabb8a2d3c2f441a98d180d7cf0759fb"


def test_bunny_fixture_matches_ply():
    # the fixture holds exactly the vertex payload of the reference's bun10k.ply
    import hashlib
    from clipper_b200 import datagen
    z = np.load(datagen.BUNNY_FIXTURE)["xyz"]
    assert z.shape == (9992, 3) and z.dtype == np.float32
    assert hashlib.sha256(z.astype("<f4").tobytes()).hexdigest() == BUN10K_PLY_VERTEX_SHA256
    c = datagen.make_cloud()
    assert c.shape == (3, 9992) and abs((c.max(axis=1) - c.min(axis=1)).max() - 1.0) < 1e-12
