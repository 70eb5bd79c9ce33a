"""Regenerates tests/golden/*.npz: seeded inputs and the oracle's outputs for them.

The reference itself cannot be built in this image (no Eigen, DESIGN.md section 5), so these vectors come from
oracle/clipper_oracle.c -- the restatement that tests/test_oracle_golden.py pins against every fixture the reference's
own tests hold.  They freeze that restatement: tests/test_oracle_golden.py::test_oracle_reproduces_golden_files fails if
the oracle's arithmetic ever drifts, and tests/test_gpu_parity.py::test_cuda_path_against_golden_files compares the
CUDA path with them on a B200.

usage:  python tests/golden/make_golden.py        (rewrites the .npz files)"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from clipper_b200 import datagen  # noqa: E402
from oracle.clipper_oracle import Oracle  # noqa: E402

CASES = {
    # name: (kind, m, rho, seed, invariant parameters)
    "euclid_m300": ("euclidean", 300, 0.90, 71, dict(sigma=0.01, epsilon=0.02, mindist=0.0)),
    "euclid_m900": ("euclidean", 900, 0.95, 72, dict(sigma=0.015, epsilon=0.05, mindist=0.0)),
    "euclid_mindist_m200": ("euclidean", 200, 0.80, 73, dict(sigma=0.02, epsilon=0.05, mindist=0.15)),
    "pointnormal_m400": ("pointnormal", 400, 0.90, 74, dict(sigp=0.5, epsp=0.5, sign=0.10, epsn=0.35)),
}


def run_case(kind, m, rho, seed, ip):
    prob = datagen.euclidean_problem(m, rho, seed) if kind == "euclidean" else datagen.pointnormal_problem(m, rho, seed)
    # keep the files small: only the points the associations touch
    A = prob["A"]
    used1, inv1 = np.unique(A[:, 0], return_inverse=True)
    used2, inv2 = np.unique(A[:, 1], return_inverse=True)
    D1 = np.asfortranarray(prob["D1"][:, used1]); D2 = np.asfortranarray(prob["D2"][:, used2])
    A = np.asfortranarray(np.stack([inv1, inv2], axis=1).astype(np.int32))
    o = Oracle()
    if kind == "euclidean":
        o.score_euclidean(D1, D2, A, **ip)
    else:
        o.score_pointnormal(D1, D2, A, **ip)
    cp, ri, val = o.get_csc(0)
    v = np.random.default_rng(seed + 1000).random(m)
    y, F = o.gradf(v, 0.75)
    s = o.solve(prob["u0"])
    return dict(kind=kind, D1=D1, D2=D2, A=A, u0=prob["u0"], param_names=np.array(sorted(ip)), param_values=np.array([ip[k] for k in sorted(ip)]),
                M_colptr=cp, M_rowidx=ri, M_val=val, v=v, d=0.75, gradf=y, Mv=o.matvec(v, 0), Cv=o.matvec(v, 1),
                nodes=s.nodes.astype(np.int32), score=s.score, u=s.u, ifinal=s.ifinal, n_evals=s.n_evals, n_inner=s.n_inner,
                d_final=s.d_final)


def load(name):
    z = np.load(os.path.join(HERE, name + ".npz"))
    out = {k: z[k] for k in z.files}
    out["params"] = dict(zip([str(k) for k in out.pop("param_names")], [float(x) for x in out.pop("param_values")]))
    out["kind"] = str(out["kind"])
    return out


if __name__ == "__main__":
    for name, (kind, m, rho, seed, ip) in CASES.items():
        r = run_case(kind, m, rho, seed, ip)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **r)
        print(name, "m", m, "nnz upper", len(r["M_val"]), "nodes", len(r["nodes"]), "F", r["score"], "evals", r["n_evals"])
