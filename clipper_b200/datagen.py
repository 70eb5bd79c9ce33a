"""Seeded synthetic association problems for tests and bench.py.

Mirrors the reference's benchmark generator (reference benchmarks/main.cpp:156-167 and
benchmarks/bm_utils.cpp:111-143,277-349) but deterministic and without its third-party
dependencies (nanoflann kd-tree, tinyply):

  * cloud: the reference's own benchmark cloud, examples/data/bun10k.ply (9992 float32 points), scaled like
    scale_to_cube(1) (main.cpp:156-160), read from its lossless fixture tests/golden/bun10k_points.npz
    (written by tests/golden/make_bunny_fixture.py); a synthetic bumpy closed surface of the same size only
    if the fixture is missing or another point count is asked for;
  * view 2: D2 = D1 + eta, eta ~ N(0, sigma^2 I3) rejection-truncated to |eta| <= beta
    (main.cpp:31-32,75-83); no rigid transform (main.cpp:161 applies none);
  * associations: ni = round(m(1-rho)) inliers (p,p) drawn without replacement, then
    no = m-ni outliers (p,q), q != p, uniform over the n x n grid without duplicates;
    outliers occupy rows [0,no), inliers rows [no,m)  (bm_utils.cpp:312-315,344);
  * u0: m draws of U[0,1) from the same stream, always passed explicitly to solve(u0)
    because the reference default is seeded from std::random_device (src/utils.cpp:24-25).

Everything is numpy (host side); arrays are returned in the reference's column-major layout.
"""
import os

import numpy as np

SEED_BASE = 0xC11BBE2
BUNNY_FIXTURE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                             "bun10k_points.npz")
_cloud_cache = {}


def read_ply_xyz(path):
    """vertices of a binary little-endian PLY whose vertex element is exactly (float x, float y, float z)"""
    with open(path, "rb") as f:
        raw = f.read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    header = raw[:end].decode("ascii", "replace").splitlines()
    if "format binary_little_endian 1.0" not in header:
        raise ValueError("unsupported PLY format")
    n = int([ln.split()[2] for ln in header if ln.startswith("element vertex")][0])
    props = [ln.split()[1:] for ln in header if ln.startswith("property")]
    if props != [["float", "x"], ["float", "y"], ["float", "z"]]:
        raise ValueError("unsupported PLY vertex layout: %r" % (props,))
    return np.frombuffer(raw, dtype="<f4", count=3 * n, offset=end).reshape(n, 3).copy()


def bunny_points():
    """(9992, 3) float32 vertices of the reference's bun10k.ply and where they came from, or (None, why)"""
    if os.path.exists(BUNNY_FIXTURE):
        return np.load(BUNNY_FIXTURE)["xyz"], "tests/golden/bun10k_points.npz (fixture of bun10k.ply)"
    return None, "synthetic surface (the bun10k.ply fixture is absent)"


def cloud_source(n=9992):
    return bunny_points()[1] if n == 9992 else "synthetic surface (n != 9992)"


def scale_to_cube(pts, side=1.0):
    """reference benchmarks/bm_utils.cpp scale_to_cube: divide by the largest axis extent"""
    ext = pts.max(axis=0) - pts.min(axis=0)
    return pts * (side / ext.max())


def make_cloud(n=9992, seed=SEED_BASE):
    """3 x n cloud scaled so that its largest axis extent is 1: the bunny for n = 9992 (see module docstring),
    else n points on a star-shaped bumpy closed surface."""
    if n == 9992:
        if "bunny" not in _cloud_cache:
            xyz, _ = bunny_points()
            _cloud_cache["bunny"] = None if xyz is None else np.asfortranarray(scale_to_cube(xyz.astype(np.float64)).T)
        if _cloud_cache["bunny"] is not None:
            return _cloud_cache["bunny"].copy(order="F")
    rng = np.random.default_rng(seed)
    v = rng.standard_normal((n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    x, y, z = v[:, 0], v[:, 1], v[:, 2]
    r = (1.0 + 0.25 * x * y + 0.2 * np.sin(3.0 * z) + 0.15 * np.cos(4.0 * x + 1.0) * y
         + 0.1 * np.sin(5.0 * y * z))
    pts = v * r[:, None] * np.array([1.0, 0.8, 0.6])
    ext = pts.max(axis=0) - pts.min(axis=0)
    pts = pts / ext.max()
    return np.asfortranarray(pts.T)  # 3 x n, column-major: each point contiguous


def bounded_normal_noise(rng, n, sigma, beta):
    eta = rng.normal(0.0, sigma, size=(n, 3))
    bad = np.linalg.norm(eta, axis=1) > beta
    while bad.any():
        eta[bad] = rng.normal(0.0, sigma, size=(int(bad.sum()), 3))
        bad = np.linalg.norm(eta, axis=1) > beta
    return eta


def make_associations(rng, n, m, rho):
    ni = int(round(m * (1.0 - rho)))
    no = m - ni
    if ni > n:
        raise ValueError("not enough points for the requested inlier count")
    inl = rng.permutation(n)[:ni]
    A = np.zeros((m, 2), dtype=np.int32, order="F")
    A[no:, 0] = inl
    A[no:, 1] = inl
    seen = set()
    k = 0
    while k < no:
        need = no - k
        p = rng.integers(0, n, size=2 * need + 16)
        q = rng.integers(0, n, size=2 * need + 16)
        for a, b in zip(p.tolist(), q.tolist()):
            if a == b or (a, b) in seen:
                continue
            seen.add((a, b))
            A[k, 0] = a
            A[k, 1] = b
            k += 1
            if k == no:
                break
    return A, ni


def euclidean_problem(m, rho, seed, n=9992, noise_sigma=0.01, noise_beta=0.0554):
    """Returns dict(D1 3xn, D2 3xn, A mx2 int32, u0 m, ni, rho)."""
    rng = np.random.default_rng(seed)
    D1 = make_cloud(n, SEED_BASE)
    eta = bounded_normal_noise(rng, n, noise_sigma, noise_beta)
    D2 = np.asfortranarray(D1 + eta.T)
    A, ni = make_associations(rng, n, m, rho)
    u0 = rng.random(m)
    return dict(D1=D1, D2=D2, A=A, u0=u0, ni=ni, rho=rho, m=m)


def pointnormal_problem(m, rho, seed, n=9992, noise_sigma=0.01, noise_beta=0.0554, normal_sigma=0.01):
    """6xn point-normal data: the cloud above plus seeded unit normals; view 2 perturbs both."""
    rng = np.random.default_rng(seed)
    P1 = make_cloud(n, SEED_BASE)
    nrm = rng.standard_normal((3, n))
    nrm /= np.linalg.norm(nrm, axis=0, keepdims=True)
    eta = bounded_normal_noise(rng, n, noise_sigma, noise_beta)
    P2 = P1 + eta.T
    n2 = nrm + rng.normal(0.0, normal_sigma, size=(3, n))
    n2 /= np.linalg.norm(n2, axis=0, keepdims=True)
    D1 = np.asfortranarray(np.vstack([P1, nrm]))
    D2 = np.asfortranarray(np.vstack([P2, n2]))
    A, ni = make_associations(rng, n, m, rho)
    u0 = rng.random(m)
    return dict(D1=D1, D2=D2, A=A, u0=u0, ni=ni, rho=rho, m=m)


# BASELINE.json configs (SURVEY.md section 8d)
CONFIGS = {
    "c1": dict(kind="euclidean", m=1000, rho=0.90, sigma=0.01, epsilon=0.02, seed=SEED_BASE + 1),
    "c2": dict(kind="euclidean", m=20000, rho=0.95, sigma=0.015, epsilon=0.05, seed=SEED_BASE + 2),
    "c3": dict(kind="pointnormal", m=10000, rho=0.95, sigp=0.5, epsp=0.5, sign=0.10, epsn=0.35,
               seed=SEED_BASE + 3),
    "c4": dict(kind="euclidean", m=80000, rho=0.95, sigma=0.015, epsilon=0.05, seed=SEED_BASE + 4),
}


def config_problem(name, m=None):
    cfg = dict(CONFIGS[name])
    if m is not None:
        cfg["m"] = int(m)
    if cfg["kind"] == "euclidean":
        prob = euclidean_problem(cfg["m"], cfg["rho"], cfg["seed"])
    else:
        prob = pointnormal_problem(cfg["m"], cfg["rho"], cfg["seed"])
    prob["cfg"] = cfg
    return prob
