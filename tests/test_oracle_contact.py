"""CPU tests of the oracle's contact restatement.
Pinning: (1) pairs_golden.json = outputs of the reference's OWN codegen compiled from the reference sources (oracle/_ref);
(2) pairs_live_golden.npz = the same codegen on a sample of seeded random stencils; (3) FD / geometric invariants; (4) brute-force sets."""
import json
import os

import numpy as np
import pytest

import oracle as orc
from ipc_b200 import mesh as M

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "pairs_golden.json")))


def close(a, b, tol=1e-11):
    a, b = np.asarray(a), np.asarray(b)
    return np.abs(a - b).max() <= tol * max(1.0, np.abs(b).max())


@pytest.mark.parametrize("k", range(len(GOLD["cases"])))
def test_pair_derivatives_vs_reference_codegen_golden(k):
    c = GOLD["cases"][k]
    X = np.array(c["X"])
    scale_tol = 1e-11 if k < 13 else 1e-6  # the last 3 cases are tiny stencils far from the origin: the codegen itself cancels
    assert close(orc.g_pair("PE", X[:3]), c["g_PE"], scale_tol) and close(orc.H_pair("PE", X[:3]), c["H_PE"], scale_tol)
    assert close(orc.g_pair("PT", X), c["g_PT"], scale_tol) and close(orc.H_pair("PT", X), c["H_PT"], scale_tol)
    assert close(orc.g_pair("EE", X), c["g_EE"], scale_tol) and close(orc.H_pair("EE", X), c["H_EE"], scale_tol)
    _, g, H = orc.ee_cross(X)
    assert close(g, c["cross_g"], scale_tol) and close(H, c["cross_H"], scale_tol)


def test_pair_derivatives_vs_reference_codegen_live():
    """a fixed sample of seeded random stencils, the reference codegen's outputs stored by golden/gen_pairs_live_golden.py"""
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "pairs_live_golden.npz"))
    rng = np.random.default_rng(7)
    assert np.array_equal(ref["X"], np.stack([rng.standard_normal((4, 3)) for _ in range(200)])[::8])
    for k, X in enumerate(ref["X"]):
        assert close(orc.g_pair("PE", X[:3]), ref["g_PE"][k]) and close(orc.H_pair("PE", X[:3]), ref["H_PE"][k])
        assert close(orc.g_pair("PT", X), ref["g_PT"][k]) and close(orc.H_pair("PT", X), ref["H_PT"][k])
        assert close(orc.g_pair("EE", X), ref["g_EE"][k]) and close(orc.H_pair("EE", X), ref["H_EE"][k])
        _, g, H = orc.ee_cross(X)
        assert close(g, ref["cross_g"][k]) and close(H, ref["cross_H"][k])


def test_barrier_and_q_vs_reference():
    for c in GOLD["barrier"]:
        b, g, H = orc.barrier(c["d"], c["dHat"])
        assert b == c["b"] and g == c["g"] and H == c["H"]  # same expressions, same order: bit-exact
    for c in GOLD["q"]:
        X = np.array([[0, 0, 0], [1, 0, 0], [0, 0, 1], [0, 1, 1.0]])  # cross norm = 1 -> scale to x
        s = np.sqrt(c["x"])
        X2 = np.array([[0, 0, 0], [s, 0, 0], [0, 0, 1], [0, 1, 1.0]])
        e, _, _ = orc.mollifier(X2, c["eps"])
        assert abs(e - c["q"]) <= 1e-14 * max(1, abs(c["q"]))
    assert orc.barrier(1.0, 1.0)[0] == 0.0 and orc.barrier(1.0, 1.0)[1] == 0.0


@pytest.mark.parametrize("kind,n", [("PP", 2), ("PE", 3), ("PT", 4), ("EE", 4)])
def test_fd_consistency(kind, n):  # derivTest_* (MeshCollisionUtils.hpp:178-225 ...): FD of d vs g, of g vs H
    rng = np.random.default_rng(3)
    for _ in range(5):
        X = rng.standard_normal((n, 3))
        g, H = orc.g_pair(kind, X), orc.H_pair(kind, X)
        h = 1e-6
        for i in range(3 * n):
            e = np.zeros(3 * n); e[i] = h
            fd = (orc.d_pair(kind, X.ravel() + e) - orc.d_pair(kind, X.ravel() - e)) / (2 * h)
            assert abs(fd - g[i]) <= 1e-6 * max(1, abs(g).max())
            fdg = (orc.g_pair(kind, X.ravel() + e) - orc.g_pair(kind, X.ravel() - e)) / (2 * h)
            assert np.abs(fdg - H[:, i]).max() <= 2e-6 * max(1, abs(H).max())
        assert np.allclose(H, H.T, atol=1e-12 * abs(H).max())


def test_mollifier_fd():
    rng = np.random.default_rng(4)
    X = np.array([[0, 0, 0], [1, 0, 0], [0.1, 0.2, 0.3], [1.1, 0.25, 0.28]]) + 0.01 * rng.standard_normal((4, 3))
    c, _, _ = orc.ee_cross(X)
    eps = 4 * c
    e, g, H = orc.mollifier(X, eps)
    assert 0 < e < 1
    h = 1e-6
    for i in range(12):
        d = np.zeros(12); d[i] = h
        ep, gp, _ = orc.mollifier(X.ravel() + d, eps)
        em, gm, _ = orc.mollifier(X.ravel() - d, eps)
        assert abs((ep - em) / (2 * h) - g[i]) <= 1e-6 * max(1, abs(g).max())
        assert np.abs((gp - gm) / (2 * h) - H[:, i]).max() <= 1e-5 * max(1, abs(H).max())
    e1, g1, H1 = orc.mollifier(X, c * 0.5)
    assert e1 == 1.0 and not g1.any() and not H1.any()


def brute_pt(p, a, b, c, n=60):
    u, v = np.meshgrid(np.linspace(0, 1, n), np.linspace(0, 1, n))
    k = u + v <= 1
    pts = a + u[k][:, None] * (b - a) + v[k][:, None] * (c - a)
    return ((pts - p) ** 2).sum(1).min()


def brute_ee(a0, a1, b0, b1, n=200):
    s = np.linspace(0, 1, n)
    A = a0 + s[:, None] * (a1 - a0)
    B = b0 + s[:, None] * (b1 - b0)
    return ((A[:, None, :] - B[None, :, :]) ** 2).sum(2).min()


def test_dtype_reference_cases_and_distances():
    # checkDType fixed cases (MeshCollisionUtils.hpp:2216-2228)
    X0 = np.array([[0, 0, 1], [0, 0, 0], [1, 0, 0], [0, 1, 0.0]])
    assert orc.dType_PT(X0) == 0 and abs(orc.point_tri_d(X0) - 1.0) < 1e-15
    rng = np.random.default_rng(5)
    seen_pt, seen_ee = set(), set()
    for _ in range(400):
        X = rng.standard_normal((4, 3))
        seen_pt.add(orc.dType_PT(X)); seen_ee.add(orc.dType_EE(X))
        d = orc.point_tri_d(X)
        assert d <= brute_pt(X[0], X[1], X[2], X[3]) * (1 + 1e-12) and d >= brute_pt(X[0], X[1], X[2], X[3]) - 0.2
        de = orc.edge_edge_d(X)
        be = brute_ee(*X)
        assert de <= be * (1 + 1e-12) and de >= be - 0.05
    assert seen_pt == set(range(7)) and seen_ee == set(range(9))


def test_nearly_parallel_ee_literals():  # Diagnostic.cpp:396-403 (mode 24): 20-digit literals, distance must stay continuous
    v = np.array([[5.80045067825167737219e-01, 1.29804572829927900024e+00, 4.11720521740031375479e-01],
                  [2.64648850028170068427e-01, 1.03339687827110893181e+00, 4.11720521740029710145e-01],
                  [3.15396217796997779814e-01, 1.61344194609627678005e+00, 4.11720521740033651437e-01],
                  [1.95835346779988131006e-16, 1.34879309606810671163e+00, 4.11720521740031986102e-01]])
    p = np.array([[-1.92857301711554124974e-14, 1.46066226496805817429e-15, 4.25214990292590645001e-04],
                  [-6.08688292835163873411e-16, 4.82431649207783937812e-14, -4.25214990338334164650e-04],
                  [5.44092882834986712421e-15, -3.69845570938928918346e-14, -4.25214990330826389867e-04],
                  [1.99012418663158535008e-14, -9.01951096008029847640e-15, 4.25214990314199173770e-04]])
    ds = np.array([orc.edge_edge_d(v + (i * 1e-9) * p) for i in range(-1000, 1001, 50)])
    assert np.all(np.isfinite(ds)) and np.all(ds > 0)
    assert np.abs(np.diff(ds)).max() < 1e-6 * ds.max()  # no jump when the classification flips near parallel
    c, _, _ = orc.ee_cross(v)
    a2 = ((v[1] - v[0]) ** 2).sum() * ((v[3] - v[2]) ** 2).sum()
    assert c < 1e-20 * a2 * 1e12  # (nearly) parallel: the dType_EE guard region


def two_cubes(gap, seed=0, n=2):
    V1, T1 = M.grid_tets(n, n, n, h=1.0 / n)
    V2, T2 = M.grid_tets(n, n, n, h=1.0 / n, origin=(0.13, 0.07, 1.0 + gap))
    rng = np.random.default_rng(seed)
    m = M.merge_meshes([(V1, T1), (V2, T2)])
    m.V = m.V_rest + 0.3 * gap * rng.standard_normal(m.V_rest.shape) * 0.1
    return m


def brute_active(m, dHat):
    """Independent numpy enumeration of the PT / EE closest-feature pairs with d < dHat (classification via oracle dType)."""
    act, counter = [], {}
    V = m.V
    for vI in m.SVI:
        for t in m.SF:
            if vI in t:
                continue
            X = np.array([V[vI], V[t[0]], V[t[1]], V[t[2]]])
            if orc.point_tri_d(X) < dHat:
                ty = orc.dType_PT(X)
                if ty < 3:
                    key = (-vI - 1, t[ty], -1); counter[key] = counter.get(key, 0) + 1
                elif ty < 6:
                    a, b = ty - 3, (ty - 2) % 3
                    key = (-vI - 1, t[a], t[b]); counter[key] = counter.get(key, 0) + 1
                else:
                    act.append((-vI - 1, t[0], t[1], t[2]))
    return act, counter


def test_constraint_set_brute_force_and_encoding():
    m = two_cubes(0.01)
    dHat = 0.02 ** 2
    s = orc.Surf(m)
    mm, pa, pe, cand = s.constraint_set(dHat)
    assert len(mm) > 0
    assert np.array_equal(mm, mm[np.lexsort((mm[:, 3], mm[:, 2], mm[:, 1], mm[:, 0]))])  # canonical order
    act_pt, counter = brute_active(m, dHat)
    got_pt = {tuple(r) for r in mm if r[0] < 0 and r[3] >= 0}
    assert got_pt == set(act_pt)
    # PP/PE multiplicities are stored negated in slot 3 (SelfCollisionHandler.cpp:2434-2476); EE-derived duplicates add to the PT-derived ones
    for r in mm:
        if r[0] < 0 and r[3] < 0:
            assert -r[3] >= counter.get((r[0], r[1], r[2]), 0) and -r[3] >= 1
    # every active entry has d < dHat, every candidate pair too (cs_PTEE)
    V = m.V
    for r in mm:
        if r[0] >= 0:
            d = orc.d_pair("EE", V[[r[0], r[1], r[2], r[3]]])
        elif r[2] < 0:
            d = orc.d_pair("PP", V[[-r[0] - 1, r[1]]])
        elif r[3] < 0:
            d = orc.d_pair("PE", V[[-r[0] - 1, r[1], r[2]]])
        else:
            d = orc.d_pair("PT", V[[-r[0] - 1, r[1], r[2], r[3]]])
        assert 0 < d < dHat
    n_pt_c = sum(1 for c in cand if c[0] < 0)
    assert n_pt_c == len(act_pt) + sum(counter.values())
    # shrinking dHat gives a subset in terms of stencils
    mm2, _, _, _ = s.constraint_set(dHat * 0.25)
    keys = {tuple(r[:3]) for r in mm}
    assert {tuple(r[:3]) for r in mm2} <= keys


def test_parallel_edges_go_to_para_set():
    # two axis-aligned cubes stacked face to face: facing edges are exactly parallel -> mollified set
    V1, T1 = M.grid_tets(1, 1, 1, h=1.0)
    V2, T2 = M.grid_tets(1, 1, 1, h=1.0, origin=(0.0, 0.0, 1.01))
    m = M.merge_meshes([(V1, T1), (V2, T2)])
    s = orc.Surf(m)
    mm, pa, pe, _ = s.constraint_set(0.02 ** 2)
    assert len(pa) > 0 and len(pa) == len(pe)
    for r, e in zip(pa, pe):
        if r[3] >= 0 and r[0] >= 0:
            assert tuple(e) == (-1, -1)  # nearly parallel EE keeps its own stencil
        else:
            assert r[3] == -1 and e[0] >= 0 and e[1] > e[0]  # PP/PE from a parallel EE remembers (eI,eJ)
    E, bad = s.barrier_energy(mm, pa, pe, 0.02 ** 2, 1e3)
    assert bad == 0 and E > 0


def test_barrier_gradient_hessian_fd():
    m = two_cubes(0.01, seed=2)
    dHat, kappa = 0.02 ** 2, 1e4
    s = orc.Surf(m)
    mm, pa, pe, _ = s.constraint_set(dHat)
    g = s.barrier_gradient(mm, pa, pe, dHat, kappa)
    rng = np.random.default_rng(1)
    dx = rng.standard_normal(m.V.shape)
    h = 1e-8
    Ep, _ = orc.Surf(m, V=m.V + h * dx).barrier_energy(mm, pa, pe, dHat, kappa)
    Em, _ = orc.Surf(m, V=m.V - h * dx).barrier_energy(mm, pa, pe, dHat, kappa)
    assert abs((Ep - Em) / (2 * h) - g @ dx.ravel()) <= 1e-5 * np.linalg.norm(g) * np.linalg.norm(dx)
    assert np.abs(g.reshape(-1, 3).sum(0)).max() <= 1e-9 * np.abs(g).max()
    # CSR assembly: PSD-projected per-pair blocks summed into the pattern that contains the contact edges
    pairs = []
    for r in list(mm) + list(pa):
        vs = [(-r[0] - 1) if r[0] < 0 else r[0]] + [x for x in r[1:] if x >= 0]
        pairs += [(a, b) for a in vs for b in vs if a < b]
    for e in pe:
        if e[0] >= 0:
            vs = list(m.SFEdges[e[0]]) + list(m.SFEdges[e[1]])
            pairs += [(a, b) for a in vs for b in vs if a != b]
    ia, ja = m.csr_pattern(1, extra_pairs=pairs)
    a = s.barrier_hessian_csr(mm, pa, pe, dHat, kappa, ia, ja, 1)
    dense = np.zeros((3 * m.nV, 3 * m.nV))
    for r in mm:
        H, nv = s.pair_hessian(r, dHat, kappa)
        vs = [(-r[0] - 1) if r[0] < 0 else r[0]] + [x for x in r[1:nv]]
        assert np.linalg.eigvalsh(H[:3 * nv, :3 * nv]).min() >= -1e-9 * abs(H).max()
        for i_, vi in enumerate(vs):
            for j_, vj in enumerate(vs):
                dense[3 * vi:3 * vi + 3, 3 * vj:3 * vj + 3] += H[3 * i_:3 * i_ + 3, 3 * j_:3 * j_ + 3]
    if len(pa) == 0:
        for r in range(3 * m.nV):
            cols = ja[ia[r] - 1:ia[r + 1] - 1] - 1
            assert np.allclose(a[ia[r] - 1:ia[r + 1] - 1], dense[r, cols], atol=1e-10 * abs(dense).max())


def test_pair_hessians_are_translation_invariant():
    """Assumption behind the GPU's 12 -> 9 reduction of makePD (DESIGN.md 3.4): every pair Hessian annihilates rigid translations of its
    stencil, for all closest-feature types incl. PP/PE multiplicities; and makePD(H) = Q^T makePD(Q H Q^T) Q for the Helmert Q."""
    from ipc_b200 import scenes
    m, info = scenes.ball_pile(3, res=6, seed=5, height=3)
    s = orc.Surf(m)
    mm, pa, pe, _ = s.constraint_set(info["dHat"], nthreads=4)
    assert len(mm) > 50
    kinds = set()
    r2, r6, r12 = 2 ** -0.5, 6 ** -0.5, 12 ** -0.5
    Q = np.kron(np.array([[r2, -r2, 0, 0], [r6, r6, -2 * r6, 0], [r12, r12, r12, -3 * r12]]), np.eye(3))

    def make_pd(M):
        w, v = np.linalg.eigh(M)
        return (v * np.maximum(w, 0)) @ v.T

    for row in mm:
        H, nv = s.pair_hessian(row, info["dHat"], 1e8)
        kinds.add((int(row[0] < 0), nv))
        scale = np.abs(H).max()
        for k in range(3):
            t = np.zeros(12)
            t[k:3 * nv:3] = 1.0
            assert np.abs(H @ t).max() <= 1e-9 * scale
        # the projected matrix is a fixed point of the reduced projection
        assert np.abs(Q.T @ make_pd(Q @ H @ Q.T) @ Q - H).max() <= 1e-9 * scale
    assert len(kinds) >= 3  # several stencil types were exercised


def test_dtype_against_an_independent_closest_feature_search():
    """dType_PT / dType_EE (MeshCollisionUtils.hpp, restated branch for branch in the oracle and the kernels) decide which distance formula a pair
    gets, hence the constraint set.  Independent check: the squared distances to every sub-feature, each from its own closed form with the
    closest point constrained to the feature's INTERIOR (vertex: always valid; edge: parameter in (0,1); triangle: barycentric coordinates > 0;
    edge-edge: both parameters in (0,1)); the valid feature with the smallest distance is the closest feature and must be the reported type,
    with the same distance."""
    rng = np.random.default_rng(17)

    def pp(a, b):
        return ((a - b) ** 2).sum()

    def pe(p, a, b):  # interior projection only
        e = b - a
        t = (p - a) @ e / (e @ e)
        return ((p - (a + t * e)) ** 2).sum() if 0.0 < t < 1.0 else np.inf

    def pt(p, a, b, c):
        n = np.cross(b - a, c - a)
        q = p - ((p - a) @ n) / (n @ n) * n
        M = np.array([b - a, c - a]).T
        uv, *_ = np.linalg.lstsq(M, q - a, rcond=None)
        return ((p - q) ** 2).sum() if uv[0] > 0 and uv[1] > 0 and uv.sum() < 1 else np.inf

    def ee(a0, a1, b0, b1):
        u, v, w = a1 - a0, b1 - b0, a0 - b0
        A = np.array([[u @ u, -(u @ v)], [-(u @ v), v @ v]])
        if abs(np.linalg.det(A)) < 1e-12 * (u @ u) * (v @ v):
            return np.inf
        s, t = np.linalg.solve(A, np.array([-(u @ w), v @ w]))
        return ((a0 + s * u - b0 - t * v) ** 2).sum() if 0 < s < 1 and 0 < t < 1 else np.inf

    seen_pt, seen_ee = set(), set()
    for _ in range(3000):
        X = rng.standard_normal((4, 3)) * rng.choice([0.3, 1.0, 3.0])
        p, a, b, c = X
        cand = [pp(p, a), pp(p, b), pp(p, c), pe(p, a, b), pe(p, b, c), pe(p, c, a), pt(p, a, b, c)]  # the reference's numbering 0..6
        k = int(np.argmin(cand))
        srt = np.sort(cand)
        if srt[1] - srt[0] > 1e-9 * (1 + srt[0]):  # (skip exact ties between features)
            assert orc.dType_PT(X) == k, (orc.dType_PT(X), k, cand)
            assert abs(orc.point_tri_d(X) - cand[k]) <= 1e-12 * (1 + cand[k])
            seen_pt.add(k)
        a0, a1, b0, b1 = X
        cand = [pp(a0, b0), pp(a0, b1), pe(a0, b0, b1), pp(a1, b0), pp(a1, b1), pe(a1, b0, b1), pe(b0, a0, a1), pe(b1, a0, a1), ee(a0, a1, b0, b1)]
        k = int(np.argmin(cand))
        srt = np.sort(cand)
        if srt[1] - srt[0] > 1e-9 * (1 + srt[0]):
            assert orc.dType_EE(X) == k, (orc.dType_EE(X), k, cand)
            assert abs(orc.edge_edge_d(X) - cand[k]) <= 1e-12 * (1 + cand[k])
            seen_ee.add(k)
    assert seen_pt == set(range(7)) and seen_ee == set(range(9))
