"""GPU parity (through the C ABI) of the lagged friction terms of the self-contact pairs and of the inertia term against the oracle
(oracle/friction.cpp; SelfCollisionHandler.cpp:2481-2987, Optimizer.cpp:1582-1595, :3227-3239, :3439-3450).
E, g <= 1e-10 relative; Hessian values <= 1e-9 of the matrix norm; lagged integer set identical."""
import numpy as np
import pytest

import oracle as orc
from ipc_b200 import scenes
from stagecheck import contact_pattern_pairs, rel, sort_rows
from test_oracle_friction import COEF, KAPPA, friction_scene, slip2

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def upload(ctx, m, Vt=None):
    ctx.set_mesh(m.V_rest_soa, m.T_soa, m.restTriInv, m.vol, m.mu, m.lam, m.mass, m.dbc, m.energy)
    ctx.set_surface(m.SVI, m.SFEdges, m.SF_soa, m.vCoDim)
    ctx.set_state(m.V_soa)
    ctx.set_canonical_order(1)
    ctx.set_contact_partition(0)
    if Vt is not None:
        ctx.set_prev_state(np.ascontiguousarray(Vt.T).ravel())


def check_friction(ctx, m, s, mm_r, Vt, dHat, eps2, host_data=False):
    """lag on the device (or upload the oracle's lagged data), then E / g / H against the oracle"""
    lam_r, co_r, ba_r = s.friction_lag(mm_r, dHat, KAPPA)
    if host_data:
        ctx.set_friction_data(mm_r, lam_r, co_r, ba_r)
    else:
        mm_g, _, _, _ = ctx.constraint_set(dHat, 0)
        assert np.array_equal(mm_g, mm_r)
        n = ctx.friction_lag(dHat, KAPPA)
        assert n == len(mm_r)
        mm_l, lam, co, ba = ctx.get_friction_data()
        assert np.array_equal(mm_l, mm_r)
        assert rel(lam, lam_r) <= RTOL and np.abs(lam / lam_r - 1).max() <= 1e-9
        # closest-point coordinates: O(1) numbers from a 2x2 solve; bases: unit vectors
        assert np.abs(co - co_r).max() <= 1e-9 and np.abs(ba - ba_r).max() <= 1e-9
    E = ctx.friction_energy(eps2, COEF)
    E_r = s.friction_energy(Vt, mm_r, lam_r, co_r, ba_r, eps2, COEF)
    assert abs(E - E_r) <= RTOL * abs(E_r), (E, E_r)
    g = ctx.friction_gradient(eps2, COEF, np.zeros(3 * m.nV))
    g_r = s.friction_gradient(Vt, mm_r, lam_r, co_r, ba_r, eps2, COEF)
    assert rel(g, g_r) <= RTOL, rel(g, g_r)
    ia, ja = m.csr_pattern(1, extra_pairs=contact_pattern_pairs(m, mm_r, np.zeros((0, 4), np.int32), np.zeros((0, 2), np.int32)))
    ctx.set_csr(ia, ja, 1)
    a = ctx.friction_hessian(eps2, COEF, 1, np.zeros(ja.size))
    a_r = s.friction_hessian_csr(Vt, mm_r, lam_r, co_r, ba_r, eps2, COEF, ia, ja, 1, projectDBC=1, nthreads=8)
    assert np.linalg.norm(a_r) > 0 and rel(a, a_r) <= 1e-9, rel(a, a_r)
    return E, g, a


@pytest.mark.parametrize("host_data", [False, True], ids=["device_lag", "host_lagged_data"])
def test_four_ball_pile_every_pair_kind(gpu_ctx, host_data):
    m, info, s, mm, Vt, lam, co, ba, eps2 = friction_scene()
    upload(gpu_ctx, m, Vt)
    u2 = slip2(m.V, Vt, mm, co, ba)
    assert (u2 > eps2).sum() > 20 and (u2 <= eps2).sum() > 20  # both branches of the clamp
    check_friction(gpu_ctx, m, s, mm, Vt, info["dHat"], eps2, host_data)


def test_dirichlet_vertices_drop_their_rows_and_columns(gpu_ctx):
    m, info, s, mm, Vt, lam, co, ba, eps2 = friction_scene()
    touched = np.unique(np.where(mm[:, 0] < 0, -mm[:, 0] - 1, mm[:, 0]))
    m.dbc[touched[::3]] = 1
    m.dbc[touched[1::3]] = 2
    s = orc.Surf(m)
    upload(gpu_ctx, m, Vt)
    lam_r, co_r, ba_r = s.friction_lag(mm, info["dHat"], KAPPA)
    gpu_ctx.set_friction_data(mm, lam_r, co_r, ba_r)
    ia, ja = m.csr_pattern(1, extra_pairs=contact_pattern_pairs(m, mm, np.zeros((0, 4), np.int32), np.zeros((0, 2), np.int32)))
    gpu_ctx.set_csr(ia, ja, 1)
    for projectDBC in (0, 1):
        a = gpu_ctx.friction_hessian(eps2, COEF, projectDBC, np.zeros(ja.size))
        a_r = s.friction_hessian_csr(Vt, mm, lam_r, co_r, ba_r, eps2, COEF, ia, ja, 1, projectDBC=projectDBC, nthreads=8)
        assert rel(a, a_r) <= 1e-9
    m.dbc[:] = 0


def test_deferred_form_and_accumulation(gpu_ctx):
    """NULL outputs: nothing is read back until ipcgpu_fetch_iteration; g / a accumulate on the device-resident arrays"""
    m, info, s, mm, Vt, lam, co, ba, eps2 = friction_scene()
    upload(gpu_ctx, m, Vt)
    ctx = gpu_ctx
    ia, ja = m.csr_pattern(1, extra_pairs=contact_pattern_pairs(m, mm, np.zeros((0, 4), np.int32), np.zeros((0, 2), np.int32)))
    ctx.set_csr(ia, ja, 1)
    ctx.constraint_set(info["dHat"], 0, fetch=False, sizes=False)
    ctx.friction_lag(info["dHat"], KAPPA, want=False)
    dt2 = 0.025 ** 2
    ctx.elastic_grad_hess(dt2, 1, 1, 1, None, None)
    ctx.friction_energy(eps2, COEF, want=False)
    ctx.friction_gradient(eps2, COEF, None)
    ctx.friction_hessian(eps2, COEF, 1, None)
    it = ctx.fetch_iteration()
    from ipc_b200 import lib as L
    g = ctx.download(L.BUF_GRADIENT, 3 * m.nV)
    a = ctx.download(L.BUF_CSR_VALUES, ja.size)
    o = orc.Elastic(m)
    lam_r, co_r, ba_r = s.friction_lag(mm, info["dHat"], KAPPA)
    g_r = s.friction_gradient(Vt, mm, lam_r, co_r, ba_r, eps2, COEF, g=o.gradient(dt2, 1, 8))
    a_r = o.hessian_csr(dt2, ia, ja, 1, 1, 1, nthreads=8)
    a_r[np.asarray(ia[:-1], dtype=np.int64)[: 3 * m.nV] - 1] += np.repeat(m.mass, 3)
    a_r = s.friction_hessian_csr(Vt, mm, lam_r, co_r, ba_r, eps2, COEF, ia, ja, 1, a=a_r, nthreads=8)
    E_r = s.friction_energy(Vt, mm, lam_r, co_r, ba_r, eps2, COEF)
    assert abs(it.energy_friction - E_r) <= RTOL * abs(E_r)
    assert rel(g, g_r) <= RTOL and rel(a, a_r) <= 1e-9


def test_inertia_energy_and_gradient(gpu_ctx):
    m, info, s, mm, Vt, lam, co, ba, eps2 = friction_scene()
    m.dbc[5:40:3] = 1
    m.dbc[7:60:5] = 2
    upload(gpu_ctx, m)
    rng = np.random.default_rng(3)
    xt = m.V + 1e-2 * m.avgEdgeLen * rng.standard_normal(m.V.shape)
    gpu_ctx.set_xtilde(np.ascontiguousarray(xt.T).ravel())
    E = gpu_ctx.inertia_energy()
    E_r = float(np.sum(np.sum((m.V - xt) ** 2, axis=1) * m.mass / 2.0))  # Optimizer.cpp:3227-3239
    assert abs(E - E_r) <= 1e-13 * E_r
    for projectDBC in (0, 1):
        g0 = rng.standard_normal(3 * m.nV)
        g = gpu_ctx.inertia_gradient(projectDBC, g0.copy())
        skip = (m.dbc == 1) | ((m.dbc == 2) & bool(projectDBC))  # Mesh::isProjectDBCVertex
        g_r = g0 + np.where(skip[:, None], 0.0, m.mass[:, None] * (m.V - xt)).ravel()  # Optimizer.cpp:3439-3450
        assert np.abs(g - g_r).max() <= 1e-13 * np.abs(g_r).max()
    m.dbc[:] = 0


@pytest.mark.skipif(not scenes.have_squeeze_out_meshes(), reason="the C4 squeeze-out meshes are too large to store: __graft_entry__.build() caches them where the reference tree is present")
def test_c4_squeeze_out_dense_contact_friction(gpu_ctx):
    """BASELINE config C4 (541,707 tets, ~53k active pairs): friction E / g / H at full size, device lag"""
    m, info = scenes.squeeze_out_tiled()
    s = orc.Surf(m)
    hvox = m.avgEdgeLen / 3.0
    mm_r, _, _, _ = s.constraint_set_hashed(info["dHat"], hvox, 64)
    assert len(mm_r) > 10_000
    rng = np.random.default_rng(7)
    p = info["p"].reshape(-1, 3)
    Vt = m.V - 0.05 * p - 1e-4 * m.avgEdgeLen * rng.standard_normal(m.V.shape)  # the slip of a plausible time step
    upload(gpu_ctx, m, Vt)
    lam, co, ba = s.friction_lag(mm_r, info["dHat"], KAPPA)
    idx = rng.choice(len(mm_r), 2000, replace=False)
    eps2 = float(np.median(slip2(m.V, Vt, mm_r[idx], co[idx], ba[idx])))
    check_friction(gpu_ctx, m, s, mm_r, Vt, info["dHat"], eps2)
