"""GPU parity (through the C ABI) of the kinematic-obstacle hand-off (SURVEY 8 row f3, MeshCO<3> on the barrier / Tight-Inclusion path):
the obstacle rides at the tail of the mesh's arrays (ipcgpu_set_obstacle_tail), the contact stages cover mesh-mesh and mesh-obstacle pairs in
one pass; results are split on the host (ipc_b200/obstacle.py, the mirror of the C++ adapter) and compared with the self-contact oracle of the
mesh alone AND the MeshCO oracle (oracle/meshco.cpp): sets identical, E / g <= 1e-10, H <= 1e-9, step bounds bit-exact."""
import numpy as np
import pytest

import oracle as orc
from ipc_b200 import lib as L
from ipc_b200 import obstacle as OB
from ipc_b200 import scenes
from test_oracle_meshco import contact_pairs

pytestmark = pytest.mark.gpu
KAPPA = 1e8
NTH = 8


def bits(x):
    return np.float64(x).view(np.uint64)


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


def lex(a):
    a = np.asarray(a)
    return a[np.lexsort(a.T[::-1])] if len(a) else a


def upload(ctx, M2, ee_as_vf=1):
    ctx.set_mesh(M2.V_rest_soa, M2.T_soa, M2.restTriInv, M2.vol, M2.mu, M2.lam, M2.mass, M2.dbc, M2.energy)
    ctx.set_surface(M2.SVI, M2.SFEdges, M2.SF_soa, M2.vCoDim)
    ctx.set_state(M2.V_soa)
    ctx.set_obstacle_tail(M2.nV_dof, ee_as_vf)


def remove_obstacle(ctx):
    ctx.set_obstacle_tail(-1)


@pytest.fixture
def ctx(gpu_ctx):
    yield gpu_ctx
    remove_obstacle(gpu_ctx)


def build(angle, **kw):
    m, info = scenes.balls_on_obstacle(plate_angle=angle, **kw)
    ob = info["obstacle"]
    s = orc.Surf(m)
    o = orc.Obstacle(s, ob["V"], ob["E"], ob["F"])
    return m, info, ob, s, o, OB.with_obstacle(m, ob["V"], ob["E"], ob["F"])


@pytest.mark.parametrize("angle,res", [(0.37, 4), (0.0, 4), (0.37, 8)])
def test_sets_energy_gradient_hessian(ctx, angle, res):
    m, info, ob, s, o, M2 = build(angle, res=res, plate=12 if res == 4 else 30)
    dHat = info["dHat"]
    upload(ctx, M2)
    mm, pa, pe, cand = ctx.constraint_set(dHat, 1)
    (smm, spa, spe), (cmm, cpa, cpe) = OB.split_sets(mm, pa, pe, m.nV, len(m.SFEdges))
    mm_s, pa_s, pe_s, cand_s = s.constraint_set(dHat, NTH)
    mm_o, pa_o, pe_o, cand_o = o.constraint_set(dHat, NTH)
    assert len(mm_o) > 10
    assert np.array_equal(lex(smm), mm_s) and np.array_equal(lex(cmm), mm_o)
    assert np.array_equal(lex(np.concatenate([spa, spe], axis=1)), np.concatenate([pa_s, pe_s], axis=1).reshape(-1, 6))
    assert np.array_equal(lex(np.concatenate([cpa, cpe], axis=1)), np.concatenate([pa_o, pe_o], axis=1).reshape(-1, 6))
    if angle == 0.0:
        assert len(pa_o) > 0
    sc, cc = OB.split_candidates(cand, len(m.SVI), len(m.SF), len(m.SFEdges))
    assert np.array_equal(lex(sc), cand_s) and np.array_equal(lex(cc), cand_o)
    # energy: the two handlers' sum (Optimizer.cpp:3268-3353)
    E_ref = s.barrier_energy(mm_s, pa_s, pe_s, dHat, KAPPA)[0] + o.energy(mm_o, pa_o, pe_o, dHat, KAPPA)[0]
    E = ctx.barrier_energy(dHat, KAPPA)
    assert abs(E - E_ref) <= 1e-10 * abs(E_ref)
    # gradient: the mesh's rows (the tail's rows are Dirichlet rows)
    g = np.zeros(3 * M2.nV)
    ctx.barrier_gradient(dHat, KAPPA, g)
    g_ref = s.barrier_gradient(mm_s, pa_s, pe_s, dHat, KAPPA)
    o.gradient(mm_o, pa_o, pe_o, dHat, KAPPA, g=g_ref)
    assert rel(g[: 3 * m.nV], g_ref) <= 1e-10
    # Hessian: the merged pattern = the mesh's pattern + identity rows of the tail; the mesh's values are a prefix of the value array
    mg, pg = o.to_merged(mm_o, pe_o)
    pag, _ = o.to_merged(pa_o, pe_o)
    extra = contact_pairs(mm_s, pa_s, pe_s, m.SFEdges, m.nV) + contact_pairs(mg, pag, pg, M2.SFEdges, m.nV)
    ia, ja = m.csr_pattern(1, extra_pairs=extra)
    ia2, ja2 = M2.csr_pattern(1, extra_pairs=extra)
    nnz = ia[3 * m.nV] - 1
    assert np.array_equal(ia2[: 3 * m.nV + 1], ia) and np.array_equal(ja2[:nnz], ja)
    ctx.set_csr(ia2, ja2, 1)
    for projectDBC in (1, 0):
        a = np.zeros(ja2.size)
        ctx.barrier_hessian(dHat, KAPPA, projectDBC, a)
        a_ref = s.barrier_hessian_csr(mm_s, pa_s, pe_s, dHat, KAPPA, ia, ja, 1, projectDBC, nthreads=NTH)
        o.hessian_csr(mm_o, pa_o, pe_o, dHat, KAPPA, ia, ja, 1, projectDBC, a=a_ref, nthreads=NTH)
        assert np.abs(a[:nnz] - a_ref).max() <= 1e-9 * np.abs(a_ref).max()
        assert np.all(a[nnz:] == 0.0)  # nothing of the barrier terms lands in the obstacle's rows


@pytest.mark.parametrize("ee_as_vf,angle,res,plate", [(1, 0.0, 4, 12), (0, 0.0, 4, 12), (1, 0.37, 6, 20), (0, 0.37, 8, 30)])
def test_step_bounds_bit_exact(ctx, ee_as_vf, angle, res, plate):
    # (on the aligned plate an edge pair sets the partial bound: 0.2597 through the vertex-face routine, 0.2617 through the edge-edge one)
    m, info, ob, s, o, M2 = build(angle, res=res, plate=plate)
    dHat, p = info["dHat"], info["p"]
    upload(ctx, M2, ee_as_vf)
    p2 = OB.pad_direction(p, M2.nV)
    ctx.constraint_set(dHat, 1)
    _, _, _, cand_s = s.constraint_set(dHat, NTH)
    _, _, _, cand_o = o.constraint_set(dHat, NTH)
    evf, eee = L.Context.ti_error(m.V_soa, m.nV, None)  # computeTightInclusionError: the mesh's box (CCDUtils.cpp:29-46)
    a = ctx.ccd_partial(p2, 1e-6, evf, eee, 1.0)
    a_self, _ = orc.ccd_partial(s, p, cand_s, 1e-6, evf, eee, 1.0, NTH)
    a_co, z = o.ccd_partial(p, cand_o, 1e-6, evf, eee, 1.0, ee_as_vf=ee_as_vf, nthreads=NTH)
    assert not z and bits(a) == bits(min(a_self, a_co)), (a, a_self, a_co)
    assert a_co < 1.0
    hvox = m.avgEdgeLen / 3.0
    ag = ctx.hash_build_swept(p2, a, hvox)
    a2, ncand = ctx.ccd_full(1e-6, evf, eee, ag)
    gs = orc.grid_swept(s, p, a, hvox)
    assert bits(gs[1]) == bits(ag)  # the swept grid's own step only looks at the mesh's motion
    a2_self, _, _ = orc.ccd_full(s, p, gs[0], gs[1], 1e-6, evf, eee, gs[1], nthreads=NTH)
    a2_co, z, npairs = o.ccd_full(p, 1e-6, evf, eee, gs[1], ee_as_vf=ee_as_vf, nthreads=NTH)
    assert not z and bits(a2) == bits(min(a2_self, a2_co)), (a2, a2_self, a2_co)
    assert ctx.ccd_stats()[2] == 0 and ncand > 0


def test_moving_the_obstacle_and_the_intersection_check(ctx):
    m, info, ob, s, o, M2 = build(0.37, res=4)
    dHat = info["dHat"]
    upload(ctx, M2)
    n0 = len(ctx.constraint_set(dHat, 0)[0])
    assert ctx.intersection_free()
    # far away: only the mesh's own pairs are left
    Vfar = ob["V"] + np.array([0.0, 0.0, -5.0])
    ctx.set_obstacle_positions(Vfar)
    mm, pa, pe, _ = ctx.constraint_set(dHat, 0)
    mm_s, pa_s, pe_s, _ = s.constraint_set(dHat, NTH)
    assert len(mm) < n0 and np.array_equal(mm, mm_s)
    # pushed into the lowest ball: mesh edges cross obstacle triangles (MeshCO.cpp:2611-2678)
    Vin = ob["V"] + np.array([0.0, 0.0, 0.3])
    ctx.set_obstacle_positions(Vin)
    assert not ctx.intersection_free()
    M3 = OB.with_obstacle(m, Vin, ob["E"], ob["F"])
    assert not orc.Surf(M3).intersection_free(nthreads=NTH)[0]
    # back in place: the first result again
    ctx.set_obstacle_positions(ob["V"])
    assert len(ctx.constraint_set(dHat, 0)[0]) == n0 and ctx.intersection_free()


def test_tail_is_validated(gpu_ctx):
    m, info, ob, s, o, M2 = build(0.37, res=4)
    bad = OB.with_obstacle(m, ob["V"], ob["E"], ob["F"])
    bad.dbc = bad.dbc.copy()
    bad.dbc[-1] = 0
    with pytest.raises(L.IpcGpuError):
        upload(gpu_ctx, bad)
    remove_obstacle(gpu_ctx)
    with pytest.raises(L.IpcGpuError):  # a tetrahedron would use an obstacle vertex
        gpu_ctx.set_mesh(m.V_rest_soa, m.T_soa, m.restTriInv, m.vol, m.mu, m.lam, m.mass, np.ones(m.nV, dtype=np.uint8), m.energy)
        gpu_ctx.set_obstacle_tail(m.nV - 1)
    remove_obstacle(gpu_ctx)


def test_c3_ball_over_the_mat_as_obstacle(ctx):
    """BASELINE config C3's bodies with the 200 x 200 mat as the obstacle (80,802 obstacle vertices, 161,600 triangles against sphere1K.msh)"""
    m, info = scenes.ball_on_obstacle_mat(200)
    ob = info["obstacle"]
    s = orc.Surf(m)
    o = orc.Obstacle(s, ob["V"], ob["E"], ob["F"])
    M2 = OB.with_obstacle(m, ob["V"], ob["E"], ob["F"])
    dHat, p = info["dHat"], info["p"]
    upload(ctx, M2)
    mm, pa, pe, cand = ctx.constraint_set(dHat, 1)
    (smm, spa, spe), (cmm, cpa, cpe) = OB.split_sets(mm, pa, pe, m.nV, len(m.SFEdges))
    mm_o, pa_o, pe_o, cand_o = o.constraint_set(dHat, NTH)
    assert len(smm) == 0 and len(mm_o) > 50 and np.array_equal(lex(cmm), mm_o)
    sc, cc = OB.split_candidates(cand, len(m.SVI), len(m.SF), len(m.SFEdges))
    assert len(sc) == 0 and np.array_equal(lex(cc), cand_o)
    E_ref = o.energy(mm_o, pa_o, pe_o, dHat, KAPPA)[0]
    assert abs(ctx.barrier_energy(dHat, KAPPA) - E_ref) <= 1e-10 * abs(E_ref)
    g = np.zeros(3 * M2.nV)
    ctx.barrier_gradient(dHat, KAPPA, g)
    assert rel(g[: 3 * m.nV], o.gradient(mm_o, pa_o, pe_o, dHat, KAPPA)) <= 1e-10
    evf, eee = L.Context.ti_error(m.V_soa, m.nV, None)
    p2 = OB.pad_direction(p, M2.nV)
    a = ctx.ccd_partial(p2, 1e-6, evf, eee, 1.0)
    a_co, z = o.ccd_partial(p, cand_o, 1e-6, evf, eee, 1.0, nthreads=NTH)
    assert not z and a_co < 1.0 and bits(a) == bits(a_co)
    # the full CCD from the untouched step: every swept mesh primitive against the mat
    hvox = m.avgEdgeLen / 3.0
    ag = ctx.hash_build_swept(p2, 1.0, hvox)
    a2, ncand = ctx.ccd_full(1e-6, evf, eee, ag)
    a2_co, z, npairs = o.ccd_full(p, 1e-6, evf, eee, ag, nthreads=NTH)
    assert not z and npairs > 0 and ncand > 0 and bits(a2) == bits(a2_co), (a2, a2_co)
    assert ctx.ccd_stats()[2] == 0 and ctx.intersection_free()


def test_no_friction_against_the_obstacle(ctx):
    """MeshCO does not implement the friction functions (CollisionObject.h:403-423): with an obstacle attached the lagged friction terms are those
    of the mesh's own pairs; the obstacle's pairs are lagged with a zero normal force"""
    from test_oracle_friction import COEF
    m, info, ob, s, o, M2 = build(0.37, res=6, plate=20)
    dHat = info["dHat"]
    rng = np.random.default_rng(3)
    Vt = m.V - 0.3 * np.sqrt(dHat) * rng.standard_normal(m.V.shape)
    upload(ctx, M2)
    ctx.set_prev_state(np.ascontiguousarray(np.concatenate([Vt, ob["V"]]).T).ravel())
    mm, _, _, _ = ctx.constraint_set(dHat, 0)
    n = ctx.friction_lag(dHat, KAPPA)
    assert n == len(mm)
    mm_l, lam, co, ba = ctx.get_friction_data()
    cross = np.array([OB.involves_obstacle(q, m.nV) for q in mm_l])
    assert cross.any() and (~cross).any() and np.all(lam[cross] == 0.0) and np.all(lam[~cross] > 0.0)
    mm_s, _, _, _ = s.constraint_set(dHat, NTH)
    lam_r, co_r, ba_r = s.friction_lag(mm_s, dHat, KAPPA)
    eps2 = 1e-2 * dHat
    E = ctx.friction_energy(eps2, COEF)
    E_r = s.friction_energy(Vt, mm_s, lam_r, co_r, ba_r, eps2, COEF)
    assert E_r > 0 and abs(E - E_r) <= 1e-10 * abs(E_r)
    g = ctx.friction_gradient(eps2, COEF, np.zeros(3 * M2.nV))
    g_r = s.friction_gradient(Vt, mm_s, lam_r, co_r, ba_r, eps2, COEF)
    assert rel(g[: 3 * m.nV], g_r) <= 1e-10 and np.all(g[3 * m.nV:] == 0.0)


def test_swept_grid_step_ignores_the_obstacle(ctx):
    """SpatialHash::build rescales the step by the mean |p| over mesh.SVI (SpatialHash.hpp:603-618): the obstacle's vertices must not dilute it"""
    m, info, ob, s, o, M2 = build(0.37, res=4)
    upload(ctx, M2)
    p = 40.0 * info["p"]
    hvox = m.avgEdgeLen / 3.0
    ag = ctx.hash_build_swept(OB.pad_direction(p, M2.nV), 1.0, hvox)
    g = orc.grid_swept(s, p, 1.0, hvox)
    assert g[1] < 1.0 and bits(ag) == bits(g[1]), (ag, g[1])
