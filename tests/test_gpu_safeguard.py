"""GPU parity of the line-search safeguards (SURVEY 8(f) rank 2): element inversion count and edge-triangle intersection check,
through the C ABI against the oracle (exact predicate: the COUNTS must be identical)."""
import numpy as np
import pytest

import oracle as orc
from ipc_b200 import mesh as M
from ipc_b200 import scenes

pytestmark = pytest.mark.gpu


def upload(ctx, m):
    ctx.set_mesh(m.V_rest_soa, m.T_soa, m.restTriInv, m.vol, m.mu, m.lam, m.mass, m.dbc, m.energy)
    ctx.set_surface(m.SVI, m.SFEdges, m.SF_soa, m.vCoDim)
    ctx.set_state(m.V_soa)


def two_cubes(dz, n=3):
    V1, T1 = M.grid_tets(n, n, n, h=1.0 / n)
    V2, T2 = M.grid_tets(n, n, n, h=1.0 / n, origin=(0.13, 0.21, dz))
    return M.merge_meshes([(V1, T1), (V2, T2)])


@pytest.mark.parametrize("dz,free", [(1.05, True), (0.8, False), (0.999, False)])
def test_intersection_check_matches_oracle(gpu_ctx, dz, free):
    m = two_cubes(dz)
    rng = np.random.default_rng(3)
    m.V = m.V_rest + 0.01 * rng.standard_normal(m.V_rest.shape)
    upload(gpu_ctx, m)
    ok_ref, hits_ref = orc.Surf(m).intersection_free(nthreads=4)
    assert ok_ref == free
    assert gpu_ctx.intersection_free() == ok_ref
    gpu_ctx.intersection_free(want=False)  # deferred form: the count comes back with the iteration
    gpu_ctx.check_inversion(want=False)
    it = gpu_ctx.fetch_iteration()
    assert it.n_intersected_triangles == hits_ref and it.n_inverted_tets == orc.Elastic(m).count_inverted()
    # all-Dirichlet pairs are skipped (:3282)
    m.dbc[:] = 1
    upload(gpu_ctx, m)
    assert gpu_ctx.intersection_free() is True
    m.dbc[:] = 0


def test_inversion_count_matches_oracle(gpu_ctx):
    m = scenes.twisted_mat(nx=10, ny=10, nz=8, energy=1, invert_frac=0.02)  # FCR scene with flipped tets
    upload(gpu_ctx, m)
    n_ref = orc.Elastic(m).count_inverted()
    assert n_ref > 0 and gpu_ctx.check_inversion() == n_ref
    m.V = m.V_rest.copy()
    upload(gpu_ctx, m)
    assert gpu_ctx.check_inversion() == 0


@pytest.mark.parametrize("scene", ["c5", pytest.param("c4", marks=pytest.mark.skipif(
    not scenes.have_squeeze_out_meshes(), reason="the C4 squeeze-out meshes are too large to store: __graft_entry__.build() caches them where the reference tree is present"))])
def test_full_size_scenes_intersection_counts(gpu_ctx, scene):
    """C5 (1M tets) is intersection free; C4's manufactured shell crosses its core in places (scenes.squeeze_out_tiled): the device
    must find exactly the triangles the oracle finds, degenerate near-coplanar configurations included."""
    import bench

    class A:
        tets, res = 1_000_000, 10

    A.scene = scene
    m = bench.build_scene(A)[0] if scene == "c5" else scenes.squeeze_out_tiled()[0]
    upload(gpu_ctx, m)
    ok_ref, hits_ref = orc.Surf(m).intersection_free(nthreads=64)
    gpu_ctx.intersection_free(want=False)
    gpu_ctx.check_inversion(want=False)
    it = gpu_ctx.fetch_iteration()
    assert it.n_intersected_triangles == hits_ref and (hits_ref == 0) == ok_ref
    assert it.n_inverted_tets == 0
