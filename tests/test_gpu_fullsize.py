"""GPU parity at BASELINE.json's FULL sizes, every stage of the hot path through the C ABI against the oracle (tests/stagecheck.py):
  C5  the 1M-tet pile bench.py times (146 x sphere1K.msh on a jittered FCC lattice; the synthetic column pile as a second case),
      in canonical order AND in the exact mode bench.py runs (canonical_order = 0, contact_partition = 1: lists compared as sorted multisets),
  C3  ball on mat, 246,851 tets (mat 200x200x1 + sphere1K.msh),
  C4  squeeze-out bodies tiled x3, 541,707 tets, dense self-contact."""
import os
import sys

import pytest

from ipc_b200 import scenes
from stagecheck import check_every_stage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu
need_c4_meshes = pytest.mark.skipif(not scenes.have_squeeze_out_meshes(), reason="the C4 squeeze-out meshes are too large to store: __graft_entry__.build() caches them where the reference tree is present")


class _Args:
    tets, res = 1_000_000, 10

    def __init__(self, scene):
        self.scene = scene


@pytest.mark.parametrize("canonical", [True, False], ids=["canonical", "bench_mode"])
def test_c5_sphere1k_fcc_pile_every_stage(gpu_ctx, canonical):
    import bench
    m, info = bench.build_scene(_Args("c5"))
    assert m.nT == 1_000_246 and m.nV == 256_960 and len(m.SVI) == 180_894  # SURVEY 8(d)
    r = check_every_stage(gpu_ctx, m, info, kappa=bench.KAPPA, canonical=canonical, min_active=1000)
    assert r["n_full_cand"] > 100_000


def test_synthetic_column_pile_every_stage(gpu_ctx):
    import bench
    m, info = bench.build_scene(_Args("pile"))
    assert m.nT >= 1_000_000
    check_every_stage(gpu_ctx, m, info, kappa=bench.KAPPA, min_active=10_000)


@pytest.mark.parametrize("canonical", [True, False], ids=["canonical", "bench_mode"])
def test_c3_ball_on_mat_250k_every_stage(gpu_ctx, canonical):
    m, info = scenes.ball_on_mat_c3(nx=200)
    assert m.nT == 246_851
    check_every_stage(gpu_ctx, m, info, canonical=canonical, min_active=20)


@need_c4_meshes
@pytest.mark.parametrize("canonical", [True, False], ids=["canonical", "bench_mode"])
def test_c4_squeeze_out_500k_every_stage(gpu_ctx, canonical):
    m, info = scenes.squeeze_out_tiled()
    assert m.nT >= 500_000
    r = check_every_stage(gpu_ctx, m, info, canonical=canonical, min_active=10_000)
    assert r["n_para"] > 0  # the dense patches contain nearly parallel edge pairs (mollified set)
