#!/usr/bin/env python
"""bench.py -- Newton-iteration hot path (assembly + CCD) on the synthetic 1M-tet ball pile.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.
  metric  : BASELINE.json's "Newton-iteration wall ms (assembly+CCD) @1M tets" -> value in ms (lower is better)
  value   : device-timed (CUDA events on the launching stream), inputs/outputs resident in HBM
  e2e     : same step through the C ABI with HOST buffers (pinned), H2D/D2H inside the timed region
  roofline: dominant kernel (per-tet gradient/Hessian) algorithmic bytes / event time vs MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the oracle restatement of the reference CPU path (OpenMP over the reference's
            TBB index spaces) on the box's host cores, on a bounded sample of the same workload.
A "step" = one Newton iteration's hot stages at a fixed state (SURVEY.md 3.2):
  computeEnergyVal + computeGradient + computePrecondMtr (elastic + mass [+ barrier]) + step-size bounds
  (inversion filter [+ CCD]).  Stages in brackets join as their kernels land; `config.stages` lists what ran.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_TET = 208 + 624 + 96  # read stencil+material, write 78 upper-triangular scalars + 12 gradient scalars
ALG_BYTES_PER_CCD_CANDIDATE = 208  # SURVEY.md 8(d): 8 B candidate + 4 vertices x (x, p) x 24 B + 8 B result


def ncu_summary(name):
    """figures of a committed `ncu --set full` capture (profiles/<name>.summary.csv, written by profiles/summarize.py from the .ncu-rep of the
    same bench command): DRAM bytes per launch, FP64-pipe / issue-slot / active-warp percentages, duration"""
    path = os.path.join(ROOT, "profiles", name + ".summary.csv")
    out = {"source": "profiles/" + name + ".summary.csv"}
    try:
        import csv
        rows = {r[0]: (r[1], r[2]) for r in csv.reader(open(path)) if len(r) >= 3}
    except OSError:
        return None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}

    def val(key):
        unit, v = rows.get(key, ("", ""))
        try:
            return float(v) * scale.get(unit, 1.0)
        except ValueError:
            return None
    rd, wr = val("dram__bytes_read.sum"), val("dram__bytes_write.sum")
    out["dram_bytes"] = (rd + wr) if rd is not None and wr is not None else None
    out["fp64_pipe_pct"] = val("sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active")
    out["issue_slots_pct"] = val("sm__issue_active.avg.pct_of_peak_sustained_elapsed")
    out["warps_active_pct"] = val("sm__warps_active.avg.pct_of_peak_sustained_active")
    out["duration_us"] = val("gpu__time_duration.sum")
    out["grid"] = rows.get("Grid Size", ("", ""))[1]
    return out


# committed captures of the dominant kernels (profiles/capture_r02.sh); the round-1 captures are the fallback
NCU_TET = ncu_summary("r02_prof_k_elastic_grad_hess") or ncu_summary("r01b_prof_k_elastic_grad_hess")
NCU_ASM = ncu_summary("r02_prof_k_assemble_csr")
NCU_TI = {k: ncu_summary("r02_prof_" + k) or ncu_summary("r02l_prof_" + k) for k in ("k_ti_stage15", "k_ti_stage2")}
DT2 = 0.025 ** 2


def build_scene(args):
    """N=1 workload = the configuration the metric is quoted on: BASELINE config C5, the 1M-tet ball pile.
    scene "c5"  : as specified in BASELINE.md / SURVEY 8(d) -- 146 x input/tetMeshes/sphere1K.msh (stored as tests/golden/sphere1K.npz)
                  on a jittered FCC lattice;
    scene "pile": round 1's synthetic pile (167 rounded L6 balls of 6000 tets stacked in columns) -- kept as a second line; it has
                  ~4x the active pairs of C5 because its balls touch over flat poles."""
    from ipc_b200 import scenes
    scene = getattr(args, "scene", "c5")
    if scene == "c5":
        n_balls = max(1, int(round(args.tets / 6851)))
        m, info = scenes.sphere_pile_fcc(n_balls, seed=5, energy=0)
        info["workload"] = f"C5: {n_balls} x sphere1K.msh on a jittered FCC lattice"
    else:
        n_balls = max(1, int(round(args.tets / (6 * args.res ** 3))))
        m, info = scenes.ball_pile(n_balls, res=args.res, seed=5, energy=0)
        info["workload"] = f"synthetic column pile: {n_balls} stacked L6 balls of {6 * args.res ** 3} tets"
    info["scene"] = scene
    return m, info


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region."""

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for k, nm in enumerate(names):
                if len(s) > 3 + k and s[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def contact_pattern_pairs(m, mm, pa, pe):
    """vertex pairs that the contact stencils add to the sparsity pattern (augmentConnectivity, SelfCollisionHandler.cpp:330-415)"""
    out = []
    for arr in (mm, pa):
        if len(arr) == 0:
            continue
        a = np.asarray(arr, dtype=np.int64).copy()
        a[:, 0] = np.where(a[:, 0] < 0, -a[:, 0] - 1, a[:, 0])
        for i in range(4):
            for j in range(i + 1, 4):
                ok = (a[:, i] >= 0) & (a[:, j] >= 0)
                out.append(np.stack([a[ok, i], a[ok, j]], axis=1))
    if len(pe):
        e = np.asarray(pe, dtype=np.int64)
        e = e[e[:, 0] >= 0]
        if len(e):
            vs = np.concatenate([m.SFEdges[e[:, 0]], m.SFEdges[e[:, 1]]], axis=1)
            for i in range(4):
                for j in range(i + 1, 4):
                    out.append(np.stack([vs[:, i], vs[:, j]], axis=1))
    return np.concatenate(out) if out else None


def oracle_step(m, info, nthreads):
    """One Newton-iteration hot path on the CPU oracle: the same stages, in the reference's own algorithmic form
    (spatial hash with serial inserts, parallel per-primitive loops, serial merges/scatters -- oracle/hash.cpp)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle as orc
    o = orc.Elastic(m)
    s = orc.Surf(m)
    dHat, p = info["dHat"], info["p"]
    hvox = m.avgEdgeLen / 3.0
    evf, eee = orc.ti_error(s.V, m.nV, None)
    if "csr" not in info:  # untimed: sparsity pattern incl. the contact stencil (the solver's set_pattern)
        mm, pa, pe, _ = s.constraint_set_hashed(dHat, hvox, nthreads)
        info["csr"] = m.csr_pattern(1, extra_pairs=contact_pattern_pairs(m, mm, pa, pe))
    ia, ja = info["csr"]
    t0 = time.perf_counter()
    mm, pa, pe, cand = s.constraint_set_hashed(dHat, hvox, nthreads)
    o.energy(DT2, nthreads)
    s.barrier_energy(mm, pa, pe, dHat, KAPPA)
    g = o.gradient(DT2, 1, nthreads)
    s.barrier_gradient(mm, pa, pe, dHat, KAPPA, g=g)
    a = o.hessian_csr(DT2, ia, ja, 1, 1, 1, nthreads=nthreads)
    s.barrier_hessian_csr(mm, pa, pe, dHat, KAPPA, ia, ja, 1, 1, a=a, nthreads=nthreads)
    alpha, _ = o.inversion_step(p, 0.2, 1.0)
    alpha, _ = orc.ccd_partial(s, p, cand, TI_TOL, evf, eee, alpha, nthreads)
    alpha, _, _ = orc.ccd_full_hashed(s, p, alpha, hvox, TI_TOL, evf, eee, nthreads)
    return (time.perf_counter() - t0) * 1e3


def cpu_baseline(args, m, info):
    """The oracle port of the reference CPU path on the box's host cores, on the SAME full-size scene (one warm-up + 3 timed
    iterations, median; ~10-30 s of CPU work at 1M tets)."""
    cores = os.cpu_count() or 1
    oracle_step(m, info, cores)  # warm-up (page-in, thread pool, untimed sparsity pattern)
    t = sorted(oracle_step(m, info, cores) for _ in range(3))
    return {"value": t[1], "unit": "ms", "cores": cores, "kind": "port", "min": t[0],
            "sample": f"the full workload ({m.nT} tets), median of 3 Newton iterations after 1 warm-up; oracle restatement of the reference CPU "
                      f"path (-O3 -march=x86-64-v3), OpenMP over the reference's TBB loops, serial stages serial as in the reference"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path = the oracle port (the reference cannot be built here:
    Eigen/TBB/libigl/SuiteSparse/CCD-Wrapper are CPM-fetched and absent), all host threads, on the SAME config as our arm: the full
    1M-tet scene, every step one whole Newton iteration's hot path.  Rank 0 only; other ranks exit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, info = build_scene(args)
    cores = os.cpu_count() or 1
    for _ in range(args.warmup):
        oracle_step(m, info, cores)
    t = [oracle_step(m, info, cores) for _ in range(args.steps)]
    ms = float(np.mean(t))
    line = {"impl": "reference", "metric": "newton_iteration_ms_assembly_ccd", "value": ms, "unit": "ms", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "median_ms": float(np.median(t)), "min_ms": float(np.min(t)), "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"synthetic 1M-tet ball pile [{info['workload']}] ({m.nT} tets, {m.nV} verts, {len(m.SVI)} surface verts), NeoHookean, dt=0.025",
                       "stages": STAGES_RUN},
            "cpu_baseline": {"value": ms, "unit": "ms", "cores": cores, "kind": "port",
                             "sample": f"every step = the full workload ({m.nT} tets); oracle restatement of the reference CPU path, OpenMP over the reference's TBB loops"},
            "e2e": {"value": ms, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


STAGES_RUN = ["constraint_set(hash+classify)", "elastic_energy", "barrier_energy", "elastic_gradient", "barrier_gradient",
              "elastic_hessian+mass->CSR", "barrier_hessian->CSR", "inversion_step_bound", "partial_CCD(TI)", "swept_hash", "full_CCD(TI)"]
KAPPA = 1e8
TI_TOL = 1e-6


DUMP_MAX_VALUES = {"gradient": 1 << 21, "csr_values": 1 << 22}  # --dump-outputs stays under 48 MB of float64 at any --tets


def dump_outputs(path, ctx, it, n_grad, own0, own1):
    """--dump-outputs: what a caller of the timed path receives after its last step, as float64 arrays.
      gradient.npy     the gradient (elastic + barrier), summed over the ranks
      csr_values.npy   the Hessian's CSR values (elastic + mass + barrier) of the rows this rank owns (all of them on one rank)
      energy.npy       [elastic, barrier] energies of the iteration record
      step_bound.npy   [inversion, partial CCD, swept grid, full CCD, final] step bounds of the iteration record
    An array longer than DUMP_MAX_VALUES[name] is written as its values at a fixed sample of positions (seed 0, increasing order)."""
    from ipc_b200 import lib as L
    os.makedirs(path, exist_ok=True)
    out = {"gradient": ctx.download(L.BUF_GRADIENT, n_grad), "csr_values": ctx.download(L.BUF_CSR_VALUES, own1)[own0:],
           "energy": np.array([it.energy_elastic, it.energy_barrier]),
           "step_bound": np.array([it.alpha_inversion, it.alpha_partial_ccd, it.alpha_swept_grid, it.alpha_full_ccd, it.alpha])}
    for name, a in out.items():
        cap = DUMP_MAX_VALUES.get(name, a.size)
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--tets", type=int, default=1_000_000)
    ap.add_argument("--res", type=int, default=10, help="ball resolution of --scene pile: 6*res^3 tets per ball")
    ap.add_argument("--scene", default="c5", choices=["c5", "pile"], help="c5 = 146 x sphere1K.msh FCC pile (BASELINE C5 as specified), pile = round-1 synthetic column pile")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity check against the oracle (rank 0, before the warm-up)")
    ap.add_argument("--eager", action="store_true", help="enqueue every launch of the timed steps one by one instead of replaying the captured CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (rank 0, see dump_outputs)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from ipc_b200 import lib as L
    m, info = build_scene(args)
    ctx = L.Context(local_rank)
    if world > 1:
        ids = [L.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(rank, world, ids[0])
    ctx.set_mesh(m.V_rest_soa, m.T_soa, m.restTriInv, m.vol, m.mu, m.lam, m.mass, m.dbc, m.energy)
    ctx.set_surface(m.SVI, m.SFEdges, m.SF_soa, m.vCoDim)
    ctx.set_state(m.V_soa)
    dHat = info["dHat"]
    hvox = m.avgEdgeLen / 3.0  # Optimizer.cpp:259,1965
    err_vf, err_ee = L.Context.ti_error(m.V_soa, m.nV, None)  # computeTightInclusionError: mesh.V only (CCDUtils.cpp:29-46)
    # sparsity pattern incl. the contact stencil (augmentConnectivity + set_pattern are the solver's job: done once, untimed)
    mm, pa, pe, cand = ctx.constraint_set(dHat, 1)
    ia, ja = m.csr_pattern(1, extra_pairs=contact_pattern_pairs(m, mm, pa, pe))
    ctx.set_csr(ia, ja, 1)
    nnz = ja.size
    n_active, n_para, n_cand = len(mm), len(pa), len(cand)
    if world > 1:  # message of the pair-list exchange: 4x the per-rank share of the contact set the pattern was just built from, at least 4096 pairs
        xcap = 4096
        while xcap < 4 * max(n_active, n_para) // world + 1024:
            xcap *= 2
        ctx.set_exchange_capacity(min(xcap, 1 << 16))
    ctx.set_contact_partition(1)  # timed steps: every rank builds and processes only its share of the contact sets
    ctx.set_canonical_order(0)    # the sets are consumed on the device: no need for the canonical sort (the reference's order is arbitrary too)

    # pinned host buffers for the e2e path
    hV = L.PinnedArray(3 * m.nV); hV.array[:] = m.V_soa
    hp = L.PinnedArray(3 * m.nV); hp.array[:] = info["p"]
    hg = L.PinnedArray(3 * m.nV)
    ha = L.PinnedArray(nnz)
    ctx.set_state(hV.array)
    ctx.set_search_dir(hp.array)  # uploaded once: device-resident for the HBM mode

    def barrier():
        ctx.sync()
        if dist is not None:
            import torch
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()

    stats = {}
    part = ctx.partition_info()
    own0, own1 = part["value_begin"], part["value_end"]  # CSR values of the rows this rank owns (everything on one rank)

    def enqueue_iteration(download=False):
        """one Newton iteration's hot path, NULL outputs everywhere: one uninterrupted stream, nothing read back.
        download=True (the e2e form): the gradient and the CSR rows this rank owns start travelling to the pinned host buffers on the copy
        stream as soon as they are final, next to the step-bound stages that follow (joined by the fetch)"""
        ctx.constraint_set(dHat, 1, fetch=False, sizes=False)
        ctx.barrier_energy(dHat, KAPPA, want=False)
        # computeEnergyVal + computeGradient + computePrecondMtr of the elastic term in ONE pass over the tets (one SVD per tet, like the
        # reference's F / SVD cache between them); zeroes the value array first (LinSysSolver::setZero)
        ctx.elastic_energy_grad_hess(DT2, 1, 1, 1, None, None)
        ctx.barrier_gradient(dHat, KAPPA, None)
        ctx.barrier_hessian(dHat, KAPPA, 1, None)
        ctx.allreduce_grad_hess(1, 0)  # one NCCL sum of the gradient; the Hessian is complete per row owner (no-op on a single rank)
        if download:
            ctx.download_range_async(L.BUF_GRADIENT, 0, hg.array)                         # D2H: gradient
            ctx.download_range_async(L.BUF_CSR_VALUES, own0, ha.array[own0:own1])       # D2H: the CSR values of the rows this rank owns
        ctx.step_bound_set(1.0)
        ctx.inversion_step(None, 0.2, None)
        ctx.ccd_partial(None, TI_TOL, err_vf, err_ee, None)
        ctx.hash_build_swept(None, None, hvox)
        ctx.ccd_full(TI_TOL, err_vf, err_ee, None)

    def step_device():
        enqueue_iteration()
        it = ctx.fetch_iteration()  # the single synchronisation of the iteration (+ the deferred cross-rank scalars)
        stats["it"] = it

    def step_e2e():
        ctx.set_state(hV.array)        # H2D: positions
        ctx.set_search_dir(hp.array)   # H2D: search direction
        if stats.get("graph_e2e") is not None:
            ctx.graph_launch(stats["graph_e2e"])
        else:
            enqueue_iteration(download=True)
        stats["it_e2e"] = ctx.fetch_iteration()  # joins the copy stream: gradient and CSR rows are in the host buffers

    # ---- parity of exactly this mode at exactly this size, inside the run (rank 0 asserts; every rank takes part in the collectives)
    parity = None
    if not args.no_parity:
        step_device()
        it = stats["it"]
        g_dev = ctx.download(L.BUF_GRADIENT, 3 * m.nV)
        ctx.allreduce_grad_hess(0, 1)  # parity only: complete the matrix on every rank so that rank 0 can compare all of it
        a_dev = ctx.download(L.BUF_CSR_VALUES, nnz)
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle as orc
            import struct
            nth = os.cpu_count() or 1
            o, s_ = orc.Elastic(m), orc.Surf(m)
            mm_r, pa_r, pe_r, cand_r = s_.constraint_set_hashed(dHat, hvox, nth)
            E_ref = o.energy(DT2, nth)[0] + s_.barrier_energy(mm_r, pa_r, pe_r, dHat, KAPPA)[0]
            g_ref = s_.barrier_gradient(mm_r, pa_r, pe_r, dHat, KAPPA, g=o.gradient(DT2, 1, nth))
            a_ref = o.hessian_csr(DT2, ia, ja, 1, 1, 1, nthreads=nth)
            diag = np.asarray(ia[:-1:1], dtype=np.int64)[: 3 * m.nV] - 1
            a_ref[diag] += np.repeat(m.mass, 3)
            a_ref = s_.barrier_hessian_csr(mm_r, pa_r, pe_r, dHat, KAPPA, ia, ja, 1, 1, a=a_ref, nthreads=nth)
            al_r, _ = o.inversion_step(info["p"], 0.2, 1.0)
            al_p, _ = orc.ccd_partial(s_, info["p"], cand_r, TI_TOL, err_vf, err_ee, al_r, nth)
            al_f, _, npairs = orc.ccd_full_hashed(s_, info["p"], al_p, hvox, TI_TOL, err_vf, err_ee, nth)
            rel = lambda x, y: float(np.linalg.norm(x - y) / np.linalg.norm(y))
            bits = lambda x: struct.pack("<d", float(x))
            parity = {"energy_rel": abs(it.energy_elastic + it.energy_barrier - E_ref) / abs(E_ref), "gradient_rel": rel(g_dev, g_ref), "csr_rel": rel(a_dev, a_ref),
                      "alpha_partial_bits_equal": bits(it.alpha_partial_ccd) == bits(al_p), "alpha_bits_equal": bits(it.alpha) == bits(al_f),
                      "alpha": it.alpha, "alpha_oracle": al_f, "ti_warnings": int(it.ti_warnings), "ranks": world}
            ok = (parity["energy_rel"] <= 1e-10 and parity["gradient_rel"] <= 1e-10 and parity["csr_rel"] <= 1e-9 and parity["alpha_partial_bits_equal"]
                  and parity["alpha_bits_equal"] and parity["ti_warnings"] == 0)
            parity["ok"] = bool(ok)
            print("PARITY", json.dumps(parity), file=sys.stderr)
            assert ok, parity

    # ---- device-resident timing --------------------------------------------------------------------
    # The iteration is captured ONCE into a CUDA graph (every argument that changes between iterations lives in device memory) and
    # replayed: one cudaGraphLaunch + one fetch per step.  --eager times the same calls enqueued one by one instead.
    for _ in range(args.warmup):
        step_device()
    graph = None
    if not args.eager:
        ctx.capture_begin()
        enqueue_iteration()
        graph = ctx.capture_end()

        def step_device():  # noqa: F811 -- the replayed form of the function above
            ctx.graph_launch(graph)
            stats["it"] = ctx.fetch_iteration()

        for _ in range(args.warmup):
            step_device()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.5)
    n0 = ctx.launch_count()
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        step_device()
    ms_total = ctx.timer_stop()
    barrier()
    launches = ctx.launch_count() - n0
    ms_step = ms_total / args.steps
    it = stats["it"]
    if rank == 0 and args.dump_outputs:  # before the passes below overwrite the device buffers
        dump_outputs(args.dump_outputs, ctx, it, 3 * m.nV, own0, own1)
    ccd_stats = ctx.ccd_stats() + ctx.ccd_stats_ex() + ctx.ccd_stats_timing()

    # ---- per-stage table (CUDA-event pairs around every stage): a separate, eagerly enqueued pass of the same K steps -- event records
    # cannot live inside a replayed graph.  The rooflines below take their kernel times from this pass (same kernels, same inputs).
    ctx.profile(1)
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        enqueue_iteration()
        ctx.fetch_iteration()
    eager_profiled_ms = ctx.timer_stop() / args.steps
    barrier()
    prof = ctx.profile_read()
    ctx.profile(0)

    # ---- end-to-end timing (host buffers through the C ABI) -----------------------------------------
    step_e2e()  # eager once (creates the copy stream), then the e2e form of the iteration is captured like the device-resident one
    if graph is not None:
        ctx.capture_begin()
        enqueue_iteration(download=True)
        stats["graph_e2e"] = ctx.capture_end()
    for _ in range(2):
        step_e2e()
    if rank == 0:  # the host buffers hold what the device holds
        assert np.array_equal(hg.array, ctx.download(L.BUF_GRADIENT, 3 * m.nV)), "e2e gradient copy differs"
        assert np.array_equal(ha.array[own0:own1], ctx.download(L.BUF_CSR_VALUES, nnz)[own0:own1]), "e2e CSR copy differs"
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    clocks = sampler.finish() if sampler else None

    if dist is not None:
        import torch
        t = torch.tensor([ms_step, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, e2e_ms = float(t[0]), float(t[1])

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        tet_ms, tet_n = prof.get("elastic_tet", (0.0, 1))
        local_tets = part["n_assembled_tets"]  # tets this rank assembles (its share plus the boundary tets of its rows)
        per_launch_s = tet_ms / max(tet_n, 1) * 1e-3
        achieved = ALG_BYTES_PER_TET * local_tets / per_launch_s / 1e9 if per_launch_s > 0 else 0.0
        per_step = lambda k: prof.get(k, (0.0, 0))[0] / args.steps
        # Hessian-to-sink path as the CSR sees it: per-tet kernel + gradient gather + CSR assembly (incl. mass/DBC diagonal)
        h2s_ms = per_step("elastic_tet") + per_step("gather_gradient") + per_step("assemble_csr")
        h2s = ALG_BYTES_PER_TET * local_tets / (h2s_ms * 1e-3) / 1e9 if h2s_ms > 0 else 0.0
        # whole CCD narrow phase (root filter + thread pass + warp pass, both the partial and the full CCD of the step)
        n_full = int(it.n_full_ccd_candidates)
        cand_per_step = float(n_cand) / world + float(n_full)
        nar_ms = per_step("ccd_narrow")
        nar = ALG_BYTES_PER_CCD_CANDIDATE * cand_per_step / (nar_ms * 1e-3) / 1e9 if nar_ms > 0 else 0.0
        line = {
            "metric": "newton_iteration_ms_assembly_ccd", "value": ms_step, "unit": "ms", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"synthetic 1M-tet ball pile [{info['workload']}] ({m.nT} tets, {m.nV} verts, {len(m.SVI)} surface verts), NeoHookean, dt=0.025, "
                                   f"dHat=(1e-3 bboxDiag)^2, {n_active} active pairs + {n_para} mollified, {n_cand} partial-CCD candidates, "
                                   f"{n_full} full-CCD candidates on rank 0, TI tol 1e-6",
                       "stages": STAGES_RUN, "csr_nnz": int(nnz), "step_bound_alpha": it.alpha,
                       "alpha_after_inversion_partial_swept_full": [it.alpha_inversion, it.alpha_partial_ccd, it.alpha_swept_grid, it.alpha_full_ccd],
                       "energy_elastic_barrier": [it.energy_elastic, it.energy_barrier],
                       "full_ccd_candidates_survivors_warnings_deferred_boxesThreadPass_boxesWarpPass_longestPairCycles_totalCycles": list(ccd_stats),
                       "l2": "working set (78 doubles/tet = %.0f MB + CSR %.0f MB) exceeds the 126 MB L2" % (m.nT * 624 / 1e6, nnz * 8 / 1e6),
                       "mode": ("device-resident iteration: every stage in its NULL-output form, one ipcgpu_fetch_iteration per step; canonical_order=0, "
                                "contact_partition=1; " + ("the iteration is captured once into a CUDA graph and replayed (one cudaGraphLaunch per step)"
                                                           if graph is not None else "launches enqueued one by one (--eager)")),
                       "eager_profiled_ms_per_step": eager_profiled_ms,
                       "stage_ms_source": "a separate eagerly enqueued pass of the same steps with CUDA-event pairs around every stage (events cannot be recorded inside a replayed graph)",
                       "partition": (f"{world} rank(s): tets block-partitioned (energy, inversion); gradient/Hessian by row owner (rank 0 assembles {local_tets} tets, "
                                     f"CSR values [{own0},{own1}) of {nnz}); queries of both broad phases partitioned; NCCL: allgather of the pair lists, "
                                     "sum-allreduce of the gradient, min-allreduce of each step bound; no Hessian reduction")},
            "stage_ms": {k: v[0] / args.steps for k, v in prof.items()},
            "sum_stage_ms": sum(v[0] for k, v in prof.items() if k != "ccd_root_filter") / args.steps,
            "roofline": {"bound": "hbm", "kernel": "k_elastic_grad_hess<NH,g,H>", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": achieved / peak_gbs, "traffic": (NCU_TET["dram_bytes"] / m.nT * local_tets) if NCU_TET and NCU_TET.get("dram_bytes") else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_tet": ALG_BYTES_PER_TET, "algorithmic_bytes_per_launch": ALG_BYTES_PER_TET * local_tets,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of the committed `ncu --set full` capture of this command at N = 1 "
                                           "(1,000,246 tets per launch), scaled to the tets this rank assembles",
                         "kernel_ms": tet_ms / max(tet_n, 1), "ncu": NCU_TET},
            "roofline_hessian_to_csr": {"bound": "hbm", "kernel": "k_elastic_grad_hess + k_gather_gradient + k_assemble_csr + k_diag_mass_dbc (what the CSR sink sees)",
                                        "achieved": h2s, "peak": peak_gbs, "unit": "GB/s", "frac": h2s / peak_gbs,
                                        "traffic": ((NCU_TET["dram_bytes"] + NCU_ASM["dram_bytes"]) / m.nT * local_tets) if NCU_TET and NCU_ASM and NCU_TET.get("dram_bytes") and NCU_ASM.get("dram_bytes") else None,
                                        "ncu_assemble": NCU_ASM,
                                        "algorithmic_bytes_per_tet": ALG_BYTES_PER_TET, "path_ms_per_step": h2s_ms},
            "roofline_ccd_narrow": {"bound": "hbm", "kernel": "k_ti_stage1 + k_ti_stage15 + k_ti_stage2 (whole Tight-Inclusion narrow phase, partial + full CCD)",
                                    "achieved": nar, "peak": peak_gbs, "unit": "GB/s", "frac": nar / peak_gbs, "traffic": None,
                                    "algorithmic_bytes_per_candidate": ALG_BYTES_PER_CCD_CANDIDATE, "candidates_per_step": cand_per_step, "path_ms_per_step": nar_ms,
                                    "root_filter_ms_per_step": per_step("ccd_root_filter"), "ncu": NCU_TI,
                                    "note": "latency/ALU-bound interval search on the surviving pairs (SURVEY 8d): the vertex data is L2-resident and the "
                                            "critical path is the deepest pair, so the HBM fraction only says how far from a pure streaming pass the stage is"},
            "e2e": {"value": e2e_ms, "unit": "ms", "h2d_bytes_per_step": int(2 * 3 * m.nV * 8), "d2h_bytes_per_step": int((3 * m.nV + (own1 - own0)) * 8 + 120),
                    "note": "host clock around: H2D of x and p (pinned), the whole iteration (graph replay), D2H of the gradient and of the CSR values of the rows "
                            "this rank owns (rank 0's byte counts) -- forked onto a copy stream as soon as they are final, i.e. next to the step-bound stages, "
                            "and joined by the fetch; checked equal to the device arrays after the warm-up"},
            "parity": parity,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, m, info)
        print(json.dumps(line))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
