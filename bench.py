#!/usr/bin/env python
"""bench.py — local-BA iterations/sec at 1 M pts/scan, 50-frame window (BASELINE.json metric), on N GPUs of one node.

A "step" is ONE Levenberg–Marquardt iteration of the sliding-window LiDAR-inertial BA (LI_BA_Optimizer::damping_iter body,
voxel_map.hpp:581-649): Hessian build over the voxel factor (+ the CPU-side IMU blocks through the callback), gauge fix,
damped LDL^T solve of the 15W system, state retraction, residual-only evaluation — i.e. one vxs_li_ba(max_iter=1) call.

  value : K steps with the voxel factor already resident in HBM (built on the GPU from the synthetic scans before timing).
  e2e   : the reference-facing call with HOST buffers: push the host LidarFactor (pinned CSR arrays, H2D), run the
          reference's 3-iteration damping_iter, read back poses + Hessian + the factor side effects (eig / pcr_adds) —
          iterations actually executed / time.
  N > 1 : one process per GPU (torchrun); the window does not need a collective (SURVEY §8e / north_star restrict the
          all-reduce to global BA), so every rank solves its own independent window: "replicas", weak scaling.
  --impl reference : the CPU restatement of the reference (oracle/, 5 threads as the reference hard-codes) on the same window
          geometry, rank 0 only.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))   # synth (scene generator / IMU stand-in) and oracle_api (CPU baseline legs only)

import synth  # noqa: E402  (tests/synth.py: seeded scenes + IMU stand-in; test / bench infrastructure)

METRIC = "local-BA LM iterations/sec (W=50 window, 1M pts/scan)"
UNIT = "iterations/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi samples DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, device):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def scene_points(vx, W, pts, L, seed):
    tr = np.stack([synth.true_pose(L, i) for i in range(W)])
    est = tr.copy()
    for i in range(1, W):
        # odometry-grade initial error.  SURVEY §8d suggests (2e-3 rad, 1e-2 m); at L=130 m a 2e-3 rad error moves far points by 0.2 m,
        # which breaks every plane of the initial map (the window leaves the convergence basin and k collapses), so the rotation
        # noise is scaled with the lever arm: 1e-4 rad * 90 m = 9 mm, the size of the point noise.
        est[i] = synth.perturb_pose(tr[i], seed * 1000 + i, 1e-4, 5e-3)
    p = np.empty((W * pts, 3), dtype=np.float64)
    for i in range(W):
        synth.gen_scan(L, i, pts, tr[i], seed=0x5EED0000 + seed, out=p[i * pts:(i + 1) * pts])
    off = np.arange(W + 1, dtype=np.int64) * pts
    return tr, est, p, off


def states_from(poses):
    s = np.zeros((poses.shape[0], 24))
    s[:, :12] = poses
    s[:, 12:15] = (0.5, 0.3, 0.0)
    s[:, 21:24] = (0.0, 0.0, -9.8)
    return s


def dist_setup(args):
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep stdout to the one JSON line (NCCL prints its version banner there otherwise)
        import torch
        import torch.distributed as dist_
        torch.cuda.set_device(local)
        dist_.init_process_group(backend="nccl" if args.impl != "reference" else "gloo")
        dist = dist_
    return rank, world, local, dist


def barrier_max(dist, local, value):
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{local}" if dist.get_backend() == "nccl" else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(dist, local):
    if dist is not None:
        import torch
        if dist.get_backend() == "nccl":
            torch.cuda.synchronize(local)
        dist.barrier()


# ---------------------------------------------------------------------------------------------------------------- ours
def run_ours(args):
    import voxel_slam_b200 as vx
    from voxel_slam_b200 import api
    rank, world, local, dist = dist_setup(args)
    W, pts, L, K, Wu = args.win, args.pts_per_scan, args.L, args.steps, args.warmup
    ctx = vx.Context(local)
    t0 = time.time()
    tr, est, p, off = scene_points(vx, W, pts, L, seed=1 + rank)
    t_gen = time.time() - t0
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    f = vx.Factor(ctx, W)
    ctx.timing(True); ctx.timing_reset()
    t0 = time.time()
    nvox = ctx.build_window_factor(mp, p, off, est, f)
    t_vox = time.time() - t0
    vox_stages = ctx.timing_read(); ctx.timing(False)
    V, E, _ = f.counts()
    log(f"[rank {rank}] scene W={W} pts/scan={pts} L={L}: generated in {t_gen:.1f}s; GPU map build {t_vox * 1e3:.1f} ms -> V={V} voxels, E={E} entries (k={E / max(V, 1):.1f})")
    del p
    # host copy of the factor exactly as the map build left it (cached eig / pcr_adds at the cut poses) — the e2e leg pushes this
    ptr, fr, cl, fx, co = f.read_structure()
    eig0, sum0 = f.read_back()
    f.cache_save()
    st0 = states_from(est)
    imu = synth.ImuWindow(tr)
    n = 15 * W

    def step():
        # every step is the FIRST LM iteration from the same map state: the factor's cached eig / pcr_adds are restored on the
        # device (9 MB D2D copy inside the timed region) so the step is accepted for the same reason each time
        imu.reset()
        f.cache_restore()
        return ctx.li_ba(f, st0, imu, with_gravity=False, max_iter=1, want_hess=False, trace_cap=4)

    # ---- value: K steps, factor resident in HBM
    sampler = ClockSampler(local); sampler.start()
    first_step = step()
    for _ in range(max(Wu, 3) - 1):
        step()
    launches0 = ctx.launches
    barrier(dist, local)
    ctx.timer_start()
    for _ in range(K):
        last = step()
    ms = ctx.timer_stop()
    if args.dump_outputs and rank == 0:
        eig_last, sum_last = f.read_back()          # the factor cache the last step left behind (read before any later step overwrites it)
        dump_outputs(args.dump_outputs, last, eig_last, sum_last)
    ms = barrier_max(dist, local, ms)
    clocks = sampler.stop()
    launches = ctx.launches - launches0
    value = world * K / (ms * 1e-3)

    # ---- per-kernel durations (CUDA events around every launch on the ctx stream), same steps
    ctx.timing(True); ctx.timing_reset()
    reps = min(K, 10)
    for _ in range(reps):
        step()
    stages = ctx.timing_read(); ctx.timing(False)
    kern = {k: {"ms_per_step": v[0] / reps, "launches_per_step": v[1] / reps, "us_per_launch": v[0] / max(v[1], 1) * 1e3} for k, v in stages.items() if v[1] > 0}

    # ---- e2e: host LidarFactor in, 3-iteration damping_iter, results out
    hp = dict(ptr=api.pinned_array(ptr.shape, np.int64), fr=api.pinned_array(fr.shape, np.int32), cl=api.pinned_array(cl.shape, np.float64),
              eig=api.pinned_array(eig0.shape, np.float64), s=api.pinned_array(sum0.shape, np.float64))
    hp["ptr"][:] = ptr; hp["fr"][:] = fr; hp["cl"][:] = cl; hp["eig"][:] = eig0; hp["s"][:] = sum0
    out_eig, out_sum = api.pinned_array(eig0.shape, np.float64), api.pinned_array(sum0.shape, np.float64)
    del cl

    def e2e_call():
        imu.reset()
        f.clear()
        f.push_voxels_async(hp["ptr"], hp["fr"], hp["cl"], hp["eig"], hp["s"])     # pinned host LidarFactor; first Hessian runs behind the upload chunks
        o = ctx.li_ba(f, st0, imu, with_gravity=False, max_iter=3, want_hess=True, trace_cap=8)
        api.lib().vxs_factor_read_back(f._p, out_eig.ctypes.data_as(C.POINTER(C.c_double)), out_sum.ctypes.data_as(C.POINTER(C.c_double)))
        return o

    o = e2e_call()
    Ke = max(3, min(K, 10))
    barrier(dist, local)
    t0 = time.perf_counter(); ctx.timer_start()
    iters = 0
    for _ in range(Ke):
        iters += len(e2e_call()["trace"])
    ms_e = ctx.timer_stop()
    wall_e = (time.perf_counter() - t0) * 1e3
    ms_e = barrier_max(dist, local, max(ms_e, wall_e))
    e2e_value = world * iters / (ms_e * 1e-3)
    it_call = iters / Ke
    h2d = (ptr.nbytes + fr.nbytes + E * 80 + V * (96 + 80)) / it_call + W * 24 * 8 * 2 + (W - 1) * (900 + 30) * 8
    d2h = (V * 176 + n * n * 8) / it_call + (3 * n + 2) * 8

    # ---- sanity of what was timed: the 3-iteration solve moves the poses towards the truth
    err0, err1 = float(np.abs(est - tr).max()), float(np.abs(o["states"][:, :12] - tr).max())

    # ---- roofline (HBM) for the kernels of the hot path; algorithmic bytes per SURVEY.md §8(d)
    peaks, src = measured_peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    fp64_peak = ctx.fp64_tflops()
    kv = E / max(V, 1)

    def roof(names, bytes_per_launch, flops=None):
        t = sum(kern[k]["ms_per_step"] for k in names if k in kern)
        if t <= 0:
            return None
        r = {"kernel": "+".join(names), "bound": "hbm", "achieved": bytes_per_launch / (t * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": bytes_per_launch / (t * 1e-3) / 1e9 / hbm,
             "traffic": None, "ms": t, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({src})", "algorithmic_bytes": bytes_per_launch}
        if flops:
            r["fp64"] = {"achieved_tflops": flops / (t * 1e-3) / 1e12, "peak_tflops": fp64_peak, "frac": flops / (t * 1e-3) / 1e12 / fp64_peak, "peak_source": "vxs_diag_fp64_tflops (measured here)"}
        return r

    nl = 6 * W
    bytes_resid = E * 80 + V * 176 + 96 * W
    bytes_hess = E * 80 + V * 176 + 8 * (nl * nl + nl + 1)
    flops_hess = V * (700.0 * kv + 110.0 * kv * kv)
    roof_hess = roof(["k_jac", "k_syrk"], bytes_hess, flops_hess)
    resid_names = ["k_residual_stream"] if "k_residual_stream" in kern else ["k_cluster_sum", "k_eig_residual"]
    roof_resid = roof(resid_names, bytes_resid)
    roof_jac = roof(["k_jac"], E * 80 + V * 176 + E * 144)
    if roof_jac is not None:   # SURVEY §8(d) counts only the cluster reads (k*80 + 176 B / voxel); the 144 B / entry of rank-3 rows written for the SYRK are this design's own intermediate
        roof_jac["bytes_counted"] = "k*80 + 176 B read + k*144 B written per voxel (the X rows the SYRK consumes)"
        roof_jac["frac_survey_8d_bytes_only"] = (E * 80 + V * 176) / (roof_jac["ms"] * 1e-3) / 1e9 / hbm
    # the dominant kernel (k_syrk: H -= X^T X on the fp64 tensor path) is compute-bound for k >~ 4 (SURVEY.md §7.3 / §8d "report both"):
    # its roofline is the fp64 mma.sync (DMMA) throughput measured in this process; the HBM view of the whole Hessian build rides along
    roof_main = roof_hess
    if "k_syrk" in kern and kern["k_syrk"]["ms_per_step"] > 0:
        try:
            dmma_peak = ctx.dmma_tflops()
        except Exception:
            dmma_peak = fp64_peak
        t_sy = kern["k_syrk"]["ms_per_step"] * 1e-3 / max(kern["k_syrk"]["launches_per_step"], 1.0)
        fl_sy = V * 108.0 * kv * kv / max(kern["k_syrk"]["launches_per_step"], 1.0)      # 3 rank-1 rows x (6k)^2 / 2 MACs per voxel
        roof_main = {"kernel": "k_syrk", "bound": "tensor", "achieved": fl_sy / t_sy / 1e12, "peak": dmma_peak, "unit": "TFLOP/s", "frac": fl_sy / t_sy / 1e12 / dmma_peak,
                     "traffic": ncu_traffic(["k_syrk"]), "peak_source": "vxs_diag_dmma_tflops: mma.sync.m8n8k4.f64 (SASS DMMA) throughput measured in this process; "
                     "MEASURED_PEAKS.json carries no fp64 figure", "algorithmic_flops": fl_sy, "us_per_launch": t_sy * 1e6,
                     "traffic_source": "profiles/r02_ncu_full_ba_kernels.txt (ncu --set full of this command, DRAM read + write per launch)",
                     "hbm_view_of_hessian_build": roof_hess,
                     "note": "the dominant kernel of the step is compute-bound on the fp64 tensor path; the HBM fractions the north_star names for the residual / Jacobian kernels are the "
                             "`roofline_residual` and `roofline_jac` keys of this line"}
    for r_, names_ in ((roof_hess, ["k_jac_slab", "k_syrk"]), (roof_resid, resid_names), (roof_jac, ["k_jac_slab"])):
        if r_ is not None:
            r_["traffic"] = ncu_traffic(names_)
            r_["traffic_source"] = "profiles/r02_ncu_full_ba_kernels.txt (ncu --set full of this command, DRAM read + write per launch)"
    dom = max(kern.items(), key=lambda kv_: kv_[1]["ms_per_step"])[0] if kern else None

    c2 = ds = None
    if rank == 0 and world == 1:
        c2 = c2_leg(vx, ctx, hbm)
        ds = ds_leg(ctx)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_from_structure(vx, W, ptr, fr, hp["cl"], eig0, sum0, st0, tr, reps=2)
    # ---- parity of what was timed, at the metric shape itself (the oracle is the checker here, never the thing measured)
    parity = None
    if rank == 0:
        try:
            parity = parity_block(vx, ctx, W, ptr, fr, hp["cl"], eig0, sum0, est, first_step, cpu)
        except Exception as e:   # never lose the bench line over the checker
            parity = {"error": repr(e)}
    # ---- the full local-mapping step on the persistent device map (SURVEY §8d "also report the full local-mapping step")
    lmap = None
    if rank == 0 and world == 1 and not args.no_local_mapping:
        try:
            f.close()
            lmap = local_mapping_leg(vx, ctx, W, pts, L, args.lm_steps)
        except Exception as e:
            lmap = {"error": repr(e)}
    # ---- the path that shards: one voxel-sharded global-BA window over all ranks, NCCL all-reduce of the pose Hessian (strong scaling)
    gba = None
    if not args.no_gba:
        try:
            gba = hba_leg(vx, local, rank, world, dist, args)
        except Exception as e:
            import traceback
            gba = {"error": repr(e), "trace": traceback.format_exc()[-1500:]}
        if args.gba_window_leg:
            try:
                gba["dense_window"] = gba_sharded_leg(vx, local, rank, world, dist, args)
            except Exception as e:
                gba["dense_window"] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(Wu, 3), "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic (seeded 3-plane room, SURVEY.md §8d; random-free IMU stand-in on the CPU callback)",
            "config": {"workload": f"metric shape M: W={W} window, {pts} pts/scan, L={L} m room, voxel 1 m, max_layer 2 -> V={V} plane voxels, E={E} (voxel,frame) clusters; n=15W={n} LI-BA system",
                       "step": "one LM iteration = vxs_li_ba(max_iter=1): Hessian build + IMU blocks (CPU callback) + damped LDLT + retraction + residual evaluation",
                       "l2": "working set (clusters 80 B x E + rank-3 rows 144 B x V x W) is larger than the 126 MB L2; no extra flush",
                       "parallelism": "replicas: one independent window per GPU, no collective" if world > 1 else "1 GPU"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "iterations_per_call": it_call,
                    "call": "vxs_factor_push_voxels_async of the host LidarFactor (pinned CSR, 4 chunks overlapped with the first Hessian build) + LI_BA damping_iter (3 iterations) + read back poses, Hessian, eig/pcr_adds"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roof_main, "roofline_residual": roof_resid, "roofline_jac": roof_jac, "dominant_kernel": dom,
            "kernels": kern, "cpu_baseline": cpu, "parity": parity, "local_mapping": lmap, "gba": gba, "c2_plane_fit": c2, "down_sampling": ds,
            "voxelize": {"ms_total": t_vox * 1e3, "points": int(W * pts), "stages_ms": {k: v[0] for k, v in vox_stages.items() if v[1] > 0}},
            "check": {"pose_err_before": err0, "pose_err_after_3_iters": err1, "trace": [[float(t["r1"]), float(t["r2"]), int(t["accepted"])] for t in o["trace"]]},
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(out_dir, o, eig12, sum10, cap=DUMP_CAP_BYTES):
    """What the last timed step returned to its caller, as DIR/<name>.npy (float64): the LI-BA states, the residual pair, the LM trace
    (r1, r2, u, v, q1, accepted, hess_built per iteration) and the factor cache the step leaves behind (eig12 / sum10 per voxel, what the
    reference's LidarFactor holds after damping_iter).  Inputs are seeded, so two builds run with the same arguments can be compared file by file;
    the fp64 atomic sums make even two runs of one build differ in the last bits (relative ~1e-9 on the smallest eigenvalues of eig12).
    Above `cap` bytes in all, the per-voxel arrays are replaced by the same fixed, seeded sample of voxels, whose indices go to voxel_index.npy."""
    tr = o["trace"]
    arrays = {"states": o["states"], "resis": o["resis"],
              "trace": np.stack([tr[k].astype(np.float64) for k in ("r1", "r2", "u", "v", "q1", "accepted", "hess_built")], axis=1).reshape(-1, 7)}
    per_voxel = {"factor_eig12": eig12, "factor_sum10": sum10}
    fixed = sum(a.nbytes for a in arrays.values())
    row_bytes = sum(a[0].nbytes for a in per_voxel.values())
    V = len(eig12)
    if fixed + V * row_bytes > cap:
        keep = max(0, (cap - fixed - 4096) // (row_bytes + 8))   # + 8 B per voxel for voxel_index.npy, 4 KB for the .npy headers
        sel = np.sort(np.random.default_rng(0).choice(V, keep, replace=False))
        per_voxel = {k: a[sel] for k, a in per_voxel.items()}
        arrays["voxel_index"] = sel.astype(np.float64)
    arrays.update(per_voxel)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))
    log(f"[dump] {len(arrays)} arrays, {sum(a.nbytes for a in arrays.values())} bytes -> {out_dir}")


def parity_block(vx, ctx, W, ptr, fr, cl, eig, s, est, first_step, cpu):
    """CUDA vs oracle AT the metric shape: (1) acc_evaluate2 on an evenly spaced ~2 % voxel sample (same sample on both sides: Hessian, gradient,
    residual), (2) the first LM iteration of the timed step against the oracle's full-size iteration that cpu_baseline ran (r1, r2, state increment)."""
    import oracle_api as oa
    V = ptr.shape[0] - 1
    sel = np.linspace(0, V - 1, max(64, V // 50)).astype(np.int64)
    cnt = np.diff(ptr)[sel]
    ent = np.concatenate([np.arange(ptr[v], ptr[v + 1]) for v in sel])
    sp = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    fs = vx.Factor(ctx, W)
    fs.push_voxels(sp, fr[ent], np.ascontiguousarray(cl[ent]), eig[sel], s[sel])
    H, J, r = ctx.evaluate_hessian(fs, est)
    fs.close()
    of = oracle_factor_from_csr(W, sp, fr[ent], cl[ent], eig[sel], s[sel])
    Hr, Jr, rr = of.hessian(est)
    rel = lambda a, b: float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(b)), 1e-300))
    out = {"shape": f"W={W}, V={V}", "hessian_sample": {"voxels": int(len(sel)), "H_relinf": rel(H, Hr), "g_relinf": rel(J, Jr), "residual_rel": abs(r - rr) / abs(rr)},
           "tolerance": "north_star: 1e-5 relative on residuals / solved increments; fp64 kernels are far inside"}
    if cpu is not None and cpu.get("first_iteration") is not None:
        o = cpu["first_iteration"]
        g = first_step
        blk = lambda a, lo, hi: np.asarray(a)[:, lo:hi]
        inc = lambda lo, hi: float(np.max(np.abs(blk(o["states"], lo, hi) - blk(o["st0"], lo, hi))))
        dif = lambda lo, hi: float(np.max(np.abs(blk(g["states"], lo, hi) - blk(o["states"], lo, hi))))
        out["first_iteration"] = {"r1_rel": abs(g["trace"][0]["r1"] - o["r1"]) / o["r1"], "r2_rel": abs(g["trace"][0]["r2"] - o["r2"]) / o["r2"],
                                  "accepted": [int(g["trace"][0]["accepted"]), int(o["accepted"])],
                                  "dx_rel_pose": dif(0, 12) / max(inc(0, 12), 1e-300), "dx_inf_pose": inc(0, 12),
                                  "dx_rel_v_bg_ba": dif(12, 21) / max(inc(12, 21), 1e-300), "dx_inf_v_bg_ba": inc(12, 21),
                                  "per_block_abs_diff": {"R": dif(0, 9), "p": dif(9, 12), "v": dif(12, 15), "bg": dif(15, 18), "ba": dif(18, 21)},
                                  "per_block_increment": {"R": inc(0, 9), "p": inc(9, 12), "v": inc(12, 15), "bg": inc(15, 18), "ba": inc(18, 21)}}
        cpu.pop("first_iteration")
    return out


def local_mapping_leg(vx, ctx, W, pts, L, steps):
    """One step of the sliding-window local-mapping loop (voxelslam.cpp:1599-1712) on the persistent device map, window full:
    vxs_map_push_scan (upload of ONE scan from pinned memory, cut_voxel_multi, multi_recut, tras_opt) -> LI_BA damping_iter (<= 3 iterations, IMU
    callbacks on the CPU) -> vxs_map_margi (multi_margi, plane_update, ring rotation).  Round 1 rebuilt the whole window per scan (~120 ms)."""
    from voxel_slam_b200 import api
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    dm = vx.LocalMap(ctx, mp, W, max_points=100)
    f = vx.Factor(ctx, W)
    nscan = W - 1 + steps + 4
    pv = api.pinned_array((pts, 12), np.float64)
    pv[:, 3:] = 0.0
    pv[:, [3, 7, 11]] = 1e-4
    xyz_tmp = np.empty((pts, 3), dtype=np.float64)
    x_buf, tr_buf = [], []
    t_fill = time.perf_counter()
    stage_ms = {}
    walls, iters = [], 0
    odom, odom_err = [], []
    for i in range(nscan):
        tr = synth.true_pose(L, i)
        est = synth.perturb_pose(tr, 77000 + i, 1e-4, 5e-3) if i else tr
        synth.gen_scan(L, i, pts, tr, seed=0x5EED0000 + 9, out=xyz_tmp)       # the generator writes a contiguous xyz array
        pv[:, :3] = xyz_tmp
        x_buf.append(est); tr_buf.append(tr)
        timed = i >= W - 1 + 4                              # window full and four warm steps behind us (the map's pools have reached their steady size)
        if timed:
            ctx.timing(True); ctx.timing_reset()
        if timed:
            # side measurement on the same scan (SURVEY §8f rank 3, the step BEFORE the map update): var_init -> 4 EKF association passes against the resident map
            # (voxelslam.cpp:860-918 runs up to num_max_iter = 4) -> pvec_update, the scan staying on the device in between.  Own try block: it must never cost the main leg.
            try:
                cloud32 = np.ascontiguousarray(xyz_tmp, dtype=np.float32)
                rot_var, tsl_var = np.eye(3) * 1e-6, np.eye(3) * 1e-4
                ta = time.perf_counter()
                ctx.var_init(cloud32, np.eye(3), np.zeros(3), 0.02, 0.05, want_out=False)
                tb = time.perf_counter()
                matched = 0
                for _ in range(4):
                    matched = dm.odom_accumulate(None, est, rot_var, tsl_var, n=pts, want_flags=False)["n"]
                tc = time.perf_counter()
                ctx.pvec_update(None, est, rot_var, tsl_var, n=pts, want_pv=False, want_pwld=False)
                td = time.perf_counter()
                odom.append(((tb - ta) * 1e3, (tc - tb) * 1e3 / 4, (td - tc) * 1e3, matched / float(pts)))
            except Exception as e:          # noqa: BLE001
                odom_err.append(repr(e))
        t0 = time.perf_counter()
        dm.push_scan(pv, np.stack(x_buf), f)
        t1 = time.perf_counter()
        if len(x_buf) >= W:
            st = states_from(np.stack(x_buf))
            imu = synth.ImuWindow(np.stack(tr_buf))
            o = ctx.li_ba(f, st, imu, with_gravity=False, max_iter=3, want_hess=False, trace_cap=8)
            t2 = time.perf_counter()
            xs = o["states"][:, :12]
            dm.margi(xs, f, mgsize=1)
            x_buf = [p for p in xs[1:]]; tr_buf = tr_buf[1:]
            t3 = time.perf_counter()
            if timed:
                walls.append((t1 - t0, t2 - t1, t3 - t2)); iters += len(o["trace"])
                for k, v in ctx.timing_read().items():
                    if v[1] > 0:
                        stage_ms[k] = stage_ms.get(k, 0.0) + v[0]
                ctx.timing(False)
    w = np.array(walls) * 1e3
    c = dm.counts()
    V, E, _ = f.counts()
    res = {"workload": f"W={W} window full, {pts} pts/scan, L={L}: push_scan + LI-BA (<=3 it) + margi per new scan; map holds {c['nodes']} nodes, {c['fix_points']} point_fix points; factor V={V}, E={E}",
           "steps": int(len(walls)), "steps_per_s": float(1e3 / w.sum(axis=1).mean()), "ms_per_step": float(w.sum(axis=1).mean()), "ms_per_step_median": float(np.median(w.sum(axis=1))),
           "ms_per_step_each": [round(float(x), 2) for x in w.sum(axis=1)],
           "ms_push_scan": float(w[:, 0].mean()), "ms_ba": float(w[:, 1].mean()), "ms_margi": float(w[:, 2].mean()), "lm_iterations_per_step": iters / max(len(walls), 1),
           "h2d_bytes_per_step": int(pts * 96), "timing": "host wall clock around the three synchronous C-ABI calls (pinned host scan; includes the 96 MB H2D)",
           "kernel_ms_per_step": {k: v / max(len(walls), 1) for k, v in sorted(stage_ms.items(), key=lambda kv: -kv[1])[:14]},
           "round1_from_scratch_rebuild_ms": 120.0, "fill_s": time.perf_counter() - t_fill}
    if odom:
        o_ = np.array(odom)
        res["odometry_front"] = {"what": "per scan, host wall around the C-ABI calls: vxs_var_init (12 MB float cloud up, records stay resident), one EKF association pass of vxs_map_odom_accumulate "
                                         "(mean of 4, against the resident map's plane rows), vxs_pvec_update (resident)",
                                 "ms_var_init": float(o_[:, 0].mean()), "ms_ekf_pass": float(o_[:, 1].mean()), "ms_pvec_update": float(o_[:, 2].mean()), "matched_fraction": float(o_[:, 3].mean()),
                                 "points": int(pts)}
    elif odom_err:
        res["odometry_front"] = {"error": odom_err[0]}
    dm.close(); f.close()
    return res


def hba_leg(vx, local, rank, world, dist, args):
    """The hierarchical global-BA step (SURVEY §8e, north_star; thd_globalmapping voxelslam.cpp:2484-2557) on K keyframes, STRONG scaling:
      bottom : every window of 10 keyframes (stride 5) = HBA_add_edge(max_iter 1): map build + Lidar_BA damping_iter(up 4) + PGO edges — vxs_hba_bottom_batch on this rank's
               share of the windows (windows are independent: no collective) — then the submap merge + down-sampling of those windows (vxs_submap_merge_batch);
      gather : the merged submap clouds go to every rank (NCCL all-gather through torch.distributed, device buffers);
      top    : ONE BA over all submaps (W = number of windows), HBA_add_edge(total_max_iter 1): the voxel map is sharded over the ranks by the hash of the root cell and
               [C | g | D | r] is all-reduced by libvxs' own NCCL communicator once per Hessian build; the 6W-dof LDLT is replicated.
    A step is one full pass; time = max over ranks."""
    from voxel_slam_b200 import api
    if world > 1:
        import torch
    K, n, per_row = args.hba_keyframes, args.hba_pts, args.hba_per_row
    ws, stride_w = 10, 5
    ctx = vx.Context(local)
    if world > 1:
        uid = [vx.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
    t0 = time.time()
    tr = np.stack([synth.lawnmower_pose(i, per_row) for i in range(K)])
    est = np.stack([tr[0]] + [synth.perturb_pose(tr[i], 100 + i, 1e-3, 1e-2) for i in range(1, K)])
    xyz = api.pinned_array((K * n, 3), np.float32)
    for i in range(K):
        synth.gen_scan_city(i, n, tr[i], rng_m=args.hba_range, out=xyz[i * n:(i + 1) * n])
    off = np.arange(K + 1, dtype=np.int64) * n
    t_gen = time.time() - t0
    fine = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    from voxel_slam_b200 import sharding
    win_first = sharding.hba_windows(K, ws, stride_w)
    nwin = len(win_first)
    lo, hi = sharding.window_share(nwin, rank, world)
    mine = win_first[lo:hi]
    dev = f"cuda:{local}"
    ph = {}
    per_step = []

    coarse = fine      # total_max_iter = 1 (GBA/total_max_iter default, voxelslam.cpp:2493): the single outer iteration already uses the fine parameters

    def step():
        t0_ = time.perf_counter()
        o = ctx.hba_pass(coarse, fine, xyz, off, est, win_size=ws, win_stride=stride_w, top_max_iter=1, nranks=world, rank=rank)
        wall = (time.perf_counter() - t0_) * 1e3
        for k, name in enumerate(("bottom_ms", "merge_ms", "exchange_ms", "top_ms")):
            ph[name] = ph.get(name, 0.0) + float(o["phase_ms"][k])
        ph["wall_ms"] = ph.get("wall_ms", 0.0) + wall
        per_step.append([round(float(x), 2) for x in o["phase_ms"][:4]] + [round(wall, 2)])
        return o

    o = step()          # warm-up passes: allocations settle (buffers keep 1/8 head room), NCCL opens its peer channels on first use
    step()
    step()
    ph.clear()
    barrier(dist, local)
    steps = args.hba_steps
    t0 = time.perf_counter()
    for _ in range(steps):
        o = step()
    ms = (time.perf_counter() - t0) * 1e3
    ms = barrier_max(dist, local, ms)
    mine_ph = [ph[k] / steps for k in ("bottom_ms", "merge_ms", "exchange_ms", "top_ms", "wall_ms")]
    per_rank = [mine_ph]
    if dist is not None:
        g = [torch.zeros(5, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor(mine_ph, dtype=torch.float64, device=dev))
        per_rank = [x.cpu().tolist() for x in g]
    # sanity: the bottom windows move their keyframes towards the truth (relative to the window's fixed first keyframe)
    k0 = int(win_first[lo]) if hi > lo else 0
    e0 = float(np.abs(est[k0 + 1:k0 + ws, 9:] - tr[k0 + 1:k0 + ws, 9:]).max()); e1 = float(np.abs(o["bottom_poses"][0][1:, 9:] - tr[k0 + 1:k0 + ws, 9:]).max())
    res = {"metric": "hierarchical global-BA passes/sec (bottom windows distributed + top level voxel-sharded; strong scaling)", "value": steps / (ms * 1e-3), "unit": "passes/s",
           "keyframes_per_s": K * steps / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "scaling": "strong", "n_gpus": world,
           "workload": f"C4-like: {K} keyframes x {n} pts (city grid, lawn-mower path, {args.hba_range} m sensor range), {nwin} bottom windows of {ws} (stride {stride_w}), top level W={nwin} (n={6 * nwin}); "
                       f"{int(o['submap_sizes'].sum())} submap points after the merge",
           "call": "vxs_hba_pass: host keyframe clouds (pinned) in; bottom BA + merge on this rank's windows, submaps exchanged device to device (NCCL), top level sharded; poses / edges out",
           "per_rank_[bottom,merge,exchange,top,wall]_ms": [[round(x, 2) for x in r] for r in per_rank],
           "per_step_[bottom,merge,exchange,top,wall]_ms_rank0": per_step[-steps:],
           "bottom": {"windows_this_rank": int(hi - lo), "plane_voxels_this_rank": int(o["phase_ms"][4]), "clusters_this_rank": int(o["phase_ms"][5]), "status_ok": int(np.sum(o["bottom_status"][: hi - lo] == 0)), "edges_mean": float(np.mean(np.sum(o["edge_valid"][: hi - lo], axis=1))),
                      "pos_err_first_window_before_after": [e0, e1]},
           "top": {"outer_iters": int(o["top_outer_iters"]), "resis": [float(x) for x in o["top_resis"][:2]],
                   "pos_err_submaps_before_after": [float(np.abs(est[win_first][1:, 9:] - tr[win_first][1:, 9:]).max()), float(np.abs(o["top_poses"][1:, 9:] - tr[win_first][1:, 9:]).max())]},
           "comm": "libvxs' own NCCL communicator (vxs_ctx_comm_init): sizes all-reduce + grouped broadcasts of the submaps + all-reduce of [C | g | D | r] per top-level Hessian build" if world > 1 else "single GPU: no collective",
           "scene_gen_s": t_gen}
    ctx.close()
    return res


def gba_sharded_leg(vx, local, rank, world, dist, args):
    """The step that shards (SURVEY §8e, north_star): ONE pose-only global-BA window whose voxel factor is sharded over the ranks by the reference
    hash of the root cell; a step = one LM iteration = sharded Hessian build -> NCCL all-reduce of [C | g | D | r] -> replicated LDLT -> sharded
    residual -> scalar all-reduce.  STRONG scaling: the same window for every N.  Own ctx, so the local-BA legs above stay unsharded."""
    import torch
    W, pts, L, K = args.gba_win, args.gba_win_pts, args.gba_L, args.gba_steps
    ctx = vx.Context(local)
    if world > 1:
        uid = [vx.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
    tr, est, p, off = scene_points(vx, W, pts, L, seed=1)
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    f = vx.Factor(ctx, W)
    t0 = time.time()
    ctx.build_window_factor(mp, p, off, est, f)          # every rank keeps the octrees whose root cell it owns
    t_vox = time.time() - t0
    del p
    V, E, _ = f.counts()
    f.cache_save()

    def step():
        f.cache_restore()
        return ctx.lidar_ba(f, est, max_iter=1, thd_num=1, want_hess=False)

    o = None
    for _ in range(3):
        o = step()
    barrier(dist, local)
    ctx.timer_start(); t0 = time.perf_counter()
    for _ in range(K):
        step()
    ms = max(ctx.timer_stop(), (time.perf_counter() - t0) * 1e3)
    ms = barrier_max(dist, local, ms)
    ctx.timing(True); ctx.timing_reset()
    for _ in range(3):
        step()
    stages = ctx.timing_read(); ctx.timing(False)
    mine = [float(V), float(E)] + [stages.get(k, (0.0, 0))[0] / 3 for k in ("k_syrk", "k_jac", "k_pairs", "k_cluster_sum", "nccl_allreduce", "k_ldlt_all")]
    per_rank = [mine]
    if dist is not None:
        g = [torch.zeros(len(mine), dtype=torch.float64, device=f"cuda:{local}") for _ in range(world)]
        dist.all_gather(g, torch.tensor(mine, dtype=torch.float64, device=f"cuda:{local}"))
        per_rank = [x.cpu().tolist() for x in g]
    res = {"metric": "global-BA LM iterations/sec, one voxel-sharded pose-only BA (strong scaling)", "value": K / (ms * 1e-3), "unit": "iterations/s", "ms_per_step": ms / K, "steps": K,
           "scaling": "strong", "n_gpus": world, "workload": f"W={W} keyframes x {pts} pts, L={L} m -> {int(sum(r[0] for r in per_rank))} plane voxels, {int(sum(r[1] for r in per_rank))} clusters; n=6W={6 * W}",
           "allreduce_bytes_per_step": 8 * ((6 * W) ** 2 + 30 * W + 2), "allreduce_ms": max(r[6] for r in per_rank), "map_build_ms_rank0": t_vox * 1e3,
           "per_rank_[V,E,syrk,jac,pairs,cluster_sum,nccl,ldlt]_ms": [[round(x, 3) for x in r] for r in per_rank],
           "comm": "NCCL all-reduce issued by libvxs on its own communicator (vxs_ctx_comm_init)" if world > 1 else "single GPU: no collective",
           "check": {"trace": [[float(t["r1"]), float(t["r2"]), int(t["accepted"])] for t in o["trace"]]}}
    f.close(); ctx.close()
    return res


def ncu_traffic(kernels):
    """DRAM bytes per launch (read + write) of the named kernels from the committed `ncu --set full` summary of this same command
    (profiles/r02_ncu_full_ba_kernels.txt); None when the summary is absent."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_ncu_full_ba_kernels.txt")
    try:
        txt = open(path).read()
    except OSError:
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    total, seen = 0.0, set()
    for blk in txt.split("== ")[1:]:
        name = blk.split()[0]
        if name not in kernels or name in seen:
            continue
        seen.add(name)
        for line in blk.splitlines():
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                total += float(f[1]) * unit.get(f[2], 1.0)
    return total if len(seen) == len(set(kernels)) else None


def ds_leg(ctx):
    """SURVEY.md §8f rows 2/4: down_sampling_voxel (tools.hpp:201) of 4 M float points at 0.25 m through the host-buffer C-ABI call."""
    n = 4_000_000
    pts = np.random.default_rng(3).uniform(-100.0, 100.0, (n, 3)).astype(np.float32)
    ctx.down_sampling(pts, 0.25)
    ctx.timing(True); ctx.timing_reset()
    t0 = time.perf_counter()
    g = ctx.down_sampling(pts, 0.25)
    wall = (time.perf_counter() - t0) * 1e3
    st = ctx.timing_read(); ctx.timing(False)
    kms = sum(v[0] for v in st.values())
    return {"points": n, "cells": int(len(g["index"])), "ms_call_pageable_host_buffers": wall, "ms_kernels": kms, "gpoints_per_s_kernels": n / max(kms, 1e-9) / 1e6,
            "algorithmic_bytes": n * 12, "stages_ms": {k: v[0] for k, v in st.items() if v[1] > 0}}


def c2_leg(vx, ctx, hbm):
    """BASELINE.json configs[1]: per-voxel covariance + 3x3 eigensolve over 1 M points / ~100 k voxels (L=183, max_layer 0):
    the GPU voxel-map build on device-resident-after-upload points; kernel times from CUDA events."""
    L, n = 183.0, 1000000
    pose = synth.true_pose(L, 0)
    pts = synth.gen_scan(L, 0, n, pose, seed=0x5EED0000 + 2000)
    off = np.array([0, n], dtype=np.int64)
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=0)
    f = vx.Factor(ctx, 1)
    ctx.build_window_factor(mp, pts, off, pose[None, :], f)          # warm-up (allocations)
    ctx.timing(True); ctx.timing_reset()
    reps = 5
    for _ in range(reps):
        nv = ctx.build_window_factor(mp, pts, off, pose[None, :], f)
    st = ctx.timing_read(); ctx.timing(False)
    ms = {k: v[0] / reps for k, v in st.items() if v[1] > 0}
    t_all = sum(ms.values())
    t_acc = ms.get("k_rec_clusters", 0.0) + ms.get("k_point_keys", 0.0) + ms.get("k_bbox", 0.0)
    f.close()
    return {"workload": f"C2: {n} pts, L={L}, max_layer=0 -> {nv} plane voxels", "kernel_ms_total": t_all, "points_per_s": n / (t_all * 1e-3), "voxels": int(nv),
            "kernels_ms": ms, "hbm_frac_transform_accumulate": (24.0 * n * 3 / (t_acc * 1e-3) / 1e9 / hbm) if t_acc > 0 else None,
            "note": "kernel time only (CUDA events); the H2D copy of the 24 MB scan is outside. transform+accumulate reads each 24-B point three times (bbox, keys, clusters)"}


def oracle_factor_from_csr(W, ptr, fr, cl, eig, s):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as oa
    V = ptr.shape[0] - 1
    dense = np.zeros((V, W, 10))
    vox = np.repeat(np.arange(V), np.diff(ptr))
    dense[vox, fr] = cl
    return oa.OracleFactor.from_dense(W, dense, None, None, eig, s)


def cpu_baseline_from_structure(vx, W, ptr, fr, cl, eig, s, st0, tr, reps=2):
    """The oracle (CPU restatement of the reference, reference thread structure: 5 threads) on the SAME factor, timed on this host."""
    of = oracle_factor_from_csr(W, ptr, fr, cl, eig, s)
    imu = synth.ImuWindow(tr)
    ts, first = [], None
    for _ in range(reps):
        imu.reset()
        t0 = time.perf_counter()
        o = of.li_ba(st0, imu, with_gravity=False, max_iter=1)
        ts.append((time.perf_counter() - t0) / max(len(o["trace"]), 1))       # seconds per LM iteration actually executed
        if first is None:
            first = {"r1": float(o["trace"][0]["r1"]), "r2": float(o["trace"][0]["r2"]), "accepted": int(o["trace"][0]["accepted"]), "states": o["states"], "st0": np.array(st0)}
    t = min(ts)
    try:
        n = 15 * W
        import oracle_api as oa
        A = np.eye(n) * 2 + 0.01 * np.ones((n, n)); t0 = time.perf_counter(); oa.ldlt_solve(A, np.ones(n)); t_fix = time.perf_counter() - t0
        allc = all_cores_variant(of, st0[:, :12], t_fix)
    except Exception as e:
        allc = {"error": str(e)}
    out = {"value": 1.0 / t, "unit": UNIT, "cores": 5, "kind": "port", "host_cores": os.cpu_count(),
           "sample": f"{reps} full-size LM iterations (all {ptr.shape[0] - 1} voxels) of the oracle LI_BA_Optimizer, best of {reps}; 5 threads as voxel_map.hpp:467,531 hard-code",
           "all_cores_variant": allc, "first_iteration": first}
    # the reference's OWN code on the same factor when oracle/_ref travelled with the repo (its damping_iter has no max_iter: one call = 3 iterations unless it
    # exits early; the count comes from the port's identical trace).  Reported beside the port — never instead of a number that was measured.
    try:
        import ref_api as ra
        if ra.available():
            V = ptr.shape[0] - 1
            dense = np.zeros((V, W, 10))
            dense[np.repeat(np.arange(V), np.diff(ptr)), fr] = cl
            imu_c = synth.ImuWindow(tr); imu_c.reset()
            iters = max(len(oracle_factor_from_csr(W, ptr, fr, cl, eig, s).li_ba(st0, imu_c, with_gravity=False, max_iter=3)["trace"]), 1)
            rimu = ra.RefImuWindow(tr)
            tr_ = []
            for _ in range(2):
                rf = ra.OracleFactor.from_dense(W, dense, None, None, eig, s)       # fresh factor: a solve overwrites the cached eig / pcr_adds
                rimu.reset()
                t0 = time.perf_counter(); rf.li_ba(st0, rimu, with_gravity=False, max_iter=3); tr_.append((time.perf_counter() - t0) / iters)
                del rf
            out["reference_sources"] = {"value": 1.0 / min(tr_), "unit": UNIT, "cores": 5, "kind": "reference", "iterations_per_call": iters,
                                        "sample": "the reference's LI_BA_Optimizer::damping_iter (voxel_map.hpp compiled unmodified against the stand-in Eigen: scalar loops, no SSE packet "
                                                  "math; real IMU_PRE objects) on the same factor, best of 2 calls, call time / iterations executed"}
        else:
            out["reference_sources"] = {"unavailable": "oracle/_ref/libvxref.so was not built (it needs the original project's sources at build time)"}
    except Exception as e:          # noqa: BLE001 — the extra figure must never cost the bench line
        out["reference_sources"] = {"error": repr(e)}
    return out


def all_cores_variant(of, poses12, t_fix, scale=1.0):
    """NOT the reference's structure (it hard-codes 5 threads, voxel_map.hpp:467,531): the oracle's Hessian and residual passes with one
    thread per host core (capped at 64), plus the serial dense LDLT — reported beside the faithful number so that the GPU/CPU ratio can
    also be read against a CPU that uses the whole box.  `scale` rescales the voxel-proportional part when `of` holds a voxel sample."""
    T = int(max(1, min(os.cpu_count() or 1, 64)))
    th = min(of.time_hessian(poses12, T, reps=1)[0] for _ in range(2))
    trs = min(of.time_residual(poses12, T, reps=1)[0] for _ in range(2))
    t = (th + trs) * scale + t_fix
    return {"value": 1.0 / t, "unit": UNIT, "cores": T, "note": "oracle Hessian + residual passes with one thread per core (max 64) + serial LDLT; not the reference's 5-thread structure, "
            "IMU factors excluded", "hessian_ms": th * scale * 1e3, "residual_ms": trs * scale * 1e3, "ldlt_ms": t_fix * 1e3}


# ---------------------------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank, world, local, dist = dist_setup(args)
    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return
    import __graft_entry__ as ge
    ge.build_checker(quiet=True)          # CPU libraries only: this process never loads libvxs.so
    import voxel_slam_b200 as vx          # ctypes struct definitions (MapParams); the CUDA library is loaded lazily and not here
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_api as oa
    W, L, K, Wu = args.win, args.L, args.steps, args.warmup
    pts_map = min(args.pts_per_scan, 200000)   # LM cost depends on voxels x frames, not on points per scan: build the map from a bounded cloud
    tr, est, p, off = scene_points(vx, W, pts_map, L, seed=1)
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    t0 = time.time()
    of = oa.build_window_factor(mp, p, off, est, threads=5)
    t_map = time.time() - t0
    V = of.size()
    log(f"[reference] oracle map build from {W}x{pts_map} points: {t_map:.1f}s, V={V}")
    st0 = states_from(est)
    ex = of.export()
    cl, eig, s = ex["clusters10"], ex["eig12"], ex["sum10"]
    # probe one iteration of the port, then bound the sample so the whole run stays within a few minutes
    imu0 = synth.ImuWindow(tr)
    t0 = time.perf_counter(); imu0.reset(); of.li_ba(st0, imu0, max_iter=1); t_full = time.perf_counter() - t0
    budget = 150.0
    # The thing timed: the reference's OWN sources (oracle/_ref/libvxref.so: voxel_map.hpp / tools.hpp / preintegration.hpp compiled unmodified
    # against stand-ins for the Eigen / PCL / ROS headers this image lacks) when that library travelled with the repo, else the hand-written port.
    # The reference's LI_BA_Optimizer::damping_iter has no max_iter: one call = 3 LM iterations (voxel_map.hpp:581) unless it exits early.
    kind, api = "port", oa
    try:
        import ref_api as ra
        if ra.available():
            kind, api = "reference", ra
    except Exception as e:
        log(f"[reference] oracle/_ref not usable ({e!r}); timing the port")
    calls = K + Wu
    phi = min(1.0, budget / (calls * t_full * (3 if kind == "reference" else 1)))
    keep = V if phi >= 1.0 else max(64, int(V * phi))
    sel = np.arange(V) if keep == V else np.linspace(0, V - 1, keep).astype(np.int64)
    phi = keep / V
    mk = lambda a: a.OracleFactor.from_dense(W, cl[sel], None, None, eig[sel], s[sel])
    fsub = mk(api)
    imu = ra.RefImuWindow(tr) if kind == "reference" else synth.ImuWindow(tr)
    # iterations one call executes, counted on the port (its LM trace is identical; the reference build exposes no trace)
    imu_c = synth.ImuWindow(tr); imu_c.reset()
    iters_per_call = max(len(mk(oa).li_ba(st0, imu_c, max_iter=3 if kind == "reference" else 1)["trace"]), 1)
    # fixed (voxel-independent) part of an iteration: the dense LDLT of the 15W system
    n = 15 * W
    A = np.eye(n) * 2 + 0.01 * np.ones((n, n)); t0 = time.perf_counter(); api.ldlt_solve(A, np.ones(n)); t_fix = time.perf_counter() - t0

    def step():
        imu.reset()
        t0 = time.perf_counter()
        fsub.li_ba(st0, imu, max_iter=1)
        return (time.perf_counter() - t0) / iters_per_call          # seconds per LM iteration

    for _ in range(Wu):
        step()
    t_steps = [step() for _ in range(K)]
    t_step = float(np.mean(t_steps))
    t_iter_full = (max(t_step - t_fix, 0.0)) / phi + t_fix      # voxel-proportional part scaled back to the full window
    value = 1.0 / t_iter_full
    what = ("the reference's own LI_BA_Optimizer::damping_iter (voxel_map.hpp compiled unmodified; Eigen stand-in = plain scalar loops, no SSE packet math; real IMU_PRE objects)"
            if kind == "reference" else "the oracle port of LI_BA_Optimizer")
    sample = (f"window geometry of the metric shape (W={W}, L={L}, V={V} voxels) built from {pts_map} pts/scan (LM cost depends on voxels x frames, not on points per scan); each step = one "
              f"call of {what} = {iters_per_call} LM iteration(s), its time divided by that count; 5 threads as voxel_map.hpp:467,531 hard-code; {phi:.3f} of the voxels, voxel-proportional "
              f"time scaled to the full window (LDLT {t_fix * 1e3:.0f} ms per iteration not scaled)")
    try:
        allc = all_cores_variant(mk(oa), st0[:, :12], t_fix, 1.0 / phi)
    except Exception as e:   # never let the extra leg break the arm
        allc = {"error": str(e)}
    port = None
    if kind == "reference":   # the hand-written restatement (oracle/vxo_*.hpp) on the same sample, for comparison with the reference's own code above
        try:
            fp, imu_p, tp = mk(oa), synth.ImuWindow(tr), []
            for _ in range(2):
                imu_p.reset(); t0 = time.perf_counter(); op = fp.li_ba(st0, imu_p, max_iter=1); tp.append((time.perf_counter() - t0) / max(len(op["trace"]), 1))
                fp = mk(oa)
            port = {"value": 1.0 / ((max(min(tp) - t_fix, 0.0)) / phi + t_fix), "unit": UNIT, "cores": 5, "kind": "port"}
        except Exception as e:
            port = {"error": str(e)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu, "ms_per_step": t_iter_full * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic (same seeded scene as the GPU arm)",
            "config": {"workload": f"metric shape M: W={W} window, L={L} m room, V={V} plane voxels; n=15W={n} LI-BA system", "parallelism": "CPU, 5 threads (reference thread structure)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 5, "kind": kind, "host_cores": os.cpu_count(), "sample": sample, "iterations_per_call": iters_per_call,
                             "all_cores_variant": allc, "hand_written_port": port},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------- global-BA workload
def run_gba(args):
    """Secondary workload (not the driver's default): one pass of the top-level hierarchical global BA (voxelslam.cpp:2374-2384:
    rebuild the GBA voxel map at the current poses, recut, Lidar_BA_Optimizer::damping_iter(up=4)) over K keyframes of a synthetic
    city-grid scene, voxel-sharded over the N GPUs with the NCCL all-reduce of the pose Hessian.  STRONG scaling: total work fixed."""
    import torch
    import voxel_slam_b200 as vx
    rank, world, local, dist = dist_setup(args)
    K, n, per_row = args.gba_keyframes, args.gba_pts, args.gba_per_row
    ctx = vx.Context(local)
    if world > 1:
        uid = [vx.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
    t0 = time.time()
    tr = np.stack([synth.lawnmower_pose(i, per_row) for i in range(K)])
    est = np.stack([tr[0]] + [synth.perturb_pose(tr[i], 100 + i, 1e-3, 1e-2) for i in range(1, K)])
    xyz = np.empty((K * n, 3), dtype=np.float32)
    for i in range(K):
        synth.gen_scan_city(i, n, tr[i], out=xyz[i * n:(i + 1) * n])
    off = np.arange(K + 1, dtype=np.int64) * n
    mp = vx.MapParams.make(voxel_size=args.gba_voxel, min_eigen_value=0.1 if args.gba_voxel >= 2 else 0.0025, max_layer=2)
    f = vx.Factor(ctx, K)
    log(f"[rank {rank}] GBA scene: {K} keyframes x {n} pts generated in {time.time() - t0:.1f}s")

    def step():
        ctx.build_gba_factor(mp, xyz, off, est, f)
        return ctx.lidar_ba(f, est, max_iter=4, thd_num=1, want_hess=False)

    o = step()
    V, E, _ = f.counts()
    for _ in range(max(args.warmup, 1)):
        step()
    barrier(dist, local)
    ctx.timer_start(); t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps):
        iters += len(step()["trace"])
    ms = max(ctx.timer_stop(), (time.perf_counter() - t0) * 1e3)
    ms = barrier_max(dist, local, ms)
    ctx.timing(True); ctx.timing_reset()
    step()
    stages = ctx.timing_read(); ctx.timing(False)
    tot = np.array([float(V), float(E)])
    if dist is not None:
        t = torch.tensor(tot, device=f"cuda:{local}"); dist.all_reduce(t); tot = t.cpu().numpy()
    if rank == 0:
        line = {"metric": "hierarchical global-BA passes/sec (top level, voxel-sharded)", "value": args.steps / (ms * 1e-3), "unit": "passes/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 1), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic city grid",
                "config": {"workload": f"{K} keyframes x {n} pts, voxel {args.gba_voxel} m, max_layer 2 -> {int(tot[0])} plane voxels, {int(tot[1])} clusters (k={tot[1] / max(tot[0], 1):.1f}); n=6K={6 * K}",
                           "step": "build GBA map (sharded by root-cell hash) + recut + Lidar_BA damping_iter(up=4) with NCCL all-reduce of [C|g|D|r]", "lm_iterations_per_pass": iters / args.steps},
                "rank0_stage_ms": {k: v[0] for k, v in sorted(stages.items(), key=lambda kv: -kv[1][0]) if v[1] > 0},
                "check": {"pose_err_before": float(np.abs(est - tr).max()), "pose_err_after_1_pass": float(np.abs(o["poses"] - tr).max())}}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


def run_gba_window(args):
    """Secondary workload: ONE large pose-only BA (Lidar_BA_Optimizer, n = 6W) whose voxel factor is sharded over the N GPUs by the
    reference hash of the root cell — the shape of a top-level HBA problem with dense co-visibility (SURVEY §8e (2)).  A step is one LM
    iteration: sharded Hessian build -> NCCL all-reduce of [C|g|D|r] -> replicated LDLT -> sharded residual -> scalar all-reduce.
    STRONG scaling: the window is the same for every N."""
    import torch
    import voxel_slam_b200 as vx
    rank, world, local, dist = dist_setup(args)
    W, pts, L, K, Wu = args.win, args.pts_per_scan, args.L, args.steps, args.warmup
    ctx = vx.Context(local)
    if world > 1:
        uid = [vx.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)
    tr, est, p, off = scene_points(vx, W, pts, L, seed=1)
    mp = vx.MapParams.make(voxel_size=1.0, min_eigen_value=0.0025, max_layer=2)
    f = vx.Factor(ctx, W)
    t0 = time.time()
    ctx.build_window_factor(mp, p, off, est, f)
    t_vox = time.time() - t0
    del p
    V, E, _ = f.counts()
    f.cache_save()

    def step():
        f.cache_restore()
        return ctx.lidar_ba(f, est, max_iter=1, thd_num=1, want_hess=False)

    o = None
    for _ in range(max(Wu, 3)):
        o = step()
    barrier(dist, local)
    ctx.timer_start(); t0 = time.perf_counter()
    for _ in range(K):
        step()
    ms = max(ctx.timer_stop(), (time.perf_counter() - t0) * 1e3)
    ms = barrier_max(dist, local, ms)
    ctx.timing(True); ctx.timing_reset()
    for _ in range(3):
        step()
    stages = ctx.timing_read(); ctx.timing(False)
    tot = np.array([float(V), float(E)])
    mine = [float(V), float(E)] + [stages.get(k, (0.0, 0))[0] / 3 for k in ("k_syrk", "k_jac", "k_cluster_sum", "nccl_allreduce", "k_ldlt_all")]
    per_rank = [mine]
    if dist is not None:
        t = torch.tensor(tot, device=f"cuda:{local}"); dist.all_reduce(t); tot = t.cpu().numpy()
        g = [torch.zeros(len(mine), dtype=torch.float64, device=f"cuda:{local}") for _ in range(world)]
        dist.all_gather(g, torch.tensor(mine, dtype=torch.float64, device=f"cuda:{local}"))
        per_rank = [x.cpu().tolist() for x in g]
    if rank == 0:
        line = {"metric": "global-BA LM iterations/sec (one voxel-sharded pose-only BA)", "value": K / (ms * 1e-3), "unit": "iterations/s", "n_gpus": world, "steps": K,
                "warmup": max(Wu, 3), "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic (seeded 3-plane room)",
                "config": {"workload": f"W={W} keyframes x {pts} pts, L={L} m -> {int(tot[0])} plane voxels, {int(tot[1])} clusters over all ranks; n=6W={6 * W}",
                           "step": "one LM iteration = vxs_lidar_ba(max_iter=1): sharded Hessian, NCCL all-reduce of (6W)^2+30W+1 doubles, replicated LDLT, sharded residual, scalar all-reduce",
                           "allreduce_bytes_per_step": 8 * ((6 * W) ** 2 + 30 * W + 2)},
                "rank0_stage_ms_per_step": {k: v[0] / 3 for k, v in sorted(stages.items(), key=lambda kv: -kv[1][0]) if v[1] > 0},
                "map_build_ms_rank0": t_vox * 1e3,
                "per_rank_[V,E,syrk,jac,cluster_sum,nccl,ldlt]_ms": [[round(x, 3) for x in r] for r in per_rank],
                "check": {"trace": [[float(t["r1"]), float(t["r2"]), int(t["accepted"])] for t in o["trace"]]}}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--win", type=int, default=50)
    ap.add_argument("--pts-per-scan", type=int, default=1000000)
    ap.add_argument("--L", type=float, default=130.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="local_ba", choices=["local_ba", "gba", "gba_window", "hba"])
    ap.add_argument("--no-local-mapping", action="store_true")
    ap.add_argument("--lm-steps", type=int, default=6)
    ap.add_argument("--no-gba", action="store_true")
    ap.add_argument("--hba-keyframes", type=int, default=2000)
    ap.add_argument("--hba-pts", type=int, default=100000)
    ap.add_argument("--hba-per-row", type=int, default=50)
    ap.add_argument("--hba-range", type=float, default=35.0)
    ap.add_argument("--hba-steps", type=int, default=5)
    ap.add_argument("--gba-window-leg", action="store_true")
    ap.add_argument("--gba-win", type=int, default=100)
    ap.add_argument("--gba-win-pts", type=int, default=200000)
    ap.add_argument("--gba-L", type=float, default=260.0)
    ap.add_argument("--gba-steps", type=int, default=10)
    ap.add_argument("--gba-keyframes", type=int, default=400)
    ap.add_argument("--gba-pts", type=int, default=50000)
    ap.add_argument("--gba-per-row", type=int, default=20)
    ap.add_argument("--gba-voxel", type=float, default=1.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (default local-BA workload of --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "local_ba" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the default local_ba workload of --impl ours")
    if args.workload == "hba":     # the hierarchical global-BA leg alone (same JSON block as the `gba` key of the default run)
        import voxel_slam_b200 as vx
        rank, world, local, dist = dist_setup(args)
        res = hba_leg(vx, local, rank, world, dist, args)
        if rank == 0:
            print(json.dumps(res), flush=True)
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return
    if args.workload == "gba":
        return run_gba(args)
    if args.workload == "gba_window":
        return run_gba_window(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
