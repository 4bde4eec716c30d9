#!/usr/bin/env python
"""bench.py -- CPD EM-iterations/sec at N = M = 100k 3-D points on N B200s (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--points 100000] [--dump-outputs DIR]
  N > 1 is launched by torchrun (one rank per GPU); rank 0 prints ONE JSON line.

A "step" is one EM iteration (probreg/cpd.py:111-113: transform -> E-step -> M-step) of rigid CPD
on the synthetic workload of BASELINE.md section 3 (anisotropic box, 30 degree rotation, 0.01 noise),
w = 0, sigma2 auto-initialised, update_scale=True.  Strong scaling: the cloud is fixed and the
targets are sharded over the ranks (one 32-double NCCL all-reduce per iteration).

  value   : iterations/s with both clouds resident in HBM; K iterations timed back to back with a
            CUDA-event pair per iteration on the library's stream, L2 flushed (256 MiB memset)
            between iterations outside the event pairs; max over ranks.
  e2e     : the same metric through the public API with HOST buffers: each step is one
            RigidCPD.registration(target, maxiter=1) -- H2D of both clouds from pinned memory, sigma2
            init, one EM iteration, D2H of the MstepResult -- timed with the host clock around it.
  roofline: the fused E-step (pass 1 + pass 2 kernels) against the FP32 issue roofline it is bound
            by, plus the HBM view (the kernel moves ~10 MB per iteration: P is never materialised).
  cpu_baseline / --impl reference: the oracle port of the reference's numpy path (oracle/cpd_oracle.py)
            on the host cores, on a bounded column sample of the same workload, extrapolated.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "cpd_em_iterations_per_sec"
UNIT = "it/s"
FLOP_PER_PAIR_ITER = 29.0     # SURVEY 8(d): pass 1 = 3D+2 = 11, pass 2 = 5D+3 = 18 at D = 3


def hbm_bytes_per_iter(n_local, m):
    # SURVEY 8(d): algorithmic traffic of the fused E-step, per iteration and rank:
    # pass 1 reads 16 B/target + 16 B/source, writes 8 B/target; pass 2 reads 32 B/target + 16 B/source
    # and writes 32 B/source (p1, px in FP64).
    return 16 * n_local + 16 * m + 8 * n_local + 32 * n_local + 16 * m + 32 * m


class ClockSampler(object):
    """SM clocks / clock-event reasons while the job runs (B200_PROFILING.md recipe).  ONE poller (rank 0) for all the job's GPUs,
    started before the warm-up.  NVML through pynvml, polled every 5 ms from a thread (a query costs microseconds, so even a
    140 ms timed region gets ~25 samples per GPU, and every sample has a timestamp: the median reported is over the samples that
    fall INTO the timed region); `nvidia-smi -lms 100` as the fallback when NVML cannot be loaded -- its samples are ~10x sparser
    and carry a utilisation averaged over the driver's own window, so there the samples since the warm-up count."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, n_gpus):
        self.n_gpus = n_gpus
        self.rows = []            # (time, gpu, sm MHz, power W, set of reason names)
        self.smax = []
        self.proc = None
        self.nvml = None
        self.stop_flag = False
        self.source = None

    def _physical(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return [int(x) for x in vis.split(",")][: self.n_gpus]
            except ValueError:
                pass
        return list(range(self.n_gpus))

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handles = [pynvml.nvmlDeviceGetHandleByIndex(i) for i in self._physical()]
            self.smax = [float(pynvml.nvmlDeviceGetMaxClockInfo(hd, pynvml.NVML_CLOCK_SM)) for hd in self.handles]
            self.nvml = pynvml
            self.source = "nvml, 5 ms"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi -lms 100"
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nvml
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]
        while not self.stop_flag:
            for g, hd in enumerate(self.handles):
                try:
                    sm = float(nv.nvmlDeviceGetClockInfo(hd, nv.NVML_CLOCK_SM))
                    mask = int(get_reasons(hd))
                    try:
                        pw = nv.nvmlDeviceGetPowerUsage(hd) / 1000.0
                    except Exception:
                        pw = None
                    self.rows.append((time.perf_counter(), g, sm, pw, {nm for b, nm in bits if mask & b}))
                except Exception:
                    pass
            time.sleep(0.005 if len(self.handles) <= 2 else 0.01)

    def _read_smi(self):
        phys = self._physical()
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 8:
                continue
            try:
                idx = int(f[0])
                if idx not in phys:
                    continue
                sm, mx = float(f[1]), float(f[2])
                try:
                    pw = float(f[3])
                except ValueError:
                    pw = None
            except ValueError:
                continue
            if mx not in self.smax:
                self.smax.append(mx)
            self.rows.append((time.perf_counter(), phys.index(idx), sm, pw,
                              {nm for nm, v in zip(self.NAMES, f[4:8]) if v.lower().startswith("active")}))

    def count(self):
        return len(self.rows)

    def stop(self, t0=None, t1=None, t_load=None):
        """t0 .. t1: the timed region; t_load: since when the GPUs have been under this job's load (end of the first warm-up)."""
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["neither NVML nor nvidia-smi available"]}
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        else:
            self.thread.join(timeout=1.0)
            try:
                self.nvml.nvmlShutdown()
            except Exception:
                pass
        rows = list(self.rows)
        slack = 0.0 if self.nvml is not None else 0.11
        timed = [r for r in rows if t0 is not None and t0 <= r[0] <= t1 + slack]
        loaded = [r for r in rows if t_load is None or t_load <= r[0] <= (t1 if t1 is not None else r[0]) + slack]
        use = timed if timed else loaded
        sm = [r[2] for r in use]
        power = [r[3] for r in use if r[3] is not None]
        reasons = set()
        for r in use:
            reasons |= r[4]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(self.smax) if self.smax else None,
                "power_w_max": max(power) if power else None, "samples_under_load": len(loaded),
                "samples_in_timed_region": len(timed), "median_over": "timed region" if timed else "since the warm-up",
                "source": self.source, "reasons": sorted(reasons)}


def workload(points, kind="rigid"):
    from probreg_b200.synthetic import synthetic_pair
    if kind == "nonrigid":                      # SURVEY 8(d) config 5: the rigid generator's source + a smooth displacement
        src, _ = synthetic_pair(points, "rigid")
        f = np.array([[1.0, 0.5, 0.0], [0.0, 1.0, 0.7], [0.3, 0.0, 1.0]])
        tgt = src + 0.03 * np.sin(2 * np.pi * src.dot(f)) + 0.002 * np.random.default_rng(9).standard_normal(src.shape)
        return src, np.ascontiguousarray(tgt)
    return synthetic_pair(points, kind)


# ---------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference (baseline/_ref/probreg, see baseline/install_ref.py) on a bounded sample;
# the oracle port beside it as a second figure
# ---------------------------------------------------------------------------------------------
WORKLOADS = {
    2: ("rigid", 100000, "rigid CPD, synthetic 3-D N=M=%d, sigma2 auto, w=0, update_scale"),
    3: ("affine", 250000, "affine CPD, synthetic 3-D N=M=%d, sigma2 auto, w=0"),
    4: ("rigid", 1000000, "rigid CPD, synthetic 3-D N=M=%d, sigma2 auto, w=0, update_scale"),
    5: ("nonrigid", 50000, "non-rigid CPD (low-rank G, K=200, beta=2, lmd=2), synthetic 3-D N=M=%d, sigma2 auto, w=0"),
}


def workload_string(config, points):
    return WORKLOADS[config][2] % points


def blas_threads():
    try:
        import threadpoolctl
        return int(max([p.get("num_threads", 1) for p in threadpoolctl.threadpool_info()] + [1]))
    except Exception:
        return int(os.cpu_count() or 1)


def reference_sample(kind, points, cols, chunk=250):
    """One EM iteration of the reference's own code (probreg/cpd.py:111-113) on `cols` of the `points` target columns:
    Transformation.transform on all sources, CoherentPointDrift.expectation_step (cpd.py:71-88) column-chunked -- exact for
    w = 0 because `den` is per column (SURVEY 8d) -- and the class's _maximization_step (cpd.py:160-192 / 219-244) on the sampled
    columns' EstepResult.  The E-step time is extrapolated to all columns; the M-step and the transform are not (they cost
    O(M + N), < 0.1 % of the iteration)."""
    from baseline import ref_loader
    rcpd, rtf = ref_loader.load()
    from probreg_b200.synthetic import synthetic_pair
    src, tgt = synthetic_pair(points, "affine" if kind == "affine" else "rigid")
    cols = min(cols, points)
    sub = tgt[:cols]
    # sigma2_0 in closed form (the reference's _initialize would allocate an M x N float32 matrix: 40 GB at 100k)
    s2 = float(((src * src).sum() / points + (tgt * tgt).sum() / points - 2.0 * src.mean(0).dot(tgt.mean(0))) / 3.0)
    reg = rcpd.AffineCPD(src) if kind == "affine" else rcpd.RigidCPD(src, update_scale=True)
    tfm = rtf.AffineTransformation(np.identity(3), np.zeros(3)) if kind == "affine" else rtf.RigidTransformation(np.identity(3), np.zeros(3))
    # one untimed chunk first: the first M x chunk float64 temporaries of a process are page-faulted in (seconds in this
    # image's sandbox), after which the allocator re-uses them -- the reference's steady state is what is timed
    reg.expectation_step(src, sub[:chunk], s2, 0.0)
    t0 = time.perf_counter()
    ts = tfm.transform(src)
    t_tf = time.perf_counter() - t0
    t0 = time.perf_counter()
    pt1, p1, px = [], np.zeros(points), np.zeros((points, 3))
    for lo in range(0, cols, chunk):
        es = reg.expectation_step(ts, sub[lo:lo + chunk], s2, 0.0)
        pt1.append(es.pt1); p1 += es.p1; px += es.px
    t_e = time.perf_counter() - t0
    es = rcpd.EstepResult(np.concatenate(pt1), p1, px, float(p1.sum()))
    t0 = time.perf_counter()
    res = reg.maximization_step(sub, es, s2)
    t_m = time.perf_counter() - t0
    t_iter = t_e * (points / float(cols)) + t_m + t_tf
    return {"value": 1.0 / t_iter, "unit": UNIT, "cores": blas_threads(), "host_cpus": os.cpu_count(), "kind": "reference",
            "sample": "unmodified probreg/cpd.py (baseline/_ref): expectation_step on %d of %d target columns x all %d sources in "
                      "chunks of %d (%.2f s, extrapolated x%.0f) + transform (%.3f s) + _maximization_step on the sampled "
                      "columns (%.3f s); numpy/scipy as the reference uses them (~90%% single-threaded, BLAS threads = %d)"
                      % (cols, points, points, chunk, t_e, points / float(cols), t_tf, t_m, blas_threads()),
            "sec_per_iter_extrapolated": t_iter, "ns_per_pair": t_e / (cols * float(points)) * 1e9,
            "sigma2_after": float(res.sigma2)}


def port_sample(points, cols):
    """The same iteration through the oracle port (oracle/cpd_oracle.py): a second CPU figure (about 3x faster than the reference)."""
    from oracle import cpd_oracle as orc
    src, tgt = workload(points)
    s2 = float(orc.sigma2_init_exact(src, tgt))
    cols = min(cols, points)
    sub = tgt[:cols]
    chunk = 250
    orc.expectation_step(src, tgt[:chunk], s2, 0.0, n_global=points)          # untimed: see reference_sample
    t0 = time.perf_counter()
    ts = orc.apply_rigid(src, np.identity(3), np.zeros(3))
    parts = [orc.expectation_step(ts, sub[lo:lo + chunk], s2, 0.0, n_global=points) for lo in range(0, cols, chunk)]
    es = orc.Estep(np.concatenate([e.pt1 for e in parts]), sum(e.p1 for e in parts), sum(e.px for e in parts),
                   float(sum(e.p1.sum() for e in parts)))
    t_e = time.perf_counter() - t0
    t0 = time.perf_counter()
    orc.mstep_rigid(src, tgt[:cols], es)
    t_m = time.perf_counter() - t0
    t_iter = t_e * (points / float(cols)) + t_m
    return {"value": 1.0 / t_iter, "unit": UNIT, "kind": "port", "sec_per_iter_extrapolated": t_iter,
            "ns_per_pair": t_e / (cols * float(points)) * 1e9,
            "sample": "oracle port, E-step on %d of %d columns (%.2f s) extrapolated + M-step on the sample (%.3f s)" % (cols, points, t_e, t_m)}


def cpu_sample(kind, points, cols):
    """cpu_baseline of the bench line: the reference when baseline/_ref travelled with the repo, else the oracle port."""
    from baseline import ref_loader
    if ref_loader.available() and kind in ("rigid", "affine"):
        out = reference_sample(kind, points, cols)
        if kind == "rigid":
            try:
                out["port"] = port_sample(points, cols)
            except Exception as e:          # noqa: BLE001
                out["port"] = {"error": str(e)[:200]}
        return out
    out = port_sample(points, cols)
    out["cores"], out["host_cpus"] = blas_threads(), os.cpu_count()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, points = args.kind, args.points
    if kind == "nonrigid":
        emit({"impl": "reference", "unavailable": "the reference has no low-rank non-rigid path (dense M x M solve: 30 GB and 1e14 flop per "
                                                  "iteration at 50k); config 5 has no CPU arm"})
        return
    cols = args.cpu_cols
    vals, last = [], None
    for _ in range(args.steps):
        last = cpu_sample(kind, points, cols)
        vals.append(last["sec_per_iter_extrapolated"])
    t = float(np.mean(vals))
    last["value"] = 1.0 / t
    out = {"impl": "reference", "metric": METRIC, "value": 1.0 / t, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_string(args.config, points)},
           "cpu_baseline": last,
           "e2e": {"value": 1.0 / t, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    from probreg_b200 import _cabi, cpd, dist as pdist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: probreg_b200 has no CPU path")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of a one-GPU run (each rank holds only its shard's sums)")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        import torch.distributed as tdist
        tdist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        comm = pdist.Communicator.from_torch(local_rank)

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    n = args.points
    kind = args.kind
    if kind == "nonrigid":
        return run_nonrigid(args, torch, _cabi, cpd, barrier, local_rank, world)
    tf_kind = _cabi.TF_AFFINE if kind == "affine" else _cabi.TF_RIGID
    src, tgt = workload(n, kind)
    lo, hi = pdist.shard_bounds(n, rank, world)
    origin = tgt.mean(axis=0)

    # ---- device-resident arm -------------------------------------------------------------------
    h = _cabi.Handle(3, device=local_rank)
    if comm is not None:
        comm.attach(h)
    h.set_source(src)
    h.set_target(tgt[lo:hi], n_global=n, frame_origin=origin)
    s2 = h.sigma2_init()
    q0 = 1.0 + n * 3 * 0.5 * np.log(s2)

    def reset():
        h.set_state(tf_kind, True, 0.0, np.identity(3), np.zeros(3), 1.0, s2, q0)

    reset()
    sampler = ClockSampler(world) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        h.em_step(read=False)
    h.sync()
    # keep the GPUs under the same load until the poller is up (its start-up must not fall into the timed
    # region); then rewind the EM state so that the timed iterations are the first ones of a registration
    t_up = time.perf_counter()
    ready = torch.zeros(1, device="cuda")
    while True:
        for _ in range(10):
            h.em_step(read=False)
        h.sync()
        ready[0] = 1.0 if (sampler is None or sampler.count() >= 2 * world or time.perf_counter() - t_up > 3.0) else 0.0
        if world > 1:
            tdist.broadcast(ready, src=0)
        if ready.item() > 0:
            break
    reset()
    for _ in range(3):
        h.em_step(read=False)
    h.sync()
    barrier()
    launches0 = h.launch_count()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        h.flush_l2()
        h.event_record(2 * i)
        h.em_step(read=False)
        h.event_record(2 * i + 1)
    h.sync()
    barrier()
    t_wall1 = time.perf_counter()
    t_wall = t_wall1 - t_wall0
    launches = h.launch_count() - launches0
    clocks = sampler.stop(t_wall0, t_wall1, t_up) if sampler else None
    if args.dump_outputs:
        lin, t, scale, sigma2, q, n_p, _ = h.em_run(0, 0.0)        # maxiter 0: the state the last step left, no further step
        pt1, p1, px, _ = h.last_estep()
        dump_outputs(args.dump_outputs, {"lin": lin, "t": t, "scale": scale, "sigma2": sigma2, "q": q, "n_p": n_p,
                                         "pt1": pt1, "p1": p1, "px": px})
    per_step = np.array([h.event_elapsed(2 * i, 2 * i + 1) for i in range(args.steps)])
    total_ms = float(per_step.sum())
    if world > 1:
        tt = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        tdist.all_reduce(tt, op=tdist.ReduceOp.MAX)
        total_ms = float(tt.item())
    ms_per_step = total_ms / args.steps
    value = 1e3 / ms_per_step
    final = h.em_step(read=True)            # the loop did real work: parameters moved towards the truth

    # ---- multi-rank runs: the sharded loop against the same iterations on ONE GPU (asserted, rank 0) ---------------
    shard_check = None
    if world > 1:
        reset()
        for _ in range(2):
            h.em_step(read=False)
        sharded = h.em_step(read=True)
        barrier()
        if rank == 0:
            h1 = _cabi.Handle(3, device=local_rank)
            h1.set_source(src)
            h1.set_target(tgt)
            s2_1 = h1.sigma2_init()
            h1.set_state(tf_kind, True, 0.0, np.identity(3), np.zeros(3), 1.0, s2_1, 1.0 + n * 3 * 0.5 * np.log(s2_1))
            for _ in range(2):
                h1.em_step(read=False)
            single = h1.em_step(read=True)
            h1.close()
            shard_check = {"iterations": 3, "sigma2_sharded": sharded[3], "sigma2_single_gpu": single[3],
                           "sigma2_rel_diff": abs(sharded[3] - single[3]) / single[3],
                           "lin_max_abs_diff": float(np.abs(sharded[0] - single[0]).max()),
                           "t_max_abs_diff": float(np.abs(sharded[1] - single[1]).max()),
                           "sigma2_0_rel_diff": abs(s2 - s2_1) / s2_1}
            shard_check["agree"] = bool(shard_check["sigma2_rel_diff"] < 1e-7 and shard_check["lin_max_abs_diff"] < 1e-7
                                        and shard_check["t_max_abs_diff"] < 1e-7)
            if not shard_check["agree"]:
                raise SystemExit("sharded run disagrees with the single-GPU run: %r" % (shard_check,))
        barrier()

    # ---- stage breakdown (profiling events, one sync per step; not part of `value`) -----------------
    h.set_profiling(True)
    stages = []
    for _ in range(5):
        h.flush_l2()
        h.em_step(read=False)
        stages.append(h.stage_times())
    h.set_profiling(False)
    st = np.median(np.array(stages), axis=0)
    names = ["pack", "pass1", "finalize1", "pass2", "finalize2", "moments_mstep"]
    t_estep_ms = float(st[1] + st[3])
    n_local = hi - lo

    # ---- end to end through the public API with host (pinned) buffers ---------------------------
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
        t.numpy()[...] = a
        return t.numpy()

    src_p, tgt_p = pinned(src), pinned(tgt)
    r = (cpd.AffineCPD if kind == "affine" else cpd.RigidCPD)(src_p, device=local_rank, comm=comm)
    r.registration(tgt_p, maxiter=1, tol=-1.0)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        res = r.registration(tgt_p, maxiter=1, tol=-1.0)
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    # amortised: one upload, K iterations, as a user's registration_cpd(maxiter=K) behaves
    t0 = time.perf_counter()
    r.registration(tgt_p, maxiter=args.steps, tol=-1.0)
    barrier()
    e2e_amort_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        tt = torch.tensor([e2e_s, e2e_amort_s], dtype=torch.float64, device="cuda")
        tdist.all_reduce(tt, op=tdist.ReduceOp.MAX)
        e2e_s, e2e_amort_s = float(tt[0].item()), float(tt[1].item())
    h2d = src.nbytes + tgt[lo:hi].nbytes
    d2h = 16 * 8

    if rank != 0:
        if world > 1:
            tdist.destroy_process_group()
        return

    # ---- rooflines -----------------------------------------------------------------------------
    probe = _cabi.microbench(local_rank)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    flops = FLOP_PER_PAIR_ITER * float(n_local) * float(n)
    ach_tf = flops / (t_estep_ms * 1e-3) / 1e12
    nominal_tf = 2.0 * 128 * probe["sm_count"] * (clocks.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12
    bytes_iter = hbm_bytes_per_iter(n_local, n)
    traffic, traffic_src = None, None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch of the two E-step kernels, from the committed ncu capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        if world == 1 and n == 100000:
            traffic = sum(k["dram_read_bytes"] + k["dram_write_bytes"] for k in tj["kernels"].values())
            traffic_src = tj["source"]
    except Exception:
        pass
    roofline = {
        "bound": "fp32",
        "kernel": "pass1_kernel + pass2_kernel (fused E-step, never materialises P)",
        "achieved": ach_tf, "peak": probe["ffma_tflops"], "unit": "TFLOP/s", "frac": ach_tf / probe["ffma_tflops"],
        "peak_source": "FFMA issue-rate probe run in this process (cpd_microbench); nominal 2*128*SMs*clk = %.1f" % nominal_tf,
        "flop_per_pair": FLOP_PER_PAIR_ITER, "pairs_per_launch": float(n_local) * float(n),
        "instruction_ceiling_frac": ach_tf / (probe["ffma_tflops"] * (29.0 / (19.0 * 2.0))),
        "mufu_ex2_gops_probe": probe["mufu_ex2_gops"],
        "traffic": traffic,
        "traffic_source": traffic_src,
        "hbm": {"bound": "hbm", "achieved": bytes_iter / (t_estep_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": bytes_iter / (t_estep_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                "algorithmic_bytes": bytes_iter,
                "materialised_equiv_gbs": 8.0 * n_local * n / (t_estep_ms * 1e-3) / 1e9,
                "materialised_equiv_frac": 8.0 * n_local * n / (t_estep_ms * 1e-3) / 1e9 / hbm_peak},
    }
    cpu = cpu_sample(kind, n, 4 * args.cpu_cols) if world == 1 and not args.no_cpu else None      # ~10-20 s of CPU work
    extras = run_extras() if world == 1 and args.extras and args.config == 2 else None
    also = run_also(args) if world == 1 and args.config == 2 and not args.no_also else None
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "dtype_note": "pair arithmetic f32 (packed f32x2); every sum beyond 64 terms, the moments and the M-step f64",
        "data": "synthetic",
        "config": {"workload": workload_string(args.config, n), "baseline_config": args.config, "also": also,
                   "sharded_equals_single_gpu": (shard_check or {}).get("agree"),
                   "parallelism": "target-sharded x%d, sources replicated, one 32-double all-reduce per iteration (%s)"
                                  % (world, "fused into the M-step kernel over NVLink peer memory" if (comm is not None and comm.use_p2p)
                                     else ("ncclAllReduce" if world > 1 else "none needed")),
                   "l2": "flushed (256 MiB memset) between timed iterations, outside the event pairs",
                   "timing": "CUDA event pair per iteration on the library stream, summed, max over ranks"},
        "wall_ms_per_step_incl_flush": t_wall * 1e3 / args.steps,
        "e2e": {"value": 1.0 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "what": "%sCPD.registration(target, maxiter=1) per step: H2D both clouds (pinned), sigma2 init, "
                        "1 EM iteration, D2H MstepResult" % ("Affine" if kind == "affine" else "Rigid"),
                "amortised_value": 1.0 / e2e_amort_s,
                "amortised_what": "registration(maxiter=%d): one upload, per-iteration D2H of the MstepResult" % args.steps},
        "gpu_launches": int(launches),
        "stage_ms": dict(zip(names, [float(x) for x in st])),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "probe": probe,
        "result_check": {"sigma2_after_run": final[3], "scale": final[2], "lin": [float(x) for x in np.ravel(final[0])],
                         "sharded_vs_single_gpu": shard_check},
        "extras": extras,
    }
    emit(out)
    if world > 1:
        tdist.destroy_process_group()


def run_also(args):
    """Short runs of BASELINE configurations 3 and 5 in SUBPROCESSES (a fault there costs the main line nothing but this key);
    the compact summaries travel inside `config`, which the driver's record keeps."""
    out = {}
    for cfg, steps in ((3, 5), (5, 10)):
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--config", str(cfg), "--steps", str(steps), "--warmup", "3",
                                "--no-cpu", "--no-also"], capture_output=True, text=True, timeout=300, cwd=ROOT)
            lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
            if r.returncode != 0 or not lines:
                out["config%d" % cfg] = {"error": "exit %d: %s" % (r.returncode, (r.stderr or r.stdout)[-300:])}
                continue
            j = json.loads(lines[-1])
            out["config%d" % cfg] = {"workload": j["config"]["workload"], "value": j["value"], "unit": j["unit"], "ms_per_step": j["ms_per_step"],
                                    "e2e": j["e2e"]["value"], "roofline_frac": j["roofline"]["frac"],
                                    "roofline_achieved": j["roofline"]["achieved"], "roofline_unit": j["roofline"]["unit"],
                                    "setup_ms": j.get("setup_ms"), "setup": j.get("setup")}
        except Exception as e:                  # noqa: BLE001
            out["config%d" % cfg] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
    return out


def gram_roofline(n, ms_four_products):
    """Tensor roofline of the G X product kernel (gi_gram_ts_kernel): 6 int8 MMAs of 128 x 112 x 32 per 32 points, row tile and column
    pass (2 passes for K = 200) against the int8 rate = twice the measured bf16 peak (MEASURED_PEAKS.json, burst)."""
    if not ms_four_products or ms_four_products <= 0:
        return None
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
        src = "2 x measured bf16 (MEASURED_PEAKS.json)"
    except Exception:
        bf16, src = 1590.0, "2 x fallback bf16 (B200_PROFILING.md)"
    tiles = (n + 127) // 128
    stages = ((n + 511) // 512 * 512) // 32
    ops = 4 * 2 * tiles * stages * 6 * 2.0 * 128 * 112 * 32            # 4 products x 2 column passes
    ach = ops / (ms_four_products * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": "gi_gram_ts_kernel (+ split / reduce / column maxima inside the timed phase)", "achieved": ach,
            "peak": 2.0 * bf16, "unit": "Top/s (int8)", "frac": ach / (2.0 * bf16), "peak_source": src}


def run_nonrigid(args, torch, _cabi, cpd, barrier, local_rank, world):
    """BASELINE configuration 5: non-rigid CPD with G ~= Q Bc Q^T of rank 200 (no reference counterpart: the reference solves the
    dense M x M system, cpd.py:296).  A step = one EM iteration (E-step + low-rank M-step, cpd_nonrigid_step); the one-off
    factorisation (range finder on tcgen05 G X products + blocked orthonormalisation) is reported as `setup_ms`."""
    rank = int(os.environ.get("RANK", "0"))
    n, K = args.points, 200
    src, tgt = workload(n, "nonrigid")
    h = _cabi.Handle(3, device=local_rank)
    h.set_source(src)
    h.set_target(tgt)
    s2 = h.sigma2_init()
    h.set_profiling(True)
    setup_wall_ms, setup_cold_ms = None, None
    for rep in range(2):          # cold: buffer allocation + the first-use self-check of the tensor-core product; warm: what a second source costs
        h.sync()
        t0 = time.perf_counter()
        h.nonrigid_lowrank_begin(2.0, 2.0, s2, 0.0, K, 2, 0)
        h.sync()
        setup_wall_ms = (time.perf_counter() - t0) * 1e3
        if rep == 0:
            setup_cold_ms = setup_wall_ms
    setup = {k: float(v) for k, v in dict(h.lowrank_setup_times()).items()}
    h.set_profiling(False)
    sampler = ClockSampler(world) if rank == 0 else None
    if sampler:
        sampler.start()
    t_up = time.perf_counter()
    while True:
        for _ in range(10):
            h.nonrigid_step()
        if sampler is None or sampler.count() >= 2 or time.perf_counter() - t_up > 3.0:
            break
    h.nonrigid_restart(2.0, s2, 0.0)
    for _ in range(max(args.warmup, 3)):
        h.nonrigid_step()
    h.sync()
    launches0 = h.launch_count()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        h.flush_l2()
        h.event_record(2 * i)
        sig = h.nonrigid_step()
        h.event_record(2 * i + 1)
    h.sync()
    t_wall1 = time.perf_counter()
    launches = h.launch_count() - launches0
    clocks = sampler.stop(t_wall0, t_wall1, t_up) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sigma2": sig, "w": h.nonrigid_w(), "moved": h.nonrigid_moved()})
    per_step = np.array([h.event_elapsed(2 * i, 2 * i + 1) for i in range(args.steps)])
    ms_per_step = float(per_step.sum()) / args.steps
    h.set_profiling(True)
    stages = []
    for _ in range(5):
        h.flush_l2()
        h.nonrigid_step()
        stages.append(h.stage_times())
    h.set_profiling(False)
    st = np.median(np.array(stages), axis=0)
    names = ["pack", "pass1", "finalize1", "pass2", "finalize2", "moments_mstep"]
    t_estep_ms = float(st[1] + st[3])

    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
        t.numpy()[...] = a
        return t.numpy()

    src_p, tgt_p = pinned(src), pinned(tgt)
    r = cpd.NonRigidCPD(src_p, beta=2.0, lmd=2.0, low_rank=K, device=local_rank)
    t0 = time.perf_counter()
    r.registration(tgt_p, maxiter=1, tol=-1.0)
    cold_s = time.perf_counter() - t0
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r.registration(tgt_p, maxiter=1, tol=-1.0)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    probe = _cabi.microbench(local_rank)
    flops = FLOP_PER_PAIR_ITER * float(n) * float(n)
    ach_tf = flops / (t_estep_ms * 1e-3) / 1e12
    gram_flop = 2.0 * float(n) * float(n) * K
    out = {
        "metric": METRIC, "value": 1e3 / ms_per_step, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "dtype_note": "pair arithmetic f32; G X products TF32 x3 (hi/lo split) on tcgen05 with FP32 TMEM accumulation per 2048-point chunk, "
                      "FP64 across chunks; factors, K x K system and its LU f64",
        "data": "synthetic",
        "config": {"workload": workload_string(args.config, n), "baseline_config": args.config,
                   "parallelism": "single GPU", "l2": "flushed (256 MiB memset) between timed iterations, outside the event pairs",
                   "timing": "CUDA event pair per iteration on the library stream, summed"},
        "setup_ms": setup_wall_ms, "setup_cold_ms": setup_cold_ms,
        "setup": dict(setup, what="one-off per source: 4 products G X (K = 200: tcgen05 kind::i8, 8-bit digit planes, A operand and int32 "
                                  "accumulators in TMEM) + 3 blocked orthonormalisations + Q^T G Q",
                      gram_tflops_useful=(4 * gram_flop / (setup["gram_products_ms"] * 1e-3) / 1e12) if setup["gram_products_ms"] > 0 else None,
                      gram_roofline=gram_roofline(n, setup["gram_products_ms"])),
        "e2e": {"value": 1.0 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(src.nbytes + tgt.nbytes), "d2h_bytes_per_step": int(8 + src.nbytes),
                "what": "NonRigidCPD(low_rank=200).registration(target, maxiter=1) per step: H2D both clouds (pinned), sigma2 init, restart on "
                        "the cached factors of the unchanged source, 1 EM iteration, D2H sigma2 + W",
                "cold_first_call_s": cold_s},
        "gpu_launches": int(launches),
        "stage_ms": dict(zip(names, [float(x) for x in st])),
        "roofline": {"bound": "fp32", "kernel": "pass1_kernel + pass2_kernel (fused E-step of the non-rigid iteration)",
                     "achieved": ach_tf, "peak": probe["ffma_tflops"], "unit": "TFLOP/s", "frac": ach_tf / probe["ffma_tflops"],
                     "peak_source": "FFMA issue-rate probe run in this process (cpd_microbench)",
                     "flop_per_pair": FLOP_PER_PAIR_ITER, "pairs_per_launch": float(n) * float(n), "traffic": None,
                     "estep_share_of_step": t_estep_ms / ms_per_step},
        "cpu_baseline": None,
        "clocks": clocks,
        "result_check": {"sigma2_after_run": float(sig)},
    }
    emit(out)


def run_extras():
    """Side measurements (BASELINE configs 3 and 5, first-hardware-run probes of the newest paths) in a SUBPROCESS, after the bench
    line's own numbers are final: whatever happens there -- an exception, a CUDA fault, a time-out -- costs the bench line
    nothing but this key.  tools/bench_extras.py prints one JSON object."""
    import subprocess

    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_extras.py")], capture_output=True, text=True, timeout=420,
                           cwd=ROOT)
        lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": "exit %d: %s" % (r.returncode, (r.stderr or r.stdout)[-400:])}
        return json.loads(lines[-1])
    except Exception as e:                      # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


DUMP_BYTES = 63 * 10 ** 6       # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(path, arrays):
    """--dump-outputs: write `arrays` as <path>/<name>.npy in float64, so that two builds run with the same arguments can be compared
    output for output.  Past DUMP_BYTES in all, every array of more than 1 MiB keeps the same share of its rows, a sample drawn with
    seed 0 from its row count alone: arrays with the same rows (p1 and px) keep the same rows, and so does a second build."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    big = [k for k, a in arrays.items() if a.nbytes > 1 << 20]
    small_bytes = sum(a.nbytes for k, a in arrays.items() if k not in big)
    big_bytes = sum(arrays[k].nbytes for k in big)
    if small_bytes + big_bytes > DUMP_BYTES:
        keep = (DUMP_BYTES - small_bytes) / float(big_bytes)
        for k in big:
            n = arrays[k].shape[0]
            rows = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * keep)), replace=False))
            arrays[k] = arrays[k][rows]
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def emit(obj):
    """The ONE JSON line goes to the real stdout; everything else this process (or NCCL, which
    prints its version banner to fd 1) writes during the run has been diverted to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json configuration: 2 rigid 100k (the metric's), 3 affine 250k, 4 rigid 1M (8 GPUs), 5 non-rigid low-rank 50k")
    ap.add_argument("--points", type=int, default=0, help="override the configuration's point count")
    ap.add_argument("--cpu-cols", type=int, default=2000, help="target columns in the CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-also", action="store_true", help="skip the short runs of configurations 3 and 5 reported under config.also")
    ap.add_argument("--extras", action="store_true", help="add the side measurements of tools/bench_extras.py (key \"extras\")")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                                                          "(float64; one GPU, --impl ours)")
    args = ap.parse_args()
    if not 1 <= args.steps <= 4096:
        ap.error("--steps must be in 1 .. 4096 (each timed step takes two of the library's 8192 event slots)")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.kind = WORKLOADS[args.config][0]
    if args.points <= 0:
        args.points = WORKLOADS[args.config][1]
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
