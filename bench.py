#!/usr/bin/env python
"""bench.py -- particle-steps/sec of the SMC hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (config 2 of BASELINE.json): bootstrap filter of the stochastic-volatility
model (StochVol defaults), N = 1e7 particles per GPU, systematic resampling,
ESSrmin = 0.5, observations = `np.random.seed(1); StochVol().simulate(1000)` (committed
fixture; cycled if K > 1000).  One "step" = one filter step (propagate -> log-weight ->
normalise/ESS -> resample if ESS < N/2) over all N particles; value = N * K / time.

* `value`  : device-timed (CUDA events on the launching stream), particles resident
             in HBM when the timed region starts;
* `e2e`    : the same filter through the public API `particles_b200.SMC(...).run()`,
             host observations in, host summaries out, wall clock around the call;
* `roofline`: algorithmic bytes of the step kernel / its CUDA-event time, against
             MEASURED_PEAKS.json `hbm_gbs`;
* `cpu_baseline`: the oracle's NumPy restatement of the reference loop, timed on the
             host cores of this box on a bounded sample (a few steps at N = 1e7).
With --impl reference the CPU arm alone runs (all host cores, replicas as in multiSMC).
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
sys.dont_write_bytecode = True     # the tree may be read-only: no __pycache__ next to the sources

N_PER_GPU = 10_000_000
ESSRMIN = 0.5
SCHEME = "systematic"
HBM_FALLBACK_GBS = 6650.0      # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_SAMPLE = 1 << 19          # particles (and summary rows) written by --dump-outputs
FP64_INST_PER_PAIR = 105       # fp64 instructions of the streaming step per pair of particles; superseded by the
                               # committed ncu capture (profiles/*_ncu_summary.json: move.fp64_inst_per_pair) when present


def load_data(K):
    g = np.load(os.path.join(ROOT, "tests", "golden", "golden_stats.npz"))
    y = g["data/sv_seed1_T1000"]
    reps = (K + len(y) - 1) // len(y)
    return np.tile(y, reps)[:K].astype(np.float64)


def parity_block(K, n_total, logLt, n_rs, note=None):
    """The north-star parity statement for THIS run: logLt after K steps against the reference's own NumPy runs
    (tests/golden/golden_sv_traj.npz: 8 seeded runs of particles.SMC at N = 1e5 on the same data, per-step
    logLt).  sigma = reference run-to-run sd scaled to this N, plus the standard error of the reference mean."""
    fn = os.path.join(ROOT, "tests", "golden", "golden_sv_traj.npz")
    if K > 1000 or not os.path.exists(fn):
        return {"logLt": logLt, "n_resample": n_rs, "note": "no reference trajectory for this K"}
    g = np.load(fn)
    ll, rc, n_ref = g["logLts"][:, K - 1], g["rs_cum"][:, K - 1], float(g["N"][0])
    mu, sd = float(ll.mean()), float(ll.std(ddof=1))
    sigma = float(np.sqrt(sd * sd * n_ref / n_total + sd * sd / len(ll)))
    out = {"logLt": logLt, "ref_mean": mu, "ref_sd_at_1e5": sd, "ref_sd_scaled": sigma,
           "n_sigma": (logLt - mu) / sigma, "rel_err": abs(logLt - mu) / abs(mu), "n_resample": n_rs,
           "ref_n_resample": [int(rc.min()), int(rc.max())],
           "within_3_sigma": bool(abs(logLt - mu) < 3 * sigma)}
    if note:
        out["note"] = note
    return out


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback"


def ncu_fp64_per_pair():
    """fp64 (DFMA/DMUL/DADD/DSETP) instructions per pair of particles of a non-resampling step, counted by ncu's
    source page in the committed capture; the constant above if there is none."""
    import glob
    for fn in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_summary.json")), reverse=True):
        try:
            return float(json.load(open(fn))["move"]["fp64_inst_per_pair"]), os.path.basename(fn)
        except Exception:
            continue
    return float(FP64_INST_PER_PAIR), "constant"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_move launch (no-resampling step) from
    the committed `ncu --set full` capture (profiles/*_ncu_summary.json); None if absent."""
    import glob
    for fn in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_ncu_summary.json")), reverse=True):
        try:
            return float(json.load(open(fn))["move"]["dram_traffic_bytes"])
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            inside = t0 <= ts <= t1 + 0.1
            try:
                if inside:
                    sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            if inside:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:   # region shorter than one sample: use the closest samples
            for ts, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "power_w_max": float(max(pw)) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------
# CPU arm: the oracle's NumPy restatement of particles.core.SMC (kind "port")
# ---------------------------------------------------------------------------------------
def _cpu_worker(args):
    n, steps, seed = args
    from oracle import smc_numpy as orc
    y = [np.atleast_1d(v) for v in load_data(steps + 1)]
    np.random.seed(seed)
    pf = orc.SMC(orc.Bootstrap(orc.StochVol(), y), N=n, resampling=SCHEME, ESSrmin=ESSRMIN)
    pf.step()                                   # warm-up step (page faults, allocator)
    t0 = time.perf_counter()
    pf.run(nsteps=steps)
    return time.perf_counter() - t0, pf.logLt


REF_DIR = os.path.join(ROOT, "oracle", "_ref")        # the live reference's package (oracle/make_ref.sh), if present


def have_live_reference():
    return os.path.isdir(os.path.join(REF_DIR, "particles"))


def _ref_worker(args):
    """The UNMODIFIED reference: particles.SMC on the same workload (oracle/_ref, copied by oracle/make_ref.sh)."""
    n, steps, seed = args
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import particles
    from particles import resampling as rrs
    from particles import state_space_models as rssm
    y = [np.atleast_1d(v) for v in load_data(steps + 1)]
    np.random.seed(seed)
    rrs.systematic(np.full(16, 1.0 / 16))         # numba JIT of inverse_cdf outside the timed region
    pf = particles.SMC(fk=rssm.Bootstrap(ssm=rssm.StochVol(), data=y), N=n, resampling=SCHEME, ESSrmin=ESSRMIN)
    next(pf)                                       # warm-up step (page faults, allocator)
    t0 = time.perf_counter()
    for _ in range(steps):
        next(pf)
    return time.perf_counter() - t0, pf.logLt


def cpu_baseline(n, steps, workers=1, live=False):
    """particle-steps/s of the live reference (`live`) or of the NumPy port; `workers` independent filters in
    processes (the reference's only parallelism is replica-level: utils.multiplexer / multiSMC)."""
    fn = _ref_worker if live else _cpu_worker
    if workers == 1:
        dt, _ = fn((n, steps, 1))
        wall = dt
    else:
        import multiprocessing as mp
        with mp.get_context("spawn").Pool(workers) as pool:
            res = pool.map(fn, [(n, steps, 1 + i) for i in range(workers)])
            wall = max(r[0] for r in res)
    return workers * n * steps / wall, wall


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                        # ~1.5 GB of NumPy temporaries per worker at N=1e7
        import psutil
        mem_workers = int(psutil.virtual_memory().available / 2.0e9)
    except Exception:
        mem_workers = 16
    # replicas beyond ~16 saturate the host's memory bandwidth on this class of box (measured: 16
    # workers 2.2e8, 32 workers 1.5e8, 128 workers 0.9e8 particle-steps/s in aggregate): capped at 16
    workers = max(1, min(cores, mem_workers, 16))
    n = N_PER_GPU
    K = args.steps
    reps = max(1, min(args.warmup, 1))
    live = have_live_reference()
    for _ in range(reps):
        cpu_baseline(n // 10, 1, 1, live)
    value, wall = cpu_baseline(n, K, workers, live)
    port_value = cpu_baseline(n, K, workers, False)[0] if live else value
    kind = "reference" if live else "port"
    what = ("the reference's own particles.SMC (oracle/_ref, copied from the reference checkout by "
            "oracle/make_ref.sh)" if live else
            "oracle NumPy restatement of particles.core.SMC (no oracle/_ref on this box)")
    out = {
        "impl": "reference", "metric": "particle-steps/sec (N x T), Bootstrap SV", "value": value,
        "unit": "particle-steps/s", "n_gpus": args.gpus, "steps": K, "warmup": reps,
        "ms_per_step": 1e3 * wall / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"StochVol bootstrap N={n} systematic ESSrmin=0.5 (config 2), "
                               f"{workers} replica filters in {workers} processes"},
        "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": workers, "kind": kind,
                         "sample": f"{K} filter steps at N={n} per worker after 1 warm-up step; " + what,
                         "port_value": port_value},
        "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
def multi_gpu_parity(table, spec, y, rank, world):
    """Driver-side evidence that the sharded filter is correct (every rank calls this):
    (1) all ranks hold bit-identical summaries of the timed run;
    (2) the EXACT global-resampling mode on `world` GPUs reproduces the single-device filter of the same seed and
        the same total N (Philox counters follow the global particle index): max |delta logLt| over all steps."""
    import torch
    import torch.distributed as dist
    from particles_b200.core import _FusedEngine
    from particles_b200.parallel import ShardedFilter
    t = torch.from_numpy(np.ascontiguousarray(table)).cuda()
    allt = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    identical = all(bool(torch.equal(o, t)) for o in allt)
    n_x, T_x = 200_000, 200
    sp = dict(spec)
    sp["data"] = y[:T_x].reshape(-1, 1).copy()
    f = ShardedFilter(sp, n_x, SCHEME, 0.5, 4242, rank, world, resampling_mode="global")
    f.step(T_x)
    f.state()
    tab = f.summ[:T_x].clone()
    f.close()
    res = torch.zeros(3, dtype=torch.float64, device="cuda")
    if rank == 0:
        e = _FusedEngine(sp, n_x * world, SCHEME, 0.5, 4242)
        e.step(T_x)
        one = e.summ[:T_x].clone()
        e.close()
        res[0] = (one[:, 1] - tab[:, 1]).abs().max()
        res[1] = float(torch.equal(one[:, 2], tab[:, 2]))
        res[2] = tab[:, 2].sum()
    dist.broadcast(res, 0)
    return {"rank_identical_summaries": identical,
            "global_vs_single_device": {"max_abs_dlogLt": float(res[0]), "same_resampling_decisions": bool(res[1] > 0),
                                        "resampling_steps": int(res[2]), "n_per_gpu": n_x, "T": T_x,
                                        "ok": bool(res[0] < 1e-9 and res[1] > 0)}}



def workload(args, K):
    """(label, make_fk(y_list) -> Feynman-Kac object, observations (K, dy), scheme, essrmin, state dim, parity?)
    for --config: c2 = BASELINE config 2 (the bench); c3i / c3ii = config 3 as SURVEY.md 8(d) splits it."""
    from particles_b200 import kalman, state_space_models as ssm
    if args.config == "c2":
        y = load_data(K).reshape(-1, 1)
        return ("StochVol bootstrap", lambda yl: ssm.Bootstrap(ssm=ssm.StochVol(), data=yl), y, SCHEME, ESSRMIN, 1, True)
    import torch
    torch.manual_seed(0)
    from particles_b200 import device
    device.seed(12345)
    if args.config == "c3i":      # BearingsOnly (IndepProd(Normal, Normal, Dirac, Dirac), d = 4), Bootstrap, stratified
        m = ssm.BearingsOnly()
        _, ys = m.simulate(K)
        y = np.array([np.asarray(v.cpu()).reshape(-1) for v in ys])
        return ("BearingsOnly bootstrap (d=4)", lambda yl: ssm.Bootstrap(ssm=ssm.BearingsOnly(), data=yl), y,
                "stratified", ESSRMIN, 4, False)
    m = kalman.MVLinearGauss_Guarniero_etal(alpha=0.4, dx=4)       # 4-D MvNormal state, optimal (guided) proposal
    _, ys = m.simulate(K)
    y = np.array([np.asarray(v.cpu()).reshape(-1) for v in ys])
    return ("MVLinearGauss (Guarniero et al, dx=4) guided", lambda yl: ssm.GuidedPF(
        ssm=kalman.MVLinearGauss_Guarniero_etal(alpha=0.4, dx=4), data=yl), y, "stratified", ESSRMIN, 4, False)


def dump_outputs(path, eng, table):
    """--dump-outputs: what a caller of the timed filter receives after its last step, as float64 .npy files:
    X (particles, (N,) or (N, d)), lw (log-weights), A (ancestors; the identity when that step did not resample, and
    so after a single step, where the public API's SMC.A is None) and the per-step ESSs / logLts / rs_flags.  Of more than DUMP_SAMPLE particles a fixed seeded sample is written (its
    indices in index.npy), of more than DUMP_SAMPLE steps the last ones: at most (d + 3) * 4 MB + 12 MB in all."""
    import torch
    cur = (table.shape[0] - 1) & 1                 # step s writes buffers [s & 1]
    idx = np.arange(eng.N)
    if eng.N > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(eng.N, DUMP_SAMPLE, replace=False))
    sel = torch.from_numpy(idx).to(eng.A.device)
    x = eng.X[cur].index_select(eng.X[cur].ndim - 1, sel)
    rows = table[-DUMP_SAMPLE:]
    out = {"index": idx, "X": x.t() if x.ndim > 1 else x, "lw": eng.lw[cur].index_select(0, sel),
           "A": eng.A.index_select(0, sel) if table[-1, 2] else sel,
           "ESSs": rows[:, 0], "logLts": rows[:, 1], "rs_flags": rows[:, 2]}
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import particles_b200 as pb
    from particles_b200 import state_space_models as ssm
    from particles_b200.core import _FusedEngine
    if world > 1:
        from particles_b200.parallel import ShardedFilter

    K, W = args.steps, max(args.warmup, 3)
    n = args.n
    label, make_fk, y, scheme, essrmin, dim, has_ref = workload(args, max(K, W))
    y_list = [np.asarray(v, dtype=np.float64).reshape(-1) for v in y[:K]]
    fk = make_fk(y_list)
    spec = ssm.fused_spec(fk)
    assert spec is not None, "this workload has no fused kernel"
    b_st, b_rs = 16.0 * dim + 16.0, 16.0 * dim + 40.0 + 16.0      # algorithmic bytes / particle (SURVEY.md 8d)

    def make_engine(nsteps, seed):
        sp = dict(spec)
        sp["data"] = np.ascontiguousarray(y[:nsteps])
        if world == 1:
            return _FusedEngine(sp, n, scheme, essrmin, seed)
        return ShardedFilter(sp, n, scheme, essrmin, seed, rank, world, resampling_mode=args.resampling_mode)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: W untimed steps on a throw-away filter (same kernels, same sizes)
    wu = make_engine(W, 123)
    wu.step(W)
    torch.cuda.synchronize()
    wu.close()

    eng = make_engine(K, 2024)
    launches0 = eng.ctx.launches
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record()
    eng.step(K)                                   # EXACTLY K steps, no host sync inside
    e1.record()
    barrier()
    tw1 = time.perf_counter()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    launches = eng.ctx.launches - launches0      # kernels launched in the timed region (counted by libsmcb)
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    table = eng.summ.cpu().numpy()
    n_rs = int(table[:, 2].sum())
    logLt = float(table[K - 1, 1])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, table)
    eng.close()

    # per-kernel CUDA-event timing of the same K steps (separate pass, same kernels)
    roof = None
    if rank == 0 and world == 1:
        eng2 = make_engine(K, 2024)
        kms, kcnt = eng2.step_timed(K)
        t2 = eng2.summ.cpu().numpy()
        nrs2 = int(t2[:, 2].sum())
        eng2.close()
        peak, how = hbm_peak()
        # algorithmic bytes of the step kernel (SURVEY.md 8d): 32 B/particle on a non-resampling step (x, lw in;
        # x', lw' out); 56 B on a resampling one (lw in, cdf out | cdf in, A out, gather x, x', lw' out)
        n_st, n_rs_k = kcnt["step"], kcnt["step_rs"]
        step_us = 1e3 * kms["step"] / n_st if n_st else float("nan")
        ach = n * b_st / (step_us * 1e-6) / 1e9
        rs_us = 1e3 * kms["step_rs"] / n_rs_k if n_rs_k else None
        roof = {"bound": "hbm", "kernel": "k_step<%s>, non-resampling steps" % label,
                "achieved": ach, "peak": peak, "peak_source": how, "unit": "GB/s",
                "frac": ach / peak, "traffic": ncu_traffic(), "traffic_source": "committed ncu capture (profiles/)",
                "avg_launch_us": step_us, "launches": n_st,
                "algorithmic_bytes_per_particle": {"no_resample": b_st, "resample": b_rs},
                "resampling_steps": {"launches": n_rs_k, "avg_launch_us": rs_us,
                                     "achieved": (n * b_rs / (rs_us * 1e-6) / 1e9) if rs_us else None,
                                     "frac": (n * b_rs / (rs_us * 1e-6) / 1e9 / peak) if rs_us else None},
                "whole_run_frac": (n * (b_st * n_st + b_rs * n_rs_k) / ((kms["step"] + kms["step_rs"]) * 1e-3) / 1e9) / peak,
                "share_of_step_time": {k: v / sum(kms.values()) for k, v in kms.items()}}
        try:                                   # secondary bound: fp64 FMA issue, measured on this device now
            import ctypes as C
            from particles_b200 import _lib, device
            ctx = device.context()
            o3 = (C.c_double * 3)()
            _lib.check(ctx.lib.smcb_measure_fp64_peak(ctx.handle, 0.0, o3))
            # fp64 work of the streaming step per pair of particles (SASS of the loop body, DESIGN.md section 5)
            per_pair, per_pair_src = ncu_fp64_per_pair()
            flops = per_pair * 2.0 * (n / 2.0)
            roof["secondary"] = {"bound": "fp64", "peak": o3[0], "unit": "TFLOP/s (DFMA = 2 flop), measured by "
                                 "smcb_measure_fp64_peak in this run",
                                 "achieved": flops / (step_us * 1e-6) / 1e12,
                                 "frac": flops / (step_us * 1e-6) / 1e12 / o3[0],
                                 "fp64_instructions_per_pair": per_pair, "fp64_instructions_source": per_pair_src}
        except Exception as exc:               # noqa: BLE001  (an older library without the probe)
            roof["secondary"] = {"bound": "fp64", "error": str(exc)}

    # end-to-end through the public API: host observations in, host summaries out
    e2e = None
    if world == 1:
        y_host = y_list
        runs = []
        # one untimed warm-up call of W steps through the same API (first-use costs of the process: the caching
        # allocator's cudaMalloc of the particle arrays, pinned staging, module loading)
        wpf = pb.SMC(fk=make_fk(y_host[:max(W, 3)]), N=n, resampling=scheme, ESSrmin=essrmin, seed=76)
        wpf.run()
        if wpf._engine is not None:
            wpf._engine.close()
        del wpf
        for rep_ in range(3):                          # whole call repeated; the median is reported
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pf = pb.SMC(fk=make_fk(y_host), N=n, resampling=scheme, ESSrmin=essrmin, seed=77)
            pf.run()
            ll = pf.logLt                              # forces the device->host read of the result
            torch.cuda.synchronize()
            runs.append(time.perf_counter() - t0)
            if pf._engine is not None:
                pf._engine.close()
            del pf
        dt = sorted(runs)[1]
        e2e = {"value": n * K / dt, "unit": "particle-steps/s", "h2d_bytes_per_step": 8 * int(y.shape[1]),
               "d2h_bytes_per_step": 32, "seconds": dt, "seconds_all_runs": runs, "logLt": ll,
               "h2d_bytes_per_step_note": "the observations (dy doubles per step)",
               "api": "particles_b200.SMC(fk=<Feynman-Kac model>, N).run(); median of 3 whole calls "
                      "(construction, pinned->device copy of the observations, T steps, device->host read of "
                      "the summaries) after one untimed warm-up call of W steps"}

    if world > 1:       # end to end through the public sharded API, every rank takes part
        from particles_b200.parallel import ShardedSMC
        y_host = y_list
        runs = []
        wsp = ShardedSMC(fk=make_fk(y_host[:max(W, 3)]), N=n, resampling=scheme, ESSrmin=essrmin, seed=76,
                         resampling_mode=args.resampling_mode)      # untimed warm-up call, as on one GPU
        wsp.run()
        wsp._engine.close()
        del wsp
        for rep_ in range(3):                          # whole call repeated; the median is reported
            barrier()
            t0 = time.perf_counter()
            sp = ShardedSMC(fk=make_fk(y_host), N=n, resampling=scheme,
                            ESSrmin=essrmin, seed=77, resampling_mode=args.resampling_mode)
            sp.run()
            ll = sp.logLt
            barrier()
            dtr = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            dist.all_reduce(dtr, op=dist.ReduceOp.MAX)
            runs.append(float(dtr.item()))
            sp._engine.close()
            del sp
        dt = sorted(runs)[1]
        e2e = {"value": n * world * K / dt, "unit": "particle-steps/s", "h2d_bytes_per_step": 8 * int(y.shape[1]),
               "d2h_bytes_per_step": 32, "seconds": dt, "seconds_all_runs": runs, "logLt": ll,
               "api": "particles_b200.parallel.ShardedSMC(fk=Bootstrap(StochVol(), data), N).run() on every rank; "
                      "median of 3 whole calls, max over ranks"}
    multi = None
    if world > 1:
        multi = multi_gpu_parity(table, spec, y, rank, world) if args.config == "c2" else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = None
    if world == 1 and not args.no_cpu and args.config == "c2":
        live = have_live_reference()
        v, wall = cpu_baseline(n, 4, 1, live)
        cpu = {"value": v, "unit": "particle-steps/s", "cores": 1, "kind": "reference" if live else "port",
               "sample": f"4 filter steps at N={n} after 1 warm-up step, single process (the reference runs one "
                         "filter on one core); " + ("the reference's own particles.SMC from oracle/_ref" if live
                                                    else "oracle NumPy restatement"),
               "port_value": cpu_baseline(n, 4, 1, False)[0] if live else v}
    total_n = n * world
    out = {
        "metric": "particle-steps/sec (N x T), Bootstrap SV", "value": total_n * K / (ms * 1e-3),
        "unit": "particle-steps/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{label} filter, N={n} particles per GPU "
                               f"(global {total_n}), T={K}, {scheme} resampling, ESSrmin={essrmin} "
                               + {"c2": "(BASELINE config 2" + (")" if world == 1 else "/4, particle-sharded)"),
                                  "c3i": "(BASELINE config 3, reference model as it is: Bootstrap)",
                                  "c3ii": "(BASELINE config 3, 4-D MvNormal guided path)"}[args.config],
                   "l2": "working set 4 x 80 MB of fp64 state per GPU > 126 MB L2 (no flush needed)",
                   "resampling_steps": n_rs, "logLt": logLt,
                   "parallelism": "single GPU" if world == 1 else
                   f"particles sharded over {world} GPUs, {args.resampling_mode} resampling"},
        "gpu_launches": launches,
        "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "e2e": e2e,
        "parity": None if not has_ref else parity_block(K, total_n, logLt, n_rs,
                               None if world == 1 or args.resampling_mode == "global" else
                               "island resampling: a different (consistent) estimator from the reference's global "
                               "scheme; logLt parity is statistical"),
    }
    if multi is not None and out["parity"] is not None:
        out["parity"]["multi_gpu"] = multi
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed filter steps (default: 1000 for c2, 500 for c3i / c3ii; 4 with --impl reference, "
                         "about 3 s per step per worker)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=None, help="particles per GPU (default: 1e7 for c2, 1e6 for c3)")
    ap.add_argument("--config", default="c2", choices=["c2", "c3i", "c3ii"],
                    help="c2 = BASELINE config 2 (the bench line); c3i / c3ii = config 3: BearingsOnly bootstrap / 4-D "
                         "MvNormal guided filter, N = 1e6, stratified")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--resampling-mode", default="island", choices=["island", "global"],
                    help="N > 1 GPUs: per-shard resampling with mass carry (default) or one exact global "
                         "resampling with ancestors pulled over NVLink")
    ap.add_argument("--essrmin", type=float, default=0.5,
                    help="0.5 = BASELINE config 2; 1.0 = resample at every step (stress case)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the timed filter computed in its last step to DIR/*.npy "
                         "(float64; more than %d particles: a fixed seeded sample; rank 0's shard on N > 1 GPUs)"
                         % DUMP_SAMPLE)
    args = ap.parse_args()
    global ESSRMIN
    ESSRMIN = args.essrmin
    if args.n is None:
        args.n = N_PER_GPU if args.config == "c2" else 1_000_000
    if args.steps is None:
        args.steps = 4 if args.impl == "reference" else 1000 if args.config == "c2" else 500
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU filter (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
