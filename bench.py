#!/usr/bin/env python
"""bench.py -- unique-reads/s through the dada() core (BASELINE.json metric) on N B200s.

A "step" is one dada_uniques()-equivalent pass over one batch of synthetic dereplicated reads.

Workload (the configuration BASELINE.json's targets are quoted on): 1e6 synthetic 250 nt uniques (Zipf abundances, 100
true variants, Illumina-like qualities, seed 12345), tperr1 error matrix, default options, one dada() pass
(selfConsist=FALSE; the selfConsist loop of configs[2] is the separate "selfconsist" leg).  BASELINE configs[1]
(1e5 uniques) is reported as the secondary "configs1" object at N = 1.

  value  : uniques/s with the packed uniques already resident in HBM (Resident.run)
  e2e    : uniques/s through the C-ABI on HOST buffers: N = 1: the one-shot dada2b_run() (pack + H2D + loop + D2H of every
           output inside the timed region); N > 1: dada2b_reupload() + dada2b_run_resident() on every rank
  N > 1  : one process per GPU (torchrun); the SAME 1e6 sample sharded over the ranks (raw r on rank r % N) -- BASELINE
           configs[3] -- "strong" scaling
  parity : at every N, rank 0 runs the reference's own C++ on the same sample once and diffs the full output; a mismatch
           makes the run exit non-zero
  --impl reference : the reference's own C++ (oracle/_ref, compiled unmodified from /root/reference/src in the build
           container) on the host cores, same workload, full size.  Threads = the CPUs this process may really use (affinity
           mask capped by the cgroup CPU quota, host_cpus(): the GPU boxes expose 128 hardware threads under a 16-CPU quota,
           where 16 threads beat 128: 35 s against 41 s per 1e6 pass).
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

NUNIQ_DEFAULT = 1000000
WORKLOAD = ("BASELINE configs[2]/[3] size: %d synthetic 250 nt uniques in ONE sample (100 variants, Zipf abundances, Illumina-like quals, seed 12345), "
            "tperr1, dada() default options, one pass (selfConsist=FALSE)")


def workload(n_uniques, seed):
    from tools import synth
    from tests import cases
    seqs, ab, q, truth = synth.illumina(n_uniques, seed=seed)
    return seqs, ab, q, cases.tperr1()


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons during the timed region through NVML (in-process: a polling
    `nvidia-smi -lms` child was observed to stall the stream synchronisations of this latency-bound loop
    for hundreds of ms at a time).  Falls back to one nvidia-smi query per second."""

    def __init__(self, index, period=2.0):      # NVML queries contend with CUDA API calls for driver locks (profiles/r2_host_stalls.md): sample sparsely
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.rows = []          # (sm_mhz, max_mhz, reasons set)
        self.stop_flag = False

    def run(self):
        if os.environ.get("DADA2B_BENCH_NOCLOCKS"):
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            while not self.stop_flag:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                except Exception:
                    r = 0
                self.rows.append((float(sm), float(mx), {k for k, bit in names.items() if r & bit}))
                time.sleep(self.period)
            return
        except Exception:
            pass
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip().split(",")
                reasons = {n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6])
                           if v.strip().lower().startswith("active")}
                self.rows.append((float(out[0]), float(out[1]), reasons))
            except Exception:
                pass
            time.sleep(1.0)

    def finish(self):
        self.stop_flag = True
        rows = list(self.rows)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = set()
        for r in rows:
            reasons |= r[2]
        return {"sm_mhz": float(np.median([r[0] for r in rows])), "sm_max_mhz": float(max(r[1] for r in rows)),
                "reasons": sorted(reasons), "samples": len(rows)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _last_lines(txt, n=2, width=300):
    """The end of a failed leg's output: the exception line, not the middle of its traceback."""
    rows = [l.strip() for l in txt.strip().splitlines() if l.strip()]
    return " | ".join(rows[-n:])[-width:]


def subprocess_leg(tag, cmd, budget_s, device):
    """A post-measurement leg in its own process under a timeout (N = 1 only); prints one `<TAG> {json}` line.
    Reported under its own key; never part of `value` / `e2e`."""
    e = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(device)))
    try:
        out = subprocess.run(cmd, env=e, capture_output=True, text=True, timeout=budget_s)
        rows = [l for l in out.stdout.splitlines() if l.startswith(tag + " ")]
        return json.loads(rows[-1][len(tag) + 1:]) if rows else {"failed": _last_lines(out.stderr or out.stdout)}
    except subprocess.TimeoutExpired:
        return {"failed": "timeout"}
    except Exception as ex:
        return {"failed": repr(ex)[:200]}


def bimera_leg(budget_s, device, cmd=None):
    """SURVEY.md 8(f3)'s bimera detection timed through its C-ABI on a synthetic sequence table, next to the reference's
    C_table_bimera2 on the host cores."""
    return subprocess_leg("BIMLEG", cmd or [sys.executable, os.path.join(ROOT, "tools", "bimera_leg.py")], budget_s, device)


def host_cpus():
    """CPUs this process may really use: the affinity mask, capped by the cgroup's CPU quota (the GPU boxes show 128 hardware threads
    under `cpu.max = 1600000 100000`, i.e. 16 CPUs: 128 runnable threads there are stopped for 7/8 of every 100 ms period).
    DADA2B_REF_THREADS overrides."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    quota = float(f[0]) / float(f[1])
            else:
                per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if float(f[0]) > 0:
                    quota = float(f[0]) / per
            break
        except Exception:
            continue
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    if os.environ.get("DADA2B_REF_THREADS"):
        n = max(1, int(os.environ["DADA2B_REF_THREADS"]))
    return n


def cpu_reference(seqs, ab, err, q):
    """One pass of the reference's own C++ (or of the port when oracle/_ref is absent) on all host cores."""
    from oracle import ref
    ncores = host_cpus()
    if ref.available():
        ref.set_threads(ncores)
        cres = ref.dada_uniques(seqs, ab, None, err, q, multithread=True)
        return cres, ref.last_native_s, ncores, "reference"        # the native call alone: Python-side marshalling is not the reference's time
    from oracle import port
    t0 = time.perf_counter()
    cres = port.dada_uniques(seqs, ab, None, err, q)
    return cres, time.perf_counter() - t0, 1, "port"


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation, all host threads, the SAME full-size workload.  One step = one
    full pass.  The run is bounded in wall time (N = 1: ~23 min, N > 1: ~7 min, where the same CPU measurement would only
    be repeated): warm-up is cut to one pass first, then the number of timed passes -- never the size; `steps` is what ran."""
    if rank != 0:
        return
    from oracle import ref
    ncores = host_cpus()
    ref.set_threads(ncores)
    seqs, ab, q, err = workload(args.nuniques, 12345)
    budget = float(os.environ.get("DADA2B_REF_BUDGET_S", 1400 if world == 1 else 420))
    t_begin = time.perf_counter()
    warm = min(args.warmup, 1) if args.nuniques >= 500000 else args.warmup
    times = []
    it = 0
    while len(times) < args.steps:
        last = ref.dada_uniques(seqs, ab, None, err, q, multithread=True)
        dt = ref.last_native_s                   # the native call alone (ctypes marshalling of 1e6 Python strings is not the reference's time)
        if it >= warm:
            times.append(dt)
        it += 1
        if times and (time.perf_counter() - t_begin) + dt > budget:
            break
    if args.dump_outputs:
        dump_outputs(last, args.dump_outputs)
    tsum = sum(times)
    val = args.nuniques * len(times) / tsum
    line = {"impl": "reference", "metric": "unique-reads/sec through dada()", "value": val, "unit": "uniques/s",
            "n_gpus": args.gpus, "steps": len(times), "warmup": warm, "steps_requested": args.steps, "warmup_requested": args.warmup,
            "ms_per_step": 1e3 * tsum / len(times),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int16/int32 + f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD % args.nuniques},
            "cpu_baseline": {"value": val, "unit": "uniques/s", "cores": ncores, "kind": "reference", "hardware_threads": os.cpu_count(),
                             "sample": "the full %d-unique workload per step, multithread=TRUE on %d threads (parallelFor shim over a "
                                       "persistent std::thread pool); %d timed passes inside a %.0f s budget" % (args.nuniques, ncores, len(times), budget)},
            "e2e": {"value": val, "unit": "uniques/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def measure(res, err, steps, warmup, flush, barrier, torch):
    """`warmup` untimed + exactly `steps` timed resident passes -> (seconds, per-step ms, device ms sum, last result)."""
    last = None
    for _ in range(warmup):
        last = res.run(err)
        flush.zero_()
    barrier()
    t0 = time.perf_counter()
    dev_ms, step_ms, step_host = 0.0, [], []
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        ts = time.perf_counter()
        last = res.run(err)
        step_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
        step_host.append([round(last["stats"][k], 2) for k in ("ms_setup", "ms_loop", "ms_final")])
        dev_ms += last["stats"]["ms_device"]
    barrier()
    return time.perf_counter() - t0, step_ms, step_host, dev_ms, last


DUMP_LIMIT_BYTES = 64 << 20
PER_UNIQUE = ("map", "pval")


def dump_outputs(res, out_dir):
    """Writes the arrays of one dada_uniques() result as out_dir/<field>.npy (clustering.pval.npy, map.npy, ...), all float64
    and all finite: integers exactly, strings as rows of ASCII codes padded with 0.  A field with NaN or infinite entries
    (the birth fields of the first cluster, which is not born by a division, are NA) holds 0 there, and
    <field>.nonfinite.npy says which entries those are and what they were: 1 NaN, 2 +inf, 3 -inf, 0 elsewhere.  When the
    whole set would pass 64 MB, the per-unique fields keep a fixed seeded sample of the uniques, whose indices go to
    sample_idx.npy."""
    from tests import cases
    arrs = {}
    for k, v in cases.flatten(res).items():
        if v.dtype.kind == "U":
            b = v.astype("S")
            v = np.frombuffer(b.tobytes(), np.uint8).reshape(len(b), b.itemsize)
        v = v.astype(np.float64)
        bad = ~np.isfinite(v)
        if bad.any():
            arrs[k + ".nonfinite"] = np.where(np.isnan(v), 1.0, np.where(v == np.inf, 2.0, np.where(v == -np.inf, 3.0, 0.0)))
            v = np.where(bad, 0.0, v)
        arrs[k] = v
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_LIMIT_BYTES:
        nraw = len(arrs["map"])
        per_unique = [k for k in arrs if k.split(".nonfinite")[0] in PER_UNIQUE]
        rest = total - sum(arrs[k].nbytes for k in per_unique)
        keep = (DUMP_LIMIT_BYTES - rest) // (8 * (len(per_unique) + 1))
        idx = np.sort(np.random.default_rng(0).choice(nraw, keep, replace=False))
        for k in per_unique:
            arrs[k] = arrs[k][idx]
        arrs["sample_idx"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def selfconsist_loop(runner, n, native_s=None):
    """BASELINE configs[2]'s selfConsist error learning (R/dada.R:256-391; learnErrors) around `runner(err, max_clust)`:
    pass 0 with the all-ones matrix and MAX_CLUST = 1, then loessErrfun refits (dada2_b200/errmodel.py: a restatement of R's
    loess, parity unpinned) until the matrix repeats or MAX_CONSIST = 10.  Per-pass and whole-loop times."""
    from dada2_b200 import errmodel
    ms = []

    def timed(e, mc):
        t0 = time.perf_counter()
        r = runner(e, mc)
        dt = time.perf_counter() - t0
        if native_s is not None:                 # CPU arm: the native call alone, without the ctypes marshalling around it
            extra[0] += dt - native_s()
            dt = native_s()
        ms.append(round(dt * 1e3, 1))
        return r
    extra = [0.0]
    t0 = time.perf_counter()
    out = errmodel.learnErrors(timed)
    loop_s = time.perf_counter() - t0 - extra[0]
    return {"passes": out["passes"], "pass_ms": ms, "loop_ms": round(loop_s * 1e3, 1), "refit_ms_total": round(loop_s * 1e3 - sum(ms), 1),
            "uniques_per_s_whole_loop": n * out["passes"] / loop_s, "converged": out["passes"] < 11,
            "nclust_final": len(out["dada"]["clustering"]["sequence"])}, out


def configs1_leg(local_rank, flush, torch, do_cpu):
    """BASELINE configs[1] (1e5 uniques, one GPU) as a secondary object: value, e2e, parity against the CPU reference."""
    import dada2_b200
    from tests import cases
    n = 100000
    seqs, ab, q, err = workload(n, 12345)
    res = dada2_b200.Resident(seqs, ab, None, q, device=local_rank)

    def barrier():
        torch.cuda.synchronize()
    t_val, step_ms, _h, dev_ms, last = measure(res, err, 10, 3, flush, barrier, torch)
    sc_gpu, sc_out = selfconsist_loop(lambda e, mc: res.run(e, max_clust=mc), n)
    res.close()
    call = dada2_b200.PackedCall(seqs, ab, None, err, q)
    call.run(unpack=False)
    e2e_ms = []
    for _ in range(10):
        flush.zero_()
        torch.cuda.synchronize()
        _r, ms = call.run(unpack=False)
        e2e_ms.append(ms)
    st = last["stats"]
    out = {"workload": "BASELINE configs[1]: 100000 synthetic 250 nt uniques, 1 GPU, 10 timed steps after 3 warm-up",
           "value": n * 10 / t_val, "unit": "uniques/s", "ms_per_step": 1e3 * t_val / 10, "ms_per_step_median": float(np.median(step_ms)),
           "e2e": {"value": n / (float(np.mean(e2e_ms)) / 1e3), "ms_per_step": float(np.mean(e2e_ms)), "ms_per_step_median": float(np.median(e2e_ms))},
           "device_ms_per_step": dev_ms / 10, "gpu_launches_per_step": int(st["gpu_launches"]),
           "kernel_ms": {k: st[k] for k in st if k.startswith("ms_k_")}}
    if do_cpu:
        cres, dt, ncores, kind = cpu_reference(seqs, ab, err, q)
        out["cpu_baseline"] = {"value": n / dt, "unit": "uniques/s", "cores": ncores, "kind": kind, "sample": "all 100000 uniques, one pass, %.1f s" % dt}
        try:
            cases.assert_same(last, cres, rtol=1e-10, label="configs1")
            out["parity"] = "identical"
        except AssertionError as e:
            out["parity"] = "MISMATCH: %s" % str(e)[:300]
        # the same selfConsist loop around the reference's C++ on the host cores: same refit code, same number of passes expected
        from oracle import ref
        if ref.available():
            sc_cpu, sc_cpu_out = selfconsist_loop(lambda e, mc: ref.dada_uniques(seqs, ab, None, e, q, max_clust=mc, multithread=True), n,
                                                  native_s=lambda: ref.last_native_s)
            same = sc_cpu["passes"] == sc_gpu["passes"] and np.array_equal(sc_cpu_out["err_out"], sc_out["err_out"])
            try:
                cases.assert_same(sc_out["dada"], sc_cpu_out["dada"], rtol=1e-10, label="selfconsist")
            except AssertionError as e:
                same = "MISMATCH: %s" % str(e)[:200]
            sc_gpu["cpu_reference_loop"] = {"loop_ms": sc_cpu["loop_ms"], "pass_ms": sc_cpu["pass_ms"], "passes": sc_cpu["passes"]}
            sc_gpu["speedup_whole_loop"] = sc_cpu["loop_ms"] / sc_gpu["loop_ms"]
            sc_gpu["identical_to_cpu_loop"] = same
            if same is not True:
                out["parity"] = "MISMATCH (selfConsist loop): %s" % same
    out["selfconsist"] = sc_gpu
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nuniques", type=int, default=NUNIQ_DEFAULT)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU reference pass (no parity diff, no cpu_baseline)")
    ap.add_argument("--no-legs", action="store_true", help="N=1: skip the secondary legs (configs1, selfconsist, config5, bimera)")
    ap.add_argument("--bimera-seconds", type=int, default=60, help="N=1: timeout of the post-measurement bimera-detection leg (0 = off)")
    ap.add_argument("--watchdog", type=int, default=1700, help="dump stacks and exit after this many seconds")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step (rank 0) as DIR/<field>.npy; the seeded inputs are the same "
                         "in every run with the same arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    import faulthandler
    faulthandler.dump_traceback_later(args.watchdog, exit=True)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import datetime
    import torch
    import torch.distributed as dist
    import dada2_b200
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(minutes=30))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    shard = world > 1
    seqs, ab, q, err = workload(args.nuniques, 12345)                      # the same sample on every rank
    nraw = len(seqs)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # ---------------- value: inputs resident in HBM ----------------
    if shard:
        from dada2_b200 import multi
        res = multi.sharded_resident(seqs, ab, None, q, device=local_rank)
    else:
        res = dada2_b200.Resident(seqs, ab, None, q, device=local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()                      # NVML start-up takes ~1 s of driver calls: keep it out of the timed region
    res.run(err)
    t_wait = time.time()
    while not sampler.rows and time.time() - t_wait < (0 if os.environ.get("DADA2B_BENCH_NOCLOCKS") else 10):
        time.sleep(0.05)
    sampler.rows.clear()
    t_val, step_ms, step_host, dev_ms, last = measure(res, err, args.steps, max(0, args.warmup - 1), flush, barrier, torch)
    st = last["stats"]

    # ---------------- e2e: host buffers in, host buffers out, through the C-ABI ----------------
    e2e_ms = []
    est = None
    if shard:
        from dada2_b200 import _abi
        pin = _abi.PackedIn(seqs, ab, None, None, q)
        ecm = np.asfortranarray(np.asarray(err, dtype=np.float64))
        ostruct = _abi.make_opts(homo_gap=-8)
        for _ in range(max(1, args.warmup)):
            res.reupload(pin); res.run_raw(ecm, ecm.shape[1], ostruct)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            ts = time.perf_counter()
            res.reupload(pin)                                   # dada2b_reupload: pack + H2D of this rank's reads, all-gather of the packed reads
            est = res.run_raw(ecm, ecm.shape[1], ostruct)       # dada2b_run_resident: loop + D2H of every output
            e2e_ms.append(round((time.perf_counter() - ts) * 1e3, 2))
        barrier()
        t_e2e = time.perf_counter() - t0
        est = dict(est)
        L0 = len(seqs[0])
        nown = (nraw - rank + world - 1) // world
        # dada2b_reupload on a sharded context: packed reads and quality rows of this rank's raws only (the other ranks' packed reads
        # arrive over NVLink: one all-gather), plus lengths / abundances / priors of every raw
        est["h2d_bytes"] += nown * ((((L0 + 15) // 16 + 3) & ~3) * 4 + ((L0 + 15) & ~15)) + nraw * 7
    else:
        call = dada2_b200.PackedCall(seqs, ab, None, err, q)
        for _ in range(max(1, args.warmup)):
            call.run(unpack=False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            r, _ms = call.run(unpack=False)
            e2e_ms.append(round(_ms, 2))
            est = r["stats"]
        barrier()
        t_e2e = time.perf_counter() - t0
    clocks = sampler.finish()

    tt = torch.tensor([t_val, t_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_val, t_e2e = float(tt[0]), float(tt[1])
    value = nraw * args.steps / t_val               # the whole job denoises the ONE sample per step
    e2e = nraw * args.steps / t_e2e

    rc = 0
    if rank == 0:
        from tests import cases
        if args.dump_outputs:
            dump_outputs(last, args.dump_outputs)
        L = len(seqs[0])
        peak, peak_src = measured_peak_gbs()
        # ---- roofline of the dominant kernel family (CUDA-event sums per family, measured inside the library on its stream) ----
        bytes_per_pair = (L + 3) // 4 + 16 + L                      # SURVEY.md 8(d): S + O + Q for an aligned pair
        pairs = st["n_nw"]
        fam = {"nw (k_nwrow / k_nwlane / k_nwfwd: loop banded NW, bound + exact)": st["ms_k_align_nw"],
               "screen (k_prescreen + k_classify)": st["ms_k_classify"],
               "final pass (k_nwrow<FINAL> + k_align<FINAL>)": st["ms_k_align_final"],
               "round control (k_tail_* / k_shuffle_* / k_p_update / k_bud_*)": st.get("ms_k_tail", 0.0)}
        dominant = max(fam, key=fam.get)
        k_ms = st["ms_k_align_nw"]
        n_launch = max(1, st["n_k_align_nw"])
        achieved = (pairs * bytes_per_pair / 1e9) / (k_ms / 1e3) if k_ms > 0 else 0.0
        prof = {}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "r2_kernel_metrics.json")))
        except Exception:
            pass
        cells_pair = L * 33 - 16 * 17
        roofline = {"bound": "hbm", "kernel": "loop NW family (dd_nwrow.cu / dd_nwlane.cu): CUDA-event sum over its launches",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": prof.get("nw_dram_bytes_per_launch"),
                    "peak_source": peak_src, "algorithmic_bytes_per_pair": bytes_per_pair,
                    "algorithmic_bytes_per_launch": bytes_per_pair * pairs / n_launch, "pairs_per_step": int(pairs),
                    "kernel_ms_per_step": k_ms, "launches_per_step": int(n_launch), "avg_launch_ms": k_ms / n_launch,
                    "nw_gcups": (pairs * cells_pair / 1e9) / (k_ms / 1e3) if k_ms > 0 else 0.0,
                    "nw_bound_ms": st.get("ms_k_nw_bound"), "nw_exact_ms": st.get("ms_k_nw_exact"),
                    "kernel_share_of_device_time": k_ms / st["ms_device"] if st["ms_device"] else None,
                    "family_ms": fam, "dominant_family": dominant,
                    "issue_bound_evidence": prof.get("nw_large_round"),
                    "note": "integer DP: 7 978 cells per 329 algorithmic bytes, bound by integer issue (DESIGN.md 4.2), so the HBM fraction is low "
                            "by construction; the HBM-streaming kernel of the path is k_prescreen, reported in roofline_screen"}
        # the DRAM-streaming kernel: one 128-byte bitmap row + 13 bytes of metadata per (centre, active raw) pair
        ps_ms, ps_rows = st.get("ms_k_prescreen", 0.0), st.get("prescreen_rows", 0)
        ps_bytes = 141
        ps_ach = (ps_rows * ps_bytes / 1e9) / (ps_ms / 1e3) if ps_ms > 0 else 0.0
        roofline_screen = {"bound": "hbm", "kernel": "k_prescreen (TMA-staged 5-mer presence bitmaps; CUDA-event sum over its launches)",
                           "achieved": ps_ach, "peak": peak, "unit": "GB/s", "frac": ps_ach / peak,
                           "algorithmic_bytes_per_row": ps_bytes, "rows_per_step": int(ps_rows), "kernel_ms_per_step": ps_ms,
                           "launches_per_step": int(st.get("n_k_prescreen", 0)),
                           "avg_launch_ms": ps_ms / max(1, st.get("n_k_prescreen", 0)),
                           "traffic": prof.get("prescreen_dram_bytes_per_launch"),
                           "note": "rows of this rank only (1/N of the sample); launches shorter than ~10 us are launch-latency bound"}
        cpu, parity = None, None
        if not args.no_cpu_baseline:
            cres, dt, ncores, kind = cpu_reference(seqs, ab, err, q)
            cpu = {"value": nraw / dt, "unit": "uniques/s", "cores": ncores, "kind": kind, "hardware_threads": os.cpu_count(),
                   "sample": "all %d uniques of the step workload, one pass, %.1f s; threads = usable CPUs (cgroup quota)" % (nraw, dt)}
            try:
                cases.assert_same(last, cres, rtol=1e-10, label="bench")
                parity = "identical: full output of rank 0 equals the CPU reference on this workload (ints exact, fp64 <= 1e-10)"
            except AssertionError as e:
                parity = "MISMATCH: %s" % str(e)[:400]
                rc = 1
        legs = {}
        clean_env = not any(k.startswith("DADA2B_") and k not in ("DADA2B_VERBOSE", "DADA2B_BENCH_NOCLOCKS", "DADA2B_REF_BUDGET_S") for k in os.environ)
        if world == 1 and not args.no_legs and clean_env:
            try:
                legs["configs1"] = configs1_leg(local_rank, flush, torch, not args.no_cpu_baseline)
                if str(legs["configs1"].get("parity", "")).startswith("MISMATCH"):
                    rc = 1
            except Exception as ex:
                legs["configs1"] = {"failed": repr(ex)[:300]}
            try:       # BASELINE configs[2]: the whole selfConsist loop on the resident 1e6 uniques (one upload, <= 11 passes)
                legs["selfconsist"] = dict(selfconsist_loop(lambda e, mc: res.run(e, max_clust=mc), nraw)[0],
                                           workload="BASELINE configs[2]: learnErrors-style selfConsist loop on the resident %d uniques" % nraw)
            except Exception as ex:
                legs["selfconsist"] = {"failed": repr(ex)[:300]}
            legs["config5"] = subprocess_leg("C5LEG", [sys.executable, os.path.join(ROOT, "tools", "config5_leg.py")], 420, local_rank)
            if args.bimera_seconds > 0:
                legs["bimera"] = bimera_leg(args.bimera_seconds, local_rank)
        line = {"metric": "unique-reads/sec through dada()", "value": value, "unit": "uniques/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_val / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "int32 DP words (score|move|nsubs) + f64 lambda/p-value", "data": "synthetic",
                "config": {"workload": WORKLOAD % nraw,
                           "per_gpu": ("the ONE sample sharded over %d GPUs (strong scaling): raw r on rank r %% N, NCCL over NVLink per split round, "
                                       "final tallies all-reduced; every rank returns the full result" % world) if shard else "one GPU",
                           "l2": "256 MB buffer written between timed iterations (resident inputs at this size: 448 MB > 126 MB L2)",
                           "nclust": len(last["clustering"]["sequence"]), "rounds": st["n_rounds"], "shuffles": st["n_shuffles"],
                           "switches": sorted(k for k in os.environ if k.startswith("DADA2B_") and k not in ("DADA2B_VERBOSE",))},
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": "uniques/s", "h2d_bytes_per_step": int(est["h2d_bytes"]),
                        "d2h_bytes_per_step": int(est["d2h_bytes"]), "ms_per_step": 1e3 * t_e2e / args.steps,
                        "ms_per_step_median": float(np.median(e2e_ms))},
                "gpu_launches": int(st["gpu_launches"]) * args.steps,
                "parity": parity,
                "ms_per_step_median": float(np.median(step_ms)),
                "device_ms_per_step": dev_ms / args.steps,
                "step_ms": step_ms, "step_host_ms": step_host, "e2e_step_ms": e2e_ms,
                "kernel_ms": {k: st[k] for k in st if k.startswith("ms_k_")},
                "host_ms": {k: st[k] for k in ("ms_setup", "ms_loop", "ms_final", "ms_total")},
                "roofline": roofline, "roofline_screen": roofline_screen, "cpu_baseline": cpu}
        line.update(legs)
        print(json.dumps(line))
        sys.stdout.flush()
    res.close()
    if world > 1:
        flag = torch.tensor([rc], dtype=torch.int32, device=dev)
        dist.broadcast(flag, src=0)
        rc = int(flag[0])
        dist.destroy_process_group()
    if rc:
        sys.stderr.write("bench.py: parity MISMATCH against the CPU reference -- failing the run\n")
        sys.exit(1)


if __name__ == "__main__":
    main()
