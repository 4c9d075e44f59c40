#!/usr/bin/env python
"""bench.py -- Viterbi GCUPS (query_L x sum(target_L) / s) of the B200 hot path.

Headline workload (`value`, BASELINE.json configs[1], the one the metric is quoted on at one GPU): a synthetic query
profile L=400 against 100,000 synthetic profile HMMs per GPU (lengths lognormal, median 200, clipped [30,2000]),
Viterbi only: forward pass + backtrace + Hit.score of every target, then the top-500 hit records.  With N GPUs the
ranks hold the N length-balanced shards (shard.balanced_shards) of ONE seeded database of N x 100k targets -- the
database shards by target, there is no data-path collective -- and exchange their top-K records with one
ncclAllGather per step INSIDE the library (hhg_plan_topk; no torch.topk / torch.distributed on the data path).

    python bench.py --gpus N --steps K --warmup W            (driver; torchrun for N > 1)
    python bench.py --impl reference ...                      (the reference's AVX2 Viterbi on the host cores)
    python bench.py --no-extras                               (skip the configs[2..4] sections)
    python bench.py --dump-outputs bench_outputs              (also write the last timed step's results as .npy)

value  : whole-job GCUPS, database resident in HBM, device-timed (CUDA events, max over ranks)
e2e    : the same through the host-buffer C-ABI calls (hhg_query_set + hhg_viterbi_search + hhg_plan_topk): per step
         the query profile and the target-id list go H2D from pinned memory, hits and paths come back D2H.
roofline : algorithmic bytes (112 B per target column + 1 B per DP cell + 40 B per hit) / forward-kernel time against
         the measured HBM peak (frac = frac_hbm), and the issue-slot fraction (frac_issue) that actually binds.
verified : number of hits of the TIMED run compared with the C oracle (score bits, end points, path) in here.
cpu_baseline / --impl reference : the reference's own Viterbi::Align + Backtrace (oracle/_ref, AVX2) on a bounded
         sample drawn from the SAME rank-0 shard, threads = min(affinity, cgroup quota), OMP_PROC_BIND=close.
configs : the other north_star configurations, each with per-stage ms:
         N = 1: configs[2] (1M HMMs, prefilter + Viterbi, one GPU) and configs[4] on one GPU (Lq=1500, full scan);
         N > 1: configs[3] (1M sharded N ways, prefilter -> Viterbi on survivors -> NCCL top-K) and configs[4].
"""
from __future__ import annotations

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

TOPK = 500          # realign_max of the reference (src/hhdecl.cpp): records exchanged per rank
BASE_SEED = 1000
# instructions per 32-cell row visit of k_viterbi<16,local> (ncu smsp__inst_executed / row visits, profiles/r2_*)
WARP_INSTR_PER_ROW_VISIT = 105.7


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--targets", type=int, default=100000, help="targets per GPU of the headline workload")
    ap.add_argument("--total-targets", type=int, default=1000000, help="database size of configs[2..4]")
    ap.add_argument("--lq", type=int, default=400)
    ap.add_argument("--cpu-sample", type=int, default=4000, help="targets in the cpu_baseline sample")
    ap.add_argument("--ref-sample", type=int, default=8000, help="targets per step of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2..4] sections")
    ap.add_argument("--no-prefilter", action="store_true", help="(kept for old command lines; same as --no-extras)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------------------------- host facts
def host_threads():
    """Threads the CPU arm may use: min(sched affinity, cgroup cpu.max quota); plus what the box has."""
    logical = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = logical
    quota = None
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(p).read().split()
            if p.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    quota = q / per
            break
        except Exception:
            continue
    physical = None
    try:
        out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=5).stdout
        kv = {ln.split(":")[0].strip(): ln.split(":", 1)[1].strip() for ln in out.splitlines() if ":" in ln}
        physical = int(kv["Socket(s)"]) * int(kv["Core(s) per socket"])
        model = kv.get("Model name")
    except Exception:
        model = None
    used = max(1, min(aff, int(quota) if quota else aff, physical or aff))
    try:
        load1 = float(open("/proc/loadavg").read().split()[0])
    except Exception:
        load1 = None
    return dict(logical=logical, physical=physical, affinity=aff, cgroup_cpus=quota, used=used, model=model, loadavg1=load1)


def headline_lengths(args, world):
    """Lengths of the ONE seeded database of the headline workload (world x targets-per-GPU targets) and its shards."""
    from hhsuite_b200 import synth, shard
    rng = np.random.default_rng(BASE_SEED)
    Lg = synth.lengths(args.targets * world, rng)
    parts = shard.balanced_shards(Lg, world) if world > 1 else [np.arange(len(Lg), dtype=np.int32)]
    return Lg, parts


def headline_shard(args, rank, world):
    """(query, rank's shard as a synth.prepared_db dict, global ids of the shard)."""
    from hhsuite_b200 import synth
    qp, qtr, qss, qpav, qcols = synth.query_profile(args.lq, seed=1)
    Lg, parts = headline_lengths(args, world)
    ids = parts[rank]
    db = synth.prepared_db(len(ids), seed=BASE_SEED + 1 + rank, query_cols=qcols, planted=64, lens=Lg[ids], fast=True)
    return (qp, qtr, qss, qpav, qcols), db, ids


def workload_config(args, world, n_rank, sum_l_rank):
    return {"workload": f"query L={args.lq} vs {args.targets} synthetic profile HMMs per GPU (one seeded database of "
                        f"{args.targets * world} targets, lognormal lengths, median 200, clip [30,2000], "
                        f"length-balanced shards), Viterbi only: forward pass + backtrace + Hit.score of every target, "
                        f"top-{TOPK} hit records" + (" merged over NCCL inside the library" if world > 1 else ""),
            "targets_per_gpu": int(args.targets), "query_L": int(args.lq), "parallelism": f"db-shard x{world}",
            "l2": "inputs larger than L2 (2.5 GB of column records + 9 GB of backtrace bytes per step)",
            "strip_rows": 16, "db_resident": True}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def captured_traffic(key):
    """dram__bytes_read+write per launch of the dominant kernel from the committed ncu capture of this workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(key)
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).
    NVML in a thread (5 ms period) is the sampler; if NVML cannot be loaded, `nvidia-smi -lms 20` is, and start()
    then waits for its first line (a fresh box can take seconds to deliver it -- longer than the timed region)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NVML_REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
                    ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.nvml = None
        self.samples = []          # (time, sm_mhz, max_mhz, set(reasons))
        self.stop_flag = False
        self.source = None

    def _nvml_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.idx < len(ids) and ids[self.idx].isdigit():
                return int(ids[self.idx])
        return self.idx

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self._sample_nvml()                      # fail here, not in the thread
            self.source = "nvml"
            self.t = threading.Thread(target=self._loop_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
            self.samples = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self._nvml_index())],
                                         stdout=subprocess.PIPE, text=True)
            self.source = "nvidia-smi"
            self.t = threading.Thread(target=self._loop_smi, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.samples and time.time() - t0 < 20.0 and self.proc.poll() is None:
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _sample_nvml(self):
        nv = self.nvml
        sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        self.samples.append((time.time(), sm, self.max_mhz, {n for n, bit in self.NVML_REASONS if mask & bit}))

    def _loop_nvml(self):
        while not self.stop_flag:
            try:
                self._sample_nvml()
            except Exception:
                pass
            time.sleep(0.005)

    def _loop_smi(self):
        for ln in self.proc.stdout:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm = float(f[1]); mx = float(f[2])
            except ValueError:
                continue
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.samples.append((time.time(), sm, mx, {n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")}))

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML and no nvidia-smi"], "samples": 0}
        if self.nvml:
            self.t.join(timeout=1)
        t0 = getattr(self, "t_begin", 0.0)
        t1 = getattr(self, "t_end", float("inf"))
        inside = [s for s in self.samples if t0 <= s[0] <= t1 + 0.02]
        use = inside or self.samples[-3:]            # a very short region may fall between two samples
        sm = [s[1] for s in use]
        reasons = set().union(*[s[3] for s in use]) if use else set()
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": use[-1][2] if use else None,
                "reasons": sorted(reasons), "samples": len(inside), "source": self.source}


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_baseline(args, qprof, db, sample, host=None):
    """Reference AVX2 Viterbi::Align + Backtrace (src/hhviterbirunner.cpp:117-128 batching) on the first `sample`
    targets of the shard.  Threads = what the container may really use (cgroup quota / affinity / physical cores),
    pinned close; best of 3 passes; the host's load average is recorded next to the number."""
    host = host or host_threads()
    threads = host["used"]
    qp, qtr, qss, qpav = qprof[:4]
    n = min(sample, len(db["L"]))
    sub = dict(L=db["L"][:n], p=db["p"], tr=db["tr"], p_off=db["p_off"][:n], tr_off=db["tr_off"][:n])
    sample_txt = (f"first {n} targets of the rank-0 shard of the workload in `config` (sum L={int(sub['L'].sum())}; the "
                  f"figure is per cell, i.e. scaled), Viterbi::Align+Backtrace only, AVX2 no-FMA build of the unmodified "
                  f"reference, OpenMP dynamic over 8-target batches, {threads} threads (container quota "
                  f"{host['cgroup_cpus']}, affinity {host['affinity']}, {host['physical']} physical / {host['logical']} "
                  f"logical CPUs, {host['model']}), OMP_PROC_BIND=close OMP_PLACES=cores, loadavg {host['loadavg1']}")
    try:
        from oracle.binding import RefShim
        R = RefShim(nocontxt=True, maxres=max(4096, int(db["L"].max()) + 8))
        R.set_query(qp, qtr, qpav, None)
        R.viterbi_bench(dict(sub, L=sub["L"][:64], p_off=sub["p_off"][:64], tr_off=sub["tr_off"][:64]), threads)  # warm
        runs = [R.viterbi_bench(sub, threads, with_backtrace=True, repeats=1)[:2] for _ in range(3)]
        sec, cells = min(runs, key=lambda x: x[0])
        return dict(value=cells / sec / 1e9, unit="GCUPS", cores=threads, kind="reference", sample=sample_txt,
                    seconds=sec, spread=[round(c / s / 1e9, 3) for s, c in runs])
    except (FileNotFoundError, OSError):
        from oracle.binding import Oracle
        O = Oracle()
        n = min(n, 200)
        t0 = time.time()
        cells = 0
        for k in range(n):
            L = int(db["L"][k])
            tp = db["p"][db["p_off"][k]:db["p_off"][k] + L + 2]
            ttr = db["tr"][db["tr_off"][k]:db["tr_off"][k] + L + 1]
            O.viterbi(qp, qtr, tp, ttr)
            cells += args.lq * L
        sec = time.time() - t0
        return dict(value=cells / sec / 1e9, unit="GCUPS", cores=1, kind="port",
                    sample=f"first {n} targets, scalar C restatement (oracle/hh_oracle.c), 1 thread", seconds=sec)


def run_reference(args, host):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # the same rank-0 shard our arm measures (same seed, same lengths); only its first ref_sample targets are timed
    qprof, db, ids = headline_shard(args, 0, world)
    times = []
    cb = None
    for s in range(args.warmup + args.steps):
        cb = cpu_baseline(args, qprof, db, args.ref_sample, host)
        if s >= args.warmup:
            times.append(cb["seconds"])
    n = min(args.ref_sample, len(db["L"]))
    cells = float(args.lq) * float(db["L"][:n].sum())
    t = float(np.mean(times))
    val = cells / t / 1e9
    cb = dict(cb, value=val)
    cb.pop("seconds", None)
    args.emit({
        "impl": "reference", "metric": "Viterbi GCUPS (query_L x sum target_L / s)", "value": val, "unit": "GCUPS",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, len(db["L"]), int(db["L"].sum())),
        "cpu_baseline": cb, "host": host,
        "e2e": {"value": val, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })
    return 0


# ----------------------------------------------------------------------------------------------- verification
def verify_sample(hh, qprof, db_h, hits, paths, k=16, seed=7):
    """Compare k random hits of the timed run with the C oracle: score bits, end points, path states."""
    from oracle.binding import Oracle
    O = Oracle()
    qp, qtr = qprof[0], qprof[1]
    rng = np.random.default_rng(seed)
    n = len(hits)
    pick = list(range(min(4, n))) + rng.choice(n, size=min(k, n), replace=False).tolist()   # planted homologs + random
    ok = 0
    for t in pick:
        L = int(db_h["L"][t])
        tp = db_h["p"][db_h["p_off"][t]:db_h["p_off"][t] + L + 2]
        ttr = db_h["tr"][db_h["tr_off"][t]:db_h["tr_off"][t] + L + 1]
        sc, i2, j2, bt = O.viterbi(qp, qtr, tp, ttr)
        h = hits[t]
        if np.float32(sc).view(np.uint32) != h["score"].view(np.uint32) or (i2, j2) != (int(h["i2"]), int(h["j2"])):
            raise SystemExit(f"bench verification FAILED: target {t}: oracle {sc} ({i2},{j2}) vs GPU {h['score']} "
                             f"({h['i2']},{h['j2']})")
        ns, i_s, j_s, st, mc = O.backtrace(bt, i2, j2)
        if ns != int(h["nsteps"]) or not np.array_equal(paths[int(h["path_off"]):int(h["path_off"]) + ns], st[1:]):
            raise SystemExit(f"bench verification FAILED: target {t}: path differs from the oracle's")
        ok += 1
    return ok


def dump_outputs(d, merged, hits, paths, n_paths=1024, seed=11):
    """The results of the last timed step as float64 .npy files, so that two builds can be compared output for output:
    the merged top-K records (topk_*), every target's hit record (hits_*) and the backtrace paths of a fixed, seeded
    sample of targets (path_targets, path_len, path_states: the states of the sampled paths, concatenated).
    With several GPUs the hit records and paths are rank 0's shard.  About 7 MB at the headline size, mostly the
    100,000 hit records."""
    os.makedirs(d, exist_ok=True)
    f64 = lambda a: np.ascontiguousarray(a, np.float64)  # noqa: E731  (exact for the int32 and float32 fields)
    np.save(os.path.join(d, "topk_target.npy"), f64(merged["target"]))
    for f in merged.dtype["hit"].names:
        if f != "path_off":              # an offset into the library's own path buffer, not a result
            np.save(os.path.join(d, f"topk_{f}.npy"), f64(merged["hit"][f]))
    for f in hits.dtype.names:
        if f != "path_off":
            np.save(os.path.join(d, f"hits_{f}.npy"), f64(hits[f]))
    pick = np.sort(np.random.default_rng(seed).choice(len(hits), min(n_paths, len(hits)), replace=False))
    ns = hits["nsteps"][pick].astype(np.int64)
    st = [paths[int(o):int(o) + int(k)] for o, k in zip(hits["path_off"][pick], ns)]
    np.save(os.path.join(d, "path_targets.npy"), f64(pick))
    np.save(os.path.join(d, "path_len.npy"), f64(ns))
    np.save(os.path.join(d, "path_states.npy"), f64(np.concatenate(st) if st else np.zeros(0)))


# ----------------------------------------------------------------------------------------------- extras
def subset_db(base, idx):
    """prepared_db dict holding base targets idx[0], idx[1], ... (repeats allowed)."""
    idx = np.asarray(idx, np.int64)
    L = base["L"][idx].astype(np.int64)

    def gather(arr, off, rows):
        starts = off[idx]
        tot = int(rows.sum())
        out_off = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
        pos = np.arange(tot, dtype=np.int64) - np.repeat(out_off, rows) + np.repeat(starts, rows)
        return arr[pos], out_off
    P, p_off = gather(base["p"], base["p_off"], L + 2)
    T, tr_off = gather(base["tr"], base["tr_off"], L + 1)
    return dict(L=L.astype(np.int32), p=P, tr=T, p_off=p_off, tr_off=tr_off)


def extras(args, hh, ctx, comm, rank, world, dev, qprof, base, dist):
    """configs[2] / configs[3] (1M HMMs, two-stage prefilter -> Viterbi on the survivors -> top-K) and configs[4]
    (Lq=1500, Viterbi over the whole database), the database = the 100k rank-0 base repeated to --total-targets and
    sharded N ways by shard.balanced_shards.  Returns a dict of per-stage times."""
    import torch
    from hhsuite_b200 import synth, shard, prefilter as pf
    out = {}
    nt = args.total_targets
    nb = len(base["L"])
    Lg = base["L"][np.arange(nt) % nb]
    parts = shard.balanced_shards(Lg, world) if world > 1 else [np.arange(nt, dtype=np.int32)]
    mine = parts[rank]
    t0 = time.perf_counter()
    sub = subset_db(base, mine % nb)
    db = hh.TargetDB(ctx, sub["L"], sub["p"], sub["tr"], sub["p_off"], sub["tr_off"])
    n_loc = len(mine)
    qp, qtr, qss, qpav, qcols = qprof
    # cs219 shard: random column states + planted noisy copies of the query's best states (so stage 2 has survivors)
    G = np.load(os.path.join(ROOT, "tests", "golden", "golden_v1.npz"))
    lib219 = G["cs219_lin"]
    prof = hh.capi.build_prefilter_profile(qp, qpav, lib219, 50, 4)
    cs = synth.cs219_db(n_loc, seed=3 + rank, lens=sub["L"])
    best = prof[:219].argmax(axis=0).astype(np.uint8)
    rng = np.random.default_rng(5 + rank)
    planted = rng.choice(n_loc, max(1, 3000 // world), replace=False)
    for t in planted:
        Lt = int(sub["L"][t]); o = int(cs["off"][t])
        a = int(rng.integers(0, max(1, args.lq - Lt + 1))) if Lt < args.lq else 0
        seg = best[a:a + Lt].copy()
        noise = rng.random(len(seg)) < 0.25
        seg[noise] = rng.integers(0, 219, int(noise.sum()), dtype=np.uint8)
        cs["seq"][o:o + len(seg)] = seg
    csdb = hh.CsDB(ctx, cs["L"], cs["off"], cs["seq"])
    setup_s = time.perf_counter() - t0
    sumL_glob = float(Lg.astype(np.int64).sum())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---- configs[2] / configs[3]: prefilter -> Viterbi(survivors) -> top-K
    def query_once():
        tm = {}
        t = time.perf_counter()
        if world == 1:
            ids = pf.prefilter_db(csdb, prof)
        else:
            def s1():
                csdb.run(prof, 50)
                return csdb.select(args.lq, 4, 10, 100)
            gl = shard.sharded_prefilter(s1, lambda li: csdb.sw(prof, ids=li, gap_open=24, gap_extend=4, bias=50),
                                         mine, sub["L"], nt, args.lq, device=dev)
            x = np.searchsorted(mine, gl)                        # survivors this rank owns (mine is id-sorted)
            x[x >= n_loc] = 0
            ids = x[mine[x] == gl].astype(np.int32)
        tm["prefilter_ms"] = (time.perf_counter() - t) * 1e3
        t = time.perf_counter()
        ctx.set_query(qp, qtr)
        if len(ids):
            hits, paths = hh.viterbi_search(ctx, db, ids=ids)
            lp = ctx.L.hhg_ctx_last_plan(ctx.h)
            top = hh.capi.plan_topk(ctx, lp, comm, TOPK, True, 0, mine[ids])
        else:                                   # a rank without survivors still joins the collective
            hits = np.zeros(0, hh.capi.HIT_DTYPE)
            ids1 = np.zeros(1, np.int32)
            hh.viterbi_search(ctx, db, ids=ids1)
            top = hh.capi.plan_topk(ctx, ctx.L.hhg_ctx_last_plan(ctx.h), comm, TOPK, True, 0, mine[ids1])
        tm["viterbi_topk_ms"] = (time.perf_counter() - t) * 1e3
        return tm, ids, top

    query_once()
    sync_all()
    best_t = None
    for _ in range(3):
        sync_all()
        t = time.perf_counter()
        tm, ids, top = query_once()
        torch.cuda.synchronize()
        tot = (time.perf_counter() - t) * 1e3
        tt = torch.tensor([tot, tm["prefilter_ms"], tm["viterbi_topk_ms"], float(len(ids)),
                           float(args.lq) * float(sub["L"][ids].sum()) if len(ids) else 0.0], device=dev, dtype=torch.float64)
        if world > 1:
            mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = tt.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            tt = torch.stack([mx[0], mx[1], mx[2], sm[3], sm[4]])
        tt = tt.cpu().numpy()
        if best_t is None or tt[0] < best_t[0]:
            best_t = tt
    name = "configs[2]" if world == 1 else "configs[3]"
    out[name] = {"workload": f"query L={args.lq} vs {nt} synthetic HMMs on {world} GPU(s), two-stage cs219 prefilter "
                             f"(ungapped over the whole shard, gapped byte SW over the stage-1 list, reference selection "
                             f"rules with the GLOBAL database size) -> Viterbi + backtrace + Hit.score on the survivors -> "
                             f"top-{TOPK}" + (" over NCCL" if world > 1 else ""),
                 "ms_per_query": float(best_t[0]), "prefilter_ms": float(best_t[1]), "viterbi_topk_ms": float(best_t[2]),
                 "survivors": int(best_t[3]), "viterbi_gcups_on_survivors": float(best_t[4] / (best_t[2] * 1e-3) / 1e9),
                 "prefilter_tcells_per_s": float(args.lq * sumL_glob / (best_t[1] * 1e-3) / 1e12),
                 "effective_gcups_whole_db": float(args.lq * sumL_glob / (best_t[0] * 1e-3) / 1e9),
                 "timing": "wall clock per query on the host (max over ranks), copies and host selection logic included, "
                           "best of 3", "setup_s": round(setup_s, 1),
                 "limiter": "prefilter stage 1 (integer-issue bound DPX kernel over the whole shard) + host-side "
                            "selection/plan latency; the survivor Viterbi is a small batch"}
    csdb.close()

    # ---- configs[4]: Lq=1500, Viterbi over the whole (sharded) database
    q5 = synth.query_profile(1500, seed=2)
    ctx.set_query(q5[0], q5[1])
    plan = hh.Plan(ctx, db)
    plan.run(); plan.topk(TOPK, comm=comm, by_hit_score=True, global_ids=mine)
    sync_all()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    nrep = 2
    for _ in range(nrep):
        plan.run()
        top = plan.topk(TOPK, comm=comm, by_hit_score=True, global_ids=mine)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / nrep], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    cells5 = 1500.0 * sumL_glob
    out["configs[4]"] = {"workload": f"query L=1500 (94 strips) vs {nt} synthetic HMMs sharded over {world} GPU(s), Viterbi "
                                     f"over the whole database + top-{TOPK}" + (" over NCCL" if world > 1 else ""),
                         "ms_per_query": float(ms.item()), "gcups": float(cells5 / (ms.item() * 1e-3) / 1e9),
                         "timing": "CUDA events on the launching stream, max over ranks, database resident",
                         "limiter": "FP32 issue rate of the forward kernel (same kernel as the headline)"}
    plan.close(); db.close()
    if world == 1:
        # database load straight from A3M alignments (SURVEY 8f-1): filter, sequence weights, frequencies, transitions
        # and pseudocounts of every alignment in CUDA kernels; wall clock incl. the host scan of the text
        lens = np.clip(np.round(np.exp(rng.normal(np.log(200), 0.5, 16))), 30, 600).astype(int)
        nseq = np.clip(np.round(np.exp(rng.normal(np.log(100), 0.7, 16))), 5, 800).astype(int)
        uniq = [synth.a3m_text(int(L_), int(N_), 700 + k, f"b{k}").encode() for k, (L_, N_) in enumerate(zip(lens, nseq))]
        pick = rng.integers(0, len(uniq), 1000)
        texts = [uniq[i] for i in pick]
        data = b"".join(t + b"\0" for t in texts)
        ln = np.array([len(t) + 1 for t in texts], np.int64)
        off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64)
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            adb = hh.TargetDB.from_a3m(ctx, data, off, ln, G["R"], G["pb"])
            dt = time.perf_counter() - t0
            cols = int(adb.Lh.sum())
            adb.close()
            best = dt if best is None else min(best, dt)
        res = int(sum(int(lens[i]) * int(nseq[i] + 1) for i in pick))
        out["loader_a3m"] = {"workload": "1000 synthetic A3M alignments (16 distinct; median 200 columns x 100 sequences) -> resident "
                                         "shard: identity filter, sequence weights, frequencies, transitions, pseudocounts",
                             "alignments_per_s": float(len(texts) / best), "aligned_residues_per_s": float(res / best),
                             "columns": cols, "text_MB": len(data) / 1e6, "seconds": best,
                             "timing": "wall clock of hhg_db_create_a3m incl. the host scan, best of 3"}
    return out


# ----------------------------------------------------------------------------------------------- main
def main():
    args = parse_args()
    # stdout carries exactly ONE line, the JSON record: anything a library prints there (NCCL's version banner, ...)
    # goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())
    args.emit = emit
    if args.no_prefilter:
        args.no_extras = True
    host = host_threads()
    if args.impl == "reference":
        # pin the reference's OpenMP team; must be in the environment before libgomp is loaded by the reference shim.
        # Only for this arm: with OMP_PROC_BIND set libgomp also pins the INITIAL thread of every process that loads it
        # (torch does), which would put the host threads of all ranks of a multi-GPU run on the same core.
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
    if args.impl == "reference":
        return run_reference(args, host)

    import torch
    import torch.distributed as dist
    import hhsuite_b200 as hh

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    qprof, db_h, gids = headline_shard(args, rank, world)
    qp, qtr, qss, qpav, qcols = qprof
    # a dedicated (non-default) torch stream: the library launches on it and torch.cuda.Event brackets it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = hh.Context(device=local_rank, stream=stream.cuda_stream)
    assert stream.cuda_stream != 0
    # the library's own communicator (NCCL inside libhhg.so); torch.distributed only carries the rendezvous id,
    # the barrier and the max-over-ranks of the timings
    comm = None
    if world > 1:
        box = [hh.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = hh.Comm(ctx, rank, world, box[0])
    ctx.set_query(qp, qtr)
    db = hh.TargetDB(ctx, db_h["L"], db_h["p"], db_h["tr"], db_h["p_off"], db_h["tr_off"])
    plan = hh.Plan(ctx, db)
    cells_rank = plan.cells
    n = plan.n

    def step():
        plan.run()
        return plan.topk(TOPK, comm=comm, by_hit_score=True, global_ids=gids)

    def timed_region(warm):
        sampler = ClockSampler(local_rank)
        sampler.start()                  # before the warm-up, so that samples exist when the timed region starts
        for _ in range(warm):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler.mark_begin()
        l0 = ctx.launches
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler.mark_end()
        return e0.elapsed_time(e1), sampler.stop(), ctx.launches - l0, out

    def bad_clocks(c):                   # the contract's rejection rule; sw_power_cap is kept and noted
        if {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]):
            return True
        return bool(c["sm_mhz"] and c["sm_max_mhz"] and c["sm_mhz"] < 0.85 * c["sm_max_mhz"] and not c["reasons"])

    el_ms, clocks, launches, merged = timed_region(max(args.warmup, 3))
    flag = torch.tensor([1.0 if bad_clocks(clocks) else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    if flag.item() > 0:                  # throttled or clock-locked run: rejected and measured once more
        first = clocks
        el_ms, clocks, launches, merged = timed_region(1)
        clocks["remeasured_after"] = first
    ms = torch.tensor([el_ms], device=dev, dtype=torch.float64)
    cells_all = torch.tensor([cells_rank], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(cells_all, op=dist.ReduceOp.SUM)
    ms_step = float(ms.item()) / args.steps
    total_cells = float(cells_all.item())
    gcups = total_cells / (ms_step * 1e-3) / 1e9

    # ---- the timed run's results against the oracle, and the merged list against this rank's own hits
    hits, paths = plan.fetch()
    verified = verify_sample(hh, qprof, db_h, hits, paths)
    own = merged[merged["owner"] == rank]
    pos = {int(g): k for k, g in enumerate(gids)}
    for r in own:
        h = hits[pos[int(r["target"])]]
        if r["hit"]["hit_score"].view(np.uint32) != h["hit_score"].view(np.uint32) or r["hit"]["nsteps"] != h["nsteps"]:
            raise SystemExit("bench verification FAILED: merged top-K record differs from the owner's hit")
    order = np.lexsort((gids, -hits["hit_score"].astype(np.float64)))[:TOPK]
    if world == 1 and not np.array_equal(merged["target"], gids[order]):
        raise SystemExit("bench verification FAILED: device top-K differs from the host sort")
    verified += len(own)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, merged, hits, paths)

    # ---- per-kernel roofline figure (forward kernel timed alone with CUDA events on the same stream)
    kt = [plan.run_timed() for _ in range(3)]
    ms_vit = float(np.mean([a for a, b in kt])); ms_bt = float(np.mean([b for a, b in kt]))
    peaks, peak_src = measured_peaks()
    ach = plan.alg_bytes / (ms_vit * 1e-3) / 1e9
    default_wl = (args.targets == 100000 and args.lq == 400)
    traffic = captured_traffic("k_viterbi_16_local_100k_lq400") if default_wl else None
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    row_visits = cells_rank / 32.0
    issue_cycles = row_visits * WARP_INSTR_PER_ROW_VISIT / (148 * 4)          # per SMSP at 1 warp-instruction / clock
    frac_issue = issue_cycles / (ms_vit * 1e-3 * sm_mhz * 1e6)
    roofline = {"bound": "issue", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "frac_hbm": ach / peaks["hbm_gbs"], "frac_issue": frac_issue,
                "traffic": traffic["bytes"] if traffic else None,
                "traffic_source": traffic["source"] if traffic else None,
                "traffic_over_algorithmic": (traffic["bytes"] / plan.alg_bytes) if traffic else None,
                "peak_source": peak_src, "kernel": "k_viterbi<16,local>", "kernel_ms": ms_vit, "backtrace_ms": ms_bt,
                "algorithmic_bytes_per_launch": plan.alg_bytes,
                "kernel_gcups": cells_rank / (ms_vit * 1e-3) / 1e9,
                "issue_model": f"{WARP_INSTR_PER_ROW_VISIT} warp instructions per 32-cell row visit (ncu) on 592 SMSPs at "
                               f"{sm_mhz:.0f} MHz (sampled); the ALU and FMA pipes each carry ~73 cycles of that",
                "note": "exact-fp32 max-plus recurrence: FP32-issue bound, not HBM bound (DESIGN.md 4.1, SURVEY 8d); frac "
                        "is the algorithmic-bytes fraction of the measured HBM peak as the contract asks, frac_issue is "
                        "the fraction of the issue-slot ceiling"}

    # ---- end to end through the host-buffer C-ABI call, pinned host buffers
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()  # noqa: E731
    qp_pin, qtr_pin = pin(qp), pin(qtr)
    ids_pin = pin(np.arange(n, dtype=np.int32))
    hits_pin = torch.empty(n * 40, dtype=torch.uint8).pin_memory().numpy().view(hh.capi.HIT_DTYPE)
    paths_pin = torch.empty(plan.path_cap, dtype=torch.uint8).pin_memory().numpy()
    h2d = qp_pin.nbytes + qtr_pin.nbytes + ids_pin.nbytes + gids.nbytes

    def e2e_step():
        ctx.set_query(qp_pin, qtr_pin)
        hts, pths = hh.viterbi_search(ctx, db, ids=ids_pin, hits=hits_pin, paths=paths_pin)
        return hh.capi.plan_topk(ctx, ctx.L.hhg_ctx_last_plan(ctx.h), comm, TOPK, True, 0, gids)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    d2h = hits_pin.nbytes + int(hits_pin["nsteps"].sum()) + TOPK * 56 * world
    if world > 1:
        dist.barrier()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    e2e_t = torch.tensor([(t1 - t0) / e2e_steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_gcups = total_cells / float(e2e_t.item()) / 1e9

    out = {
        "metric": "Viterbi GCUPS (query_L x sum target_L / s)", "value": gcups, "unit": "GCUPS", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, n, int(db_h["L"].sum())),
        "e2e": {"value": e2e_gcups, "unit": "GCUPS", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": float(e2e_t.item()) * 1e3,
                "note": "hhg_query_set + hhg_viterbi_search + hhg_plan_topk with pinned host buffers (plan reused across "
                        "queries, paths compacted on the device before D2H); the target DB stays resident on the GPU "
                        "(loaded once, like the reference's mmap'd ffindex DB)"},
        "gpu_launches": int(launches),
        "verified": int(verified),
        "clocks": clocks,
        "roofline": roofline,
        "sum_target_L_this_rank": int(db_h["L"].sum()),
    }
    if not args.no_extras:
        out["configs"] = extras(args, hh, ctx, comm, rank, world, dev, qprof, db_h if rank == 0 and world == 1 else
                                headline_shard(args, 0, 1)[1], dist)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the CPU figure comes from the reference arm itself, run as a child process on a bounded sample of the same
        # shard (own environment: OpenMP pinning must be set before libgomp loads, and must not leak into this process)
        env = dict(os.environ, RANK="0", WORLD_SIZE="1")
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "1",
                            "--ref-sample", str(args.cpu_sample), "--targets", str(args.targets), "--lq", str(args.lq)],
                           capture_output=True, text=True, env=env, timeout=600)
        try:
            ref = json.loads(r.stdout.strip().splitlines()[-1])
            out["cpu_baseline"] = ref["cpu_baseline"]
            out["host"] = ref["host"]
        except Exception:
            out["cpu_baseline"] = {"value": None, "unit": "GCUPS", "cores": host["used"], "kind": "reference",
                                   "sample": "reference arm failed: " + (r.stderr or r.stdout)[-300:]}
    if rank == 0:
        args.emit(out)
    plan.close(); db.close()
    if comm is not None:
        comm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
