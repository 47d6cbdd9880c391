#!/usr/bin/env python
"""bench.py -- distinct states/sec of the explicit-state BFS hot path (BASELINE.json metric).

A "step" is one complete breadth-first model-checking job of the workload model (every reachable state -- or, for a
state space that does not end, every state of the first L levels -- with the invariants checked on every expanded
state) on N GPUs.  Workloads (committed compiled fixtures, tests/golden/):

  MCPaxos3_b4 (default)  BASELINE config #3 scaled to a single-GPU-sized space: examples/Paxos, 3 acceptors / 2 values,
                         ballots 0..4, Inv1-Inv4 -- 352,133,865 distinct / 3,462,635,854 generated states, depth 41
  MCssi_4x3              BASELINE config #5 at its stated bound: serializableSnapshotIsolation.tla, 4 transactions x
                         3 keys, all eight invariants, deadlock ON; the space does not end (levels grow ~9x), the job
                         is its first 10 levels: 168,052,153 distinct states (>= 10^8, the size the metric is quoted on)
  MCraft_t4l3            BASELINE config #4 at its stated bound: raft.tla, 3 servers, MaxTerm 4, MaxLogLen 3 (message
                         bag bounded to 3 distinct messages: raft.tla:471 makes it infinite otherwise): 11,296,712 states

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--engine sliced|interp]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  Keys beyond the base contract: roofline (the wave kernels of the step), k1_roofline (the
fingerprint/probe kernel alone on SURVEY 8d's synthetic batch), cpu_baseline, e2e, clocks, gpu_launches,
other_workloads (configs #4 and #5 run once each next to the headline, counts and digests checked).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# depth bound of the workloads whose state space does not end (levels that exist when the job stops)
WORKLOAD_LEVELS = {"MCssi_4x3": 10}
# the CPU arm's bounded sample: a job of more than 2 x CPU_SAMPLE_STATES states is cut at the end of the level that
# reaches CPU_SAMPLE_STATES; depth-bounded workloads are cut one level earlier than the GPU job (SSI: levels 1..9 =
# 21,264,097 states, whose expansion is 2.4 M states' worth of invariant + Next evaluation)
CPU_SAMPLE_STATES = 30_000_000
CPU_SAMPLE_LEVELS = {"MCssi_4x3": 9}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    def __init__(self, dev=0):
        super().__init__(daemon=True)
        self.dev = dev
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.dev)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def expected(exp, levels):
    """the oracle's record for the whole job, or for its first `levels` levels (cumulative per-level record)"""
    o2 = exp["o2"]
    if not levels:
        return dict(verdict=o2["verdict"], generated=o2["generated"], distinct=o2["distinct"], depth=o2["depth"],
                    fp_xor=o2["fp_xor"], fp_sum=o2["fp_sum"], init=o2["levels"][0])
    x, sm, gen = o2["level_digests"][levels - 1]
    return dict(verdict=0, generated=gen, distinct=sum(o2["levels"][:levels]), depth=levels, fp_xor=x, fp_sum=sm,
                init=o2["levels"][0])


def cpu_reference(cm, init, info, threads, want, levels):
    """The reference arm: the path's CPU implementation (ORACLE O2, oracle/tlag_cpu.c -- TLC itself needs a JVM, which
    neither this image nor the reference provides) on all host cores, same model.  Bounded sample: a workload of more
    than 2 x CPU_SAMPLE_STATES states is cut at the end of the level that reaches CPU_SAMPLE_STATES."""
    from oracle import cpu_engine
    stop = CPU_SAMPLE_STATES if (want["distinct"] > 2 * CPU_SAMPLE_STATES and not levels) else 0
    size = min(want["distinct"], 12 * CPU_SAMPLE_STATES) if stop else want["distinct"]
    cap = max(1 << 16, int(size * 1.25) + 4096)
    r = cpu_engine.run(cm, init, n_threads=threads, deadlock=info["deadlock"], max_states=cap, stop_after=stop,
                       max_levels=levels)
    part = r["distinct"] < want["distinct"]
    r["sample"] = ((f"BFS prefix: the first {r['distinct']} distinct states (levels 1..{len(r['levels'])}) of the workload"
                    if part else "the whole workload job once") + " (oracle/tlag_cpu.c: persistent pinned workers, "
                   "first-touched table/store, all cores)")
    return r


def cpu_arm(cm, init, info, threads, want, levels, repeats, exp=None, workload=None):
    """median + spread over `repeats` runs of the bounded sample (depth-bounded workloads: a shorter prefix, sized
    from the oracle's per-level record)"""
    if workload in CPU_SAMPLE_LEVELS and exp is not None:
        levels = CPU_SAMPLE_LEVELS[workload]
        want = dict(want, distinct=sum(exp["o2"]["levels"][:levels]))
        rs = [cpu_reference(cm, init, info, threads, want, levels) for _ in range(repeats)]
        for r in rs:
            r["sample"] = r["sample"].replace("the whole workload job once",
                                              f"BFS prefix: levels 1..{levels} of the workload ({r['distinct']} distinct states)")
        return _summ(rs, repeats)
    return _summ([cpu_reference(cm, init, info, threads, want, levels) for _ in range(repeats)], repeats)


def _summ(rs, repeats):
    vals = sorted(r["distinct"] / r["seconds"] for r in rs)
    gvals = sorted(r["generated"] / r["seconds"] for r in rs)
    med = vals[len(vals) // 2]
    return rs[-1], med, {"distinct_per_s": [round(v, 1) for v in vals], "generated_per_s_median": round(gvals[len(gvals) // 2], 1),
                         "spread": round((vals[-1] - vals[0]) / med, 4) if med else None, "repeats": repeats}


def k1_microbench(dev, peak):
    """SURVEY.md 8(d): n = 2^27 candidates x W = 20 words, 50 % duplicates, table 2^28 slots.
    Algorithmic bytes per candidate = S + 8 + p*8 + 1 = 93 (S = 80, p = 0.5)."""
    import torch
    from tla_rust_b200.engine import Engine, ProbeOnlyModel
    W, n = 20, 1 << 27
    g = torch.Generator(device=dev).manual_seed(0x5EED)
    half = torch.randint(-2**31, 2**31 - 1, (n // 2, W), dtype=torch.int32, device=dev, generator=g)
    perm = torch.randint(0, n // 2, (n // 2,), device=dev, generator=g)
    states = torch.cat([half, half[perm]])
    del half, perm
    flags = torch.zeros(n, dtype=torch.uint8, device=dev)
    e = Engine(ProbeOnlyModel(W), table_log2=28, device=torch.device(dev).index or 0, native=False)
    times = []
    for it in range(2 + 5):
        e.reset_table()
        ms = e.probe_batch_device(states.data_ptr(), n, flags.data_ptr())
        if it >= 2:
            times.append(ms)
    n_new = int(flags.sum().item())
    med = float(np.median(times))
    bytes_per = 80 + 8 + 0.5 * 8 + 1
    ach = bytes_per * n / (med * 1e-3) / 1e9
    launches = e.launches()
    e.close()
    del states, flags
    torch.cuda.empty_cache()
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_probe"]
        if tj["n"] == n and tj["W"] == W:
            traffic = tj["bytes_per_launch"]
    except Exception:
        pass
    return {"kernel": "k_probe_staged", "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
            "frac": round(ach / peak, 4), "traffic": traffic, "n": n, "W": W, "p_new": n_new / n,
            "ms_per_launch": round(med, 4), "candidates_per_s": round(n / (med * 1e-3), 1),
            "bytes_per_candidate": bytes_per}, launches


DUMP_BYTES = 48 << 20        # budget of the state sample (float64 words); the whole dump stays under 64 MB
DUMP_CHUNK = 1 << 24         # states read back from the device at a time


def _sample_key(words):
    """64-bit mix of each state's words: a sample key that does not depend on the order the states were stored in"""
    h = np.zeros(words.shape[0], dtype=np.uint64)
    with np.errstate(over="ignore"):
        for j in range(words.shape[1]):
            h = (h ^ words[:, j].astype(np.uint64)) * np.uint64(0x9E3779B97F4A7C15)
            h ^= h >> np.uint64(29)
    return h


def dump_outputs(out_dir, e, r):
    """What the caller of one job receives: the result record, the state set's fingerprint digest and the stored states.
    The state set is too large to write whole; the sample is the states with the smallest sample keys, sorted, so that it
    is the same whatever order the parallel search stored them in."""
    os.makedirs(out_dir, exist_ok=True)
    keys = ("verdict", "detail", "generated", "distinct", "depth", "init_states", "queue_left")
    np.save(os.path.join(out_dir, "result.npy"), np.array([r[k] for k in keys], dtype=np.float64))
    x, s = e.digest()
    np.save(os.path.join(out_dir, "digest.npy"),
            np.array([x >> 32, x & 0xFFFFFFFF, s >> 32, s & 0xFFFFFFFF], dtype=np.float64))
    n, W = int(r["distinct"]), e.cm.W
    want = max(1, min(n, DUMP_BYTES // (8 * W)))
    cut = np.uint64(min(2**64 - 1, int(2**64 * min(1.0, 2.0 * want / n))))     # keeps ~2x the sample per chunk
    keep_w, keep_k = [], []
    for first in range(0, n, DUMP_CHUNK):
        w = e.read_states(first, min(DUMP_CHUNK, n - first))
        k = _sample_key(w)
        m = k <= cut
        keep_w.append(w[m])
        keep_k.append(k[m])
    w, k = np.concatenate(keep_w), np.concatenate(keep_k)
    order = np.lexsort(tuple(w[:, j] for j in range(W - 1, -1, -1)) + (k,))[:want]
    np.save(os.path.join(out_dir, "states_sample.npy"), w[order].astype(np.float64))


def side_workload(name, engine, local_rank, timeout, label):
    """another BASELINE config run once next to the headline (child process with a time limit; not part of `value`)"""
    try:
        if not os.path.exists(os.path.join(ROOT, "tests", "golden", name + ".tlagz")):
            return None
        cmd = [sys.executable, os.path.join(ROOT, "tools", "fixture_bench.py"), name, "--reps", "2"]
        if engine == "sliced":
            cmd.append("--sliced")
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout,
                           env=dict(os.environ, TLAG_NO_BUILD="1",
                                    CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank))))
        r3 = json.loads(p.stdout.strip().splitlines()[-1])
        return {"workload": label, "W": r3["W"], "distinct": r3["distinct"], "generated": r3["generated"],
                "depth": r3["depth"], "kernel_s": r3["device_s"], "distinct_per_s": r3["distinct_per_s"],
                "generated_per_s": r3["generated_per_s"], "engine_build": engine,
                "counts_match_oracle": r3["counts_match_oracle"], "digest_matches_oracle": r3["digest_matches_oracle"]}
    except Exception as ex:  # noqa: BLE001
        return {"workload": label, "error": str(ex)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="MCPaxos3_b4")
    ap.add_argument("--engine", default=os.environ.get("TLAG_BENCH_ENGINE", "sliced"), choices=["sliced", "interp"])
    ap.add_argument("--no-k1", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU arm (multi-GPU sessions: the other ranks' boxes idle meanwhile)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy "
                                                          "(result counts, digest, a fixed sample of the state set)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if os.environ.get("TLAG_BENCH_WATCHDOG"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["TLAG_BENCH_WATCHDOG"]), exit=True)

    from tla_rust_b200.compiled import load_compiled
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cm, init, exp, info = load_compiled(os.path.join(ROOT, "tests", "golden", args.workload + ".tlagz"))
    levels = WORKLOAD_LEVELS.get(args.workload, 0)
    want = expected(exp, levels)
    native = "sliced" if args.engine == "sliced" else False
    cfg = {"workload": f"{args.workload}: {info.get('source', '')} (compiled fixture), W={cm.W} words/state, "
                       f"{want['distinct']} distinct / {want['generated']} generated states"
                       + (f" in the first {levels} levels of an unending space" if levels else "")
                       + f", {len(cm.invariants)} invariants",
           "l2": "state store + seen-set rebuilt every step (restart), working set streamed; see DESIGN.md",
           "parallelism": f"state space partitioned by hash x{args.gpus}",
           "engine_build": "sliced native (one sm_100a kernel per invariant / disjunct of Next)" if native else "bytecode interpreter"}
    threads = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return
        r, v, spread = cpu_arm(cm, init, info, threads, want, levels, repeats=3, exp=exp, workload=args.workload)
        line = {"impl": "reference", "metric": "distinct states/sec", "value": round(v, 1), "unit": "states/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(1e3 * want["distinct"] / v, 3), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": round(v, 1), "unit": "states/s", "cores": threads, "kind": "port",
                                 "sample": r["sample"] + "; TLC itself needs a JVM: absent", **spread},
                "e2e": {"value": round(v, 1), "unit": "states/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from tla_rust_b200.engine import Engine
    dev = f"cuda:{local_rank}"
    torch.cuda.set_device(local_rank)
    peak, peak_src = load_peaks()
    multi = world > 1 or bool(os.environ.get("TLAG_FORCE_ROUTE"))   # knob: exercise the routed path on one GPU
    if multi and args.dump_outputs:
        sys.exit("--dump-outputs: single-process runs only (each rank of a partitioned run holds a shard of the states)")
    if multi:
        if world == 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29533")
            dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device(dev))
        else:
            dist.init_process_group("nccl", device_id=torch.device(dev))

    def barrier():
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    W = cm.W
    S = 4 * W
    h2d = int(cm.code.nbytes + cm.cpool.nbytes + cm.layout.nbytes + init.nbytes)
    stats = {}

    def check(r, digest):
        got = (r["verdict"] if r["verdict"] != 5 else 0, r["generated"], r["distinct"], r["depth"])
        assert got == (want["verdict"], want["generated"], want["distinct"], want["depth"]), (got, want)
        assert tuple(digest) == (want["fp_xor"], want["fp_sum"]), "fingerprint digest differs from the oracle's"

    if not multi:
        def job(e):
            if not levels:
                return e.run()
            for _ in range(levels - 1):
                e.step()
            return e.result()
        e = Engine(cm, deadlock=info["deadlock"], device=local_rank, native=native)
        e.seed(init)
        for _ in range(max(args.warmup, 1)):
            e.restart()
            r = job(e)
        check(r, e.digest())
        if sampler:
            sampler.start()
        barrier()
        t0 = time.perf_counter()
        kern_s = 0.0
        l0 = e.launches()
        for _ in range(args.steps):
            e.restart()
            r = job(e)
            kern_s += r["device_seconds"]
        barrier()
        dt = time.perf_counter() - t0
        launches = e.launches() - l0
        distinct, generated = r["distinct"], r["generated"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, e, r)
        # end to end through the C ABI with host buffers: create + seed(H2D) + run + result(D2H) + destroy
        e.close()
        barrier()
        t1 = time.perf_counter()
        for _ in range(args.steps):
            e2 = Engine(cm, deadlock=info["deadlock"], device=local_rank, native=native)
            e2.seed(init)
            r2 = job(e2)
            e2.close()
        torch.cuda.synchronize()
        dt_e2e = time.perf_counter() - t1
        assert r2["distinct"] == distinct
        stats = dict(kern_s=kern_s)
    else:
        from tla_rust_b200.dist import DistributedBFS
        # exchange buffers: ~4 GB of send regions per rank (the inbox is twice that), chunks sized so that a chunk's
        # records fit its regions at up to 20 successors per state (an overflow rolls the level back and halves the chunk)
        cap_rec = min(1 << 27, int(4e9 // ((cm.W + 2) * 4)))
        chunk_st = max(1 << 16, min(1 << 22, cap_rec // 20))
        e = Engine(cm, deadlock=info["deadlock"], device=local_rank, native=native)
        d = DistributedBFS(e, cm, rank, world, dev, cap_records=cap_rec, chunk_states=chunk_st)
        d.seed(init)
        exch, exch_note = d.exchange, d.exchange_note
        first = [True]

        def one():
            if not first[0]:
                e.restart()          # keeps the grown store / table / exchange buffers, re-seeds this rank's initial states
            first[0] = False
            l0 = e.launches()
            c0 = d.comm_ms
            out = d.run(max_levels=(levels - 1) if levels else 1 << 20)
            return out, out["local"]["device_seconds"], e.launches() - l0, d.comm_ms - c0
        for _ in range(max(args.warmup, 1)):
            out, _, _, _ = one()
        # bit-exact across ranks: counts AND the XOR / SUM digest of every rank's shard combined
        check(dict(out, verdict=out["verdict"]), d.global_digest())
        if sampler:
            sampler.start()
        barrier()
        t0 = time.perf_counter()
        kern_s, launches, comm_ms = 0.0, 0, 0.0
        for _ in range(args.steps):
            out, ks, ln, cms = one()
            kern_s += ks
            launches += ln
            comm_ms += cms
        barrier()
        dt = time.perf_counter() - t0
        tmax = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dt = float(tmax.item())
        distinct, generated = out["distinct"], out["generated"]
        # end to end: fresh engine + exchange buffers + host-side seed every step (host buffers in, result out)
        e.close()
        del d
        barrier()
        t1 = time.perf_counter()
        for _ in range(args.steps):
            e2 = Engine(cm, deadlock=info["deadlock"], device=local_rank, native=native)
            d2 = DistributedBFS(e2, cm, rank, world, dev, cap_records=cap_rec, chunk_states=chunk_st)
            d2.seed(init)
            out2 = d2.run(max_levels=(levels - 1) if levels else 1 << 20)
            e2.close()
            del d2
        barrier()
        dt_e2e = time.perf_counter() - t1
        tmax = torch.tensor([dt_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dt_e2e = float(tmax.item())
        assert out2["distinct"] == distinct
        stats = dict(kern_s=kern_s, comm_ms=comm_ms, exchange=exch, exchange_note=exch_note)

    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if rank != 0:
        if multi:
            dist.destroy_process_group()
        return

    value = distinct * args.steps / dt
    # roofline of the wave kernels (per level: the invariant kernels + one kernel per disjunct of Next, or the one
    # interpreter kernel): algorithmic bytes per step = S*expanded (frontier read) + 8*generated (slot probe) +
    #                      discovered*(8 slot write + S state write + 8 parent/meta)   [SURVEY 8d, fused form]
    expanded = distinct - (exp["o2"]["levels"][levels - 1] if levels else 0)
    bytes_step = S * expanded + 8 * generated + (distinct - want["init"]) * (8 + S + 8)
    ach = bytes_step * args.steps / max(stats["kern_s"], 1e-9) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["wave"]
        if tj["workload"] == args.workload and tj["engine"] == args.engine:
            traffic = tj["bytes_per_step"]
    except Exception:
        pass
    roof = {"kernel": ("k_sl_inv_* / k_sl_next_* (one kernel per invariant and per disjunct of Next over the frontier: "
                       "unpack, evaluate, pack, fingerprint, probe/insert, append)") if native else
                      "k_wave (bytecode interpreter: fused expand+fingerprint+probe+compact)",
            "bound": "hbm", "achieved": round(ach, 3), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 6),
            "traffic": traffic, "peak_source": peak_src, "bytes_per_step": int(bytes_step),
            "kernel_s_per_step": round(stats["kern_s"] / args.steps, 6),
            "note": "integer / hash work bound by instruction issue, not by HBM: see profiles/ for issue-active, "
                    "instructions per state and DRAM bytes per launch"}
    k1 = None
    k1_launches = 0
    if not args.no_k1 and not multi:
        try:
            k1, k1_launches = k1_microbench(dev, peak)
            k1["peak_source"] = peak_src
        except Exception as ex:  # noqa: BLE001
            k1 = {"error": str(ex)}
    if args.no_cpu:
        cpu_r, cpu_v, cpu_spread = {"sample": "skipped (--no-cpu)"}, 0.0, {}
    else:
        cpu_r, cpu_v, cpu_spread = cpu_arm(cm, init, info, threads, want, levels, repeats=3 if not multi else 1, exp=exp,
                                           workload=args.workload)
    others = []
    if not multi and not args.no_k1:
        for name, label, tmo in (
                ("MCraft_t4l3", "BASELINE config #4: examples/raft.tla via models/MCraft.tla, 3 servers, MaxTerm 4, MaxLogLen 3, "
                                "MaxMessages 3 (compiled fixture, whole state space)", 300),
                ("MCssi_4x3", "BASELINE config #5: examples/serializableSnapshotIsolation.tla via models/MCssi.tla, 4 transactions x "
                              "3 keys, 8 invariants, deadlock ON, first 10 levels = 168,052,153 states (compiled fixture)", 900)):
            if name != args.workload:
                o = side_workload(name, args.engine, local_rank, tmo, label)
                if o:
                    others.append(o)
    line = {"metric": "distinct states/sec", "value": round(value, 1), "unit": "states/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * dt / args.steps, 3),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": cfg, "generated_per_s": round(generated * args.steps / dt, 1),
            "roofline": roof, "k1_roofline": k1,
            "cpu_baseline": {"value": round(cpu_v, 1), "unit": "states/s", "cores": threads,
                             "kind": "port", "sample": cpu_r["sample"], **cpu_spread},
            "e2e": {"value": round(distinct * args.steps / dt_e2e, 1), "unit": "states/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 96},
            "gpu_launches": int(launches), "clocks": sampler.summary() if sampler else None,
            "parity": {"counts_match_oracle": True, "digest_matches_oracle": True},
            "other_workloads": others}
    if multi:
        # p2p: the exchange is device code inside the level (k_push / k_insert_inbox), no separate communication time;
        # nccl: time between the expand kernel and the end of the payload all_to_all
        line["exchange"] = ("peer memory over NVLink (CUDA IPC inboxes, k_push / k_insert_inbox)" if stats["exchange"] == "p2p"
                            else "NCCL all_to_all" + (f" ({stats['exchange_note']})" if stats["exchange_note"] else ""))
        line["comm_ms_per_step"] = round(stats["comm_ms"] / args.steps, 3)
        dist.destroy_process_group()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
