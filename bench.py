#!/usr/bin/env python3
"""bench.py -- genome-pairs/sec of the `skani triangle` hot path on synthetic 5 Mbp bacterial genomes.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config north|c2|dense|c5] [--shuffle-order] ...
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...)

A "step" is one full pass of the hot path (FracMinHash seeding -> marker screen -> chaining/ANI) over the whole
synthetic genome set.  `value` = genome pairs / second with the ASCII genomes already resident in HBM; `e2e` is the same
metric through the C ABI with HOST (pinned) buffers: H2D of every base and D2H of every result inside the timed region
(the call converts a share of every sub-batch to 2-bit on the host cores while the previous one is uploaded: that
packing is inside the timed region too).
After the timed legs the run VERIFIES itself (outside the timed regions): the kept-pair count and an order-independent
checksum of (ref, query, ani, af_ref, af_query) are all-reduced over the ranks (identical for every N), and a random
sample of kept pairs is re-chained by the CPU oracle (1e-4).  With N > 1 (or --shuffle-order) the whole measurement is
repeated on a seeded random permutation of the genome order (input order unrelated to relatedness: the worst case of the
multi-GPU exchange) and reported under "shuffled".
`--dump-outputs DIR` writes the kept pairs of the last timed step of the headline leg to DIR/<field>.npy (see dump_outputs),
so that two builds run with the same arguments can be compared output for output.
`--impl reference` times the reference's CPU algorithm (the C++ restatement in oracle/: the Rust crate cannot be built
in this image) on all host cores on the SAME configuration (full genome set).
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

UNIT = "genome-pairs/s"
CONFIGS = {   # BASELINE.json configs that are a triangle on one box (c3 = search, see tools/bench_search.py)
    "north": dict(genomes=10000, genome_len=5_000_000, cluster=20, c=125, marker_c=1000, rescue_small=True,
                  metric="genome-pairs/sec, skani triangle 10k x 5 Mbp synthetic"),
    "c2": dict(genomes=1000, genome_len=5_000_000, cluster=20, c=125, marker_c=1000, rescue_small=True,
               metric="genome-pairs/sec, skani triangle 1k x 5 Mbp synthetic (BASELINE.json configs[1])"),
    "c4": dict(genomes=50000, genome_len=5_000_000, cluster=20, c=125, marker_c=1000, rescue_small=True,
               metric="genome-pairs/sec, skani triangle 50k x 5 Mbp synthetic (BASELINE.json configs[3]; needs --gpus 8: 31 GB of bases and 14 GB of sketches per GPU; not measured this round)"),
    "dense": dict(genomes=2000, genome_len=5_000_000, cluster=2000, c=125, marker_c=1000, rescue_small=True,
                  metric="genome-pairs/sec, skani triangle 2000 x 5 Mbp synthetic, ONE cluster (every pair is chained)"),
    "c5": dict(genomes=200000, genome_len=30_000, cluster=10, c=30, marker_c=200, rescue_small=False,
               metric="genome-pairs/sec, skani triangle --small-genomes on 200k x 30 kb synthetic contigs (BASELINE.json configs[4] shape)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="north", choices=sorted(CONFIGS))
    ap.add_argument("--genomes", type=int, default=None)
    ap.add_argument("--genome-len", type=int, default=None)
    ap.add_argument("--cluster", type=int, default=None)
    ap.add_argument("--cpu-sample", type=int, default=400, help="genomes in the bounded CPU-baseline sample of the b200 arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shuffle-order", action="store_true", help="also measure a seeded random permutation of the genome order (always on for N > 1)")
    ap.add_argument("--no-2bit", action="store_true", help="skip the third leg (genomes already 2-bit packed in host memory)")
    ap.add_argument("--no-shuffle", action="store_true", help="skip the permuted-order measurement (A/B sessions)")
    ap.add_argument("--perm-seed", type=int, default=12345)
    ap.add_argument("--spot-check", type=int, default=200, help="kept pairs re-chained by the CPU oracle after the timed legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<field>.npy (rows sorted by ref_id, query_id)")
    a = ap.parse_args()
    cfg = dict(CONFIGS[a.config])
    for k in ("genomes", "genome_len", "cluster"):
        if getattr(a, k) is not None:
            cfg[k] = getattr(a, k)
    a.cfg = cfg
    a.genomes, a.genome_len, a.cluster = cfg["genomes"], cfg["genome_len"], cfg["cluster"]
    if a.genomes != CONFIGS[a.config]["genomes"]:
        cfg["metric"] = cfg["metric"] + " [--genomes %d]" % a.genomes
    return a


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle = C++ restatement of the reference algorithm; "port")
# ------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads for the CPU arm: all host CPUs this process may actually use.  The GPU boxes expose 128 logical CPUs but the
    container's cgroup grants a CPU-time quota (cpu.max, 16 CPUs on the round-1 boxes); running 128 threads under that quota
    is SLOWER than 32 (measured: seeding speed-up 15.9x at 16 threads, 18.7x at 32, 9.2x at 128), so use 2 threads per
    granted CPU, capped by the visible CPUs."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        pass
    if quota:
        n = max(1, min(n, int(round(2 * quota))))
    return n, quota


def oracle_setup(native):
    """Bind the oracle for baseline timing: -march=native build (made on this box) when possible, 4-lane AVX2 seeder on."""
    import oracle_py as O
    how = "-march=x86-64-v3 (portable build)"
    if native:
        path = O.build_native()
        if path and os.path.exists(path):
            O.use_library(path)
            how = "-march=native (built on this box)"
    simd = O.set_avx2_intrinsics(True)
    return O, how + (", AVX2 4-lane seeder (src/avx2_seeding.rs instruction mix)" if simd else ", scalar lane-by-lane seeder (no AVX2)")


def cpu_triangle(O, cfg, n_genomes, threads, ids=None):
    """Times seeding + screen + chain of the oracle on the first n_genomes synthetic genomes. Returns seconds and details."""
    from bench_support import synth
    L, G = cfg["genome_len"], cfg["cluster"]
    if ids is None:
        bases, off, goc = synth.generate(0, n_genomes, L, G=G)
    else:
        bases, off, goc = synth.generate_ids(ids, L, G=G)
    t0 = time.perf_counter()
    # seeding: OpenMP threads over genomes inside the oracle, the reference's own parallel structure (src/file_io.rs:149)
    sk = O.sketch_many(bases, off, goc, n_genomes, c=cfg["c"], marker_c=cfg["marker_c"], threads=threads)
    t1 = time.perf_counter()
    del bases
    res, info = O.triangle(sk, O.cmd(rescue_small=cfg["rescue_small"]), threads=threads)
    t2 = time.perf_counter()
    return dict(t_seed=t1 - t0, t_pairs=t2 - t1, t_total=t2 - t0, n_kept=len(res), n_chained=info["n_chained"],
                t_screen=info["t_screen"], t_chain=info["t_chain"])


def cpu_single_thread(O, cfg):
    """Per-thread rates of the oracle (1 thread): ms per genome seeded, ms per chained pair."""
    from bench_support import synth
    L, G = cfg["genome_len"], cfg["cluster"]
    n = min(G, 8)
    bases, off, goc = synth.generate(0, n, L, G=G, threads=1)
    t0 = time.perf_counter()
    sk = O.sketch_many(bases, off, goc, n, c=cfg["c"], marker_c=cfg["marker_c"], threads=1)
    t1 = time.perf_counter()
    res, info = O.triangle(sk, O.cmd(rescue_small=cfg["rescue_small"]), threads=1)
    t2 = time.perf_counter()
    return {"seed_ms_per_genome": (t1 - t0) * 1e3 / n, "chain_ms_per_pair": (t2 - t1) * 1e3 / max(info["n_chained"], 1)}


def expected_pairs(n, G):
    """chained pairs of the clustered set: every pair inside a cluster"""
    return (n // G) * (G * (G - 1) // 2) + ((n % G) * (n % G - 1) // 2)


def scale_sample(d, S, N, G):
    """sample -> full set: seeding and the marker index are linear in the genomes, chaining in the chained pairs"""
    return (d["t_seed"] + d["t_screen"]) * (N / S) + (d["t_total"] - d["t_seed"] - d["t_screen"]) * (expected_pairs(N, G) / max(expected_pairs(S, G), 1))


def cpu_sample_baseline(O, how, args, threads):
    """Bounded sample (b200 arm, rank 0): the first S genomes, scaled linearly to the full set (extrapolation, labelled)."""
    cfg = args.cfg
    S = min(args.cpu_sample, args.genomes)
    if args.cluster <= S:
        S = max(args.cluster, (S // args.cluster) * args.cluster)
    d = cpu_triangle(O, cfg, S, threads)
    N = args.genomes
    t_full = scale_sample(d, S, N, args.cluster)
    value = (N * (N - 1) / 2) / t_full
    one = cpu_single_thread(O, cfg)
    return {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "single_thread": one, "extrapolated": S != N,
            "cgroup_cpu_quota": host_threads()[1], "build": how,
            "sample": "oracle (C++ restatement of skani 0.3.0; Rust reference not buildable here) triangle on %d of the %d genomes "
                      "(%d clusters): %.2f s (seeding %.2f s; serial marker index + screen %.2f s; chain %.2f s for %d pairs) scaled "
                      "to the full set (seeding + index x%.1f, chaining by the number of chained pairs); the full-size measurement is "
                      "`bench.py --impl reference`" % (S, N, max(S // args.cluster, 1), d["t_total"], d["t_seed"], d["t_screen"],
                                                      d["t_chain"], d["n_chained"], N / S)}, d


def workload_name(cfg):
    """config.workload, identical for both arms (same synthetic set, same sketch parameters)"""
    return ("triangle %d x %d bp synthetic clustered (G=%d, subst 0.1-5%%, inversions, 50-contig members), c=%d k=15 m=%d%s; "
            "inputs %.1f GB >> L2 (no flush needed)" % (cfg["genomes"], cfg["genome_len"], cfg["cluster"], cfg["c"], cfg["marker_c"],
                                                        "" if cfg["rescue_small"] else " --faster-small",
                                                        cfg["genomes"] * cfg["genome_len"] / 1e9))


# ------------------------------------------------------------------------------------------------------------
# reference arm: the CPU algorithm on the SAME configuration (all genomes), all host threads
# ------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = args.cfg
    threads, quota = host_threads()
    O, how = oracle_setup(native=True)
    N = args.genomes
    total_pairs = N * (N - 1) // 2
    runs = []
    warm = args.warmup
    for i in range(warm + args.steps):
        d = cpu_triangle(O, cfg, N, threads)
        if i >= warm:
            runs.append(d)
    t = float(np.mean([r["t_total"] for r in runs]))
    v = total_pairs / t
    last = runs[-1]
    # the b200 arm's bounded sample, measured here as well, to say how good the linear extrapolation is
    S = min(args.cpu_sample, N)
    if args.cluster <= S:
        S = max(args.cluster, (S // args.cluster) * args.cluster)
    extrap = None
    if S < N:
        ds = cpu_triangle(O, cfg, S, threads)
        ve = total_pairs / scale_sample(ds, S, N, args.cluster)
        extrap = {"sample_genomes": S, "extrapolated_value": ve, "measured_over_extrapolated": v / ve}
    cb = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "cgroup_cpu_quota": quota, "build": how, "extrapolated": False,
          "sample_extrapolation_check": extrap,
          "sample": "oracle (C++ restatement of skani 0.3.0; Rust reference not buildable here) triangle on ALL %d genomes: %.2f s "
                    "(seeding %.2f s; serial marker index + screen %.2f s; chain %.2f s for %d pairs; %d kept), %d step(s), no scaling"
                    % (N, last["t_total"], last["t_seed"], last["t_screen"], last["t_chain"], last["n_chained"], last["n_kept"], len(runs))}
    line = {"impl": "reference", "metric": cfg["metric"], "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(runs), "warmup": warm,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(cfg), "genomes": N, "genome_len": args.genome_len, "pairs": total_pairs,
                       "kept_pairs": last["n_kept"]},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------
# verification helpers (outside every timed region)
# ------------------------------------------------------------------------------------------------------------
def result_checksum(res):
    """Order-independent 64-bit checksum of the kept results: sum over rows of a mix of (ref, query, ani, af_ref, af_query) bits."""
    if len(res) == 0:
        return 0
    u64 = np.uint64
    a = (res["ref_id"].astype(u64) << u64(32)) | res["query_id"].astype(u64)
    b = (res["ani"].view(np.uint32).astype(u64) << u64(32)) | res["af_ref"].view(np.uint32).astype(u64)
    c = res["af_query"].view(np.uint32).astype(u64)
    with np.errstate(over="ignore"):
        x = a * u64(0x9E3779B97F4A7C15) ^ b * u64(0xBF58476D1CE4E5B9) ^ c * u64(0x94D049BB133111EB)
        x ^= x >> u64(31)
        x = x * u64(0xD6E8FEB86659FD93)
        x ^= x >> u64(29)
        return int(np.sum(x, dtype=u64))


def allreduce_count_checksum(count, cks, world):
    if world == 1:
        return count, cks
    import torch
    t = torch.tensor([count, cks & 0xFFFFFFFF, cks >> 32], dtype=torch.int64, device="cuda")
    torch.distributed.all_reduce(t)
    c, lo, hi = [int(x) for x in t.cpu().tolist()]
    return c, (lo + (hi << 32)) & 0xFFFFFFFFFFFFFFFF


def oracle_spot_check(res, ids, cfg, n_sample, seed):
    """Re-chain a random sample of the kept pairs with the CPU oracle: |d ani|, |d af| <= 1e-4 (north_star's tolerance)."""
    import oracle_py as O
    from bench_support import synth
    if len(res) == 0 or n_sample <= 0:
        return {"pairs": 0}
    rng = np.random.default_rng(seed)
    pick = res[np.sort(rng.choice(len(res), min(n_sample, len(res)), replace=False))]
    slots = np.unique(np.concatenate([pick["ref_id"], pick["query_id"]]))
    bases, off, goc = synth.generate_ids(ids[slots], cfg["genome_len"], G=cfg["cluster"])
    threads = host_threads()[0]
    osk = O.sketch_many(bases, off, goc, len(slots), c=cfg["c"], marker_c=cfg["marker_c"], threads=threads)   # named by rank = slot order
    del bases
    worst = 0.0
    cp = O.cmd(rescue_small=cfg["rescue_small"])
    for r in pick:
        o = O.chain(osk[int(np.searchsorted(slots, r["ref_id"]))], osk[int(np.searchsorted(slots, r["query_id"]))], cp)
        for f in ("ani", "af_ref", "af_query"):
            worst = max(worst, abs(float(r[f]) - float(getattr(o, f))))
    return {"pairs": int(len(pick)), "max_abs_diff": worst, "tolerance": 1e-4, "ok": bool(worst <= 1e-4)}


DUMP_LIMIT = 64 << 20


def pair_key(res):
    """64-bit mix of (ref_id, query_id): a fixed pseudo-random order of the pairs, the same whichever build computed them."""
    u64 = np.uint64
    with np.errstate(over="ignore"):
        x = ((res["ref_id"].astype(u64) << u64(32)) | res["query_id"].astype(u64)) * u64(0x9E3779B97F4A7C15)
        x ^= x >> u64(31)
        return x * u64(0xD6E8FEB86659FD93)


def dump_outputs(res, out_dir):
    """One DIR/<field>.npy per RESULT_DTYPE field of the kept pairs, rows sorted by (ref_id, query_id): scores in float32 as
    computed, ids and counts in float64 (exact).  When all rows would exceed 64 MB, the pairs with the smallest pair_key
    are written, so that two builds sample the same pairs."""
    cols = [(n, np.float32 if res.dtype[n] == np.float32 else np.float64) for n in res.dtype.names]
    row_bytes = sum(np.dtype(t).itemsize for _, t in cols)
    n_max = (DUMP_LIMIT - (1 << 20)) // row_bytes          # 1 MB left for the .npy headers
    sampled = len(res) > n_max
    if sampled:
        res = res[np.argsort(pair_key(res), kind="stable")[:n_max]]
    res = res[np.lexsort((res["query_id"], res["ref_id"]))]
    os.makedirs(out_dir, exist_ok=True)
    for n, t in cols:
        np.save(os.path.join(out_dir, n + ".npy"), res[n].astype(t))
    return {"dir": out_dir, "rows": int(len(res)), "sampled": sampled}


# ------------------------------------------------------------------------------------------------------------
# b200 arm
# ------------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import skani_b200 as sk
    from skani_b200 import _lib
    from bench_support import synth

    cfg = args.cfg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    if world != args.gpus and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE %d" % (args.gpus, world), file=sys.stderr)

    N, L, G = args.genomes, args.genome_len, args.cluster
    # genome shard of this rank (contiguous block of slots; global genome order = rank-major)
    g0, g1 = (N * rank) // world, (N * (rank + 1)) // world
    nloc = g1 - g0
    pinned = torch.empty(nloc * L, dtype=torch.uint8, pin_memory=True)
    host = pinned.numpy()
    ctx = sk.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    sp = sk.sketch_params(cfg["c"], 15, cfg["marker_c"])
    mp = sk.map_params(rescue_small=cfg["rescue_small"])
    total_pairs = N * (N - 1) // 2
    tri = None
    if world > 1:
        from skani_b200.multi_gpu import DistTriangle
        tri = DistTriangle(ctx, world, rank, sp, mp)
    clocks = ClockSampler(local_rank)

    def measure(order):
        """value leg + e2e leg + verification on one genome order; returns a dict (rank 0) / None."""
        ids = np.arange(N, dtype=np.uint64) if order == "contiguous" else synth.shuffled_ids(N, args.perm_seed)
        t_gen0 = time.perf_counter()
        synth.generate_ids(ids[g0:g1], L, G=G, out=host)
        off, goc = synth.layout_ids(ids[g0:g1], L, G)
        t_gen = time.perf_counter() - t_gen0
        dev_bases = pinned.to("cuda", non_blocking=False)
        last = {}
        packed = {}

        def step(e2e):
            if e2e == "2bit":           # genomes already 2-bit packed in (pinned) host memory: SURVEY 8(d)'s other starting point
                if world == 1:
                    res, st = sk.triangle_2bit(ctx, packed["units"], None, packed["lens"], goc, nloc, sp, mp)
                    last["res"] = res
                    return len(res)
                kept = tri.step(None, 0, off, goc, nloc, g0, N, packed=(packed["units"], None, packed["lens"]))
                last["res"] = tri.last_results
                return kept
            if world == 1:
                if e2e:
                    res, st = sk.triangle(ctx, host, off, goc, nloc, sp, mp, as_array=True)
                    last["res"] = res
                    return len(res)
                # genomes resident in HBM: sketch -> screen -> chain back to back on one stream (sk_triangle also accepts the device
                # pointer, but its two-stream pipeline buys nothing without an upload to hide: 460 vs 441 ms, session r2l)
                gs = sk.sketch_contigs(ctx, None, off, goc, nloc, sp, device_ptr=dev_bases.data_ptr())
                pairs = sk.screen_triangle(ctx, gs, mp)
                res = sk.chain_pairs(ctx, gs, gs, pairs, mp, as_array=True)
                res = res[res["ani"] > 0.1]
                gs.free()
                last["res"] = res
                return len(res)
            kept = tri.step(host if e2e else None, dev_bases.data_ptr() if dev_bases is not None else 0, off, goc, nloc, g0, N)
            last["res"] = tri.last_results
            return kept

        def timed(e2e, n_steps):
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = ctx.launches
            t0 = time.perf_counter()
            ev0.record(stream)
            kept = 0
            per_step = []
            for _ in range(n_steps):
                ts = time.perf_counter()
                kept = step(e2e)                      # blocks until the step's results are on the host
                per_step.append(round((time.perf_counter() - ts) * 1e3, 1))
            ev1.record(stream)
            torch.cuda.synchronize()
            if world > 1:
                torch.distributed.barrier()
            wall = time.perf_counter() - t0
            dev_ms = ev0.elapsed_time(ev1)
            ms = max(dev_ms, wall * 1e3)  # the step blocks on its own D2H copies; wall >= device span. report the larger
            if world > 1:
                t = torch.tensor([ms], device="cuda")
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
                ms = float(t.item())
            last["step_ms_2bit" if e2e == "2bit" else "step_ms_e2e" if e2e else "step_ms_value"] = per_step   # rank-local wall clock of each step (spread, not the metric)
            return ms / n_steps, kept, ctx.launches - l0

        # value leg first (needs the device-resident copy of the bases), then the roofline probes, then drop the device copy
        # before the end-to-end leg so that both legs run with comfortable HBM headroom
        for _ in range(max(args.warmup, 0)):
            step(False)
        ms_val, _, launches = timed(False, args.steps)
        ck_val = allreduce_count_checksum(len(last["res"]), result_checksum(last["res"]), world)
        dumped = None
        if args.dump_outputs and order == "contiguous":
            res = last["res"]
            if world > 1:
                parts = [None] * world
                torch.distributed.all_gather_object(parts, res)
                res = np.concatenate(parts)
            if rank == 0:
                dumped = dump_outputs(res, args.dump_outputs)
        roof = roof_chain = None
        if rank == 0 and order == "contiguous":
            roof = measure_hashpass(ctx, dev_bases, off, goc, nloc, sp, L)
            roof_chain = measure_chain(ctx, dev_bases, off, goc, nloc, sp, mp, L, G)
        dev_bases = None
        torch.cuda.empty_cache()
        for _ in range(max(args.warmup, 0)):
            step(True)
        ms_e2e, kept, _ = timed(True, args.steps)
        res = last["res"]
        step_ms_e2e = last.get("step_ms_e2e")
        pack_share = ctx.last_pack_share
        d2h = len(res) * C.sizeof(_lib.AniResult)
        ck_e2e = allreduce_count_checksum(len(res), result_checksum(res), world)
        if world > 1:
            t = torch.tensor([d2h], dtype=torch.int64, device="cuda")
            torch.distributed.all_reduce(t)
            d2h = int(t.item())
        spot = None
        if rank == 0:
            spot = oracle_spot_check(res, ids, cfg, args.spot_check, 99)
        # third leg: the same call on genomes that are ALREADY 2-bit packed in host memory (sk_triangle_2bit): 0.25 B/base leave
        # host DRAM instead of 1, which is what bounds the ASCII leg when several GPUs share one host
        ms_2bit = ck_2bit = None
        if not args.no_2bit and order == "contiguous":
            import concurrent.futures
            lens = np.diff(off).astype(np.uint32)
            uoff = np.concatenate([[0], np.cumsum((lens.astype(np.uint64) + 31) // 32)]).astype(np.int64)
            pu = torch.empty(max(int(uoff[-1]), 1), dtype=torch.int64, pin_memory=True)
            scratch_nm = np.zeros(int(((lens.astype(np.int64) + 31) // 32).max()) if len(lens) else 1, np.uint32)
            ua = pu.numpy().view(np.uint64)
            Lh = _lib.load()
            def pack_range(lo, hi):
                nm = np.zeros_like(scratch_nm)
                for i in range(lo, hi):
                    Lh.sk_pack_contig(host.ctypes.data + int(off[i]), int(lens[i]), ua.ctypes.data + 8 * int(uoff[i]), nm.ctypes.data)
            nthr = max(1, min(16, len(os.sched_getaffinity(0)) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
            cuts = np.linspace(0, len(lens), nthr + 1).astype(int)
            with concurrent.futures.ThreadPoolExecutor(nthr) as ex:
                list(ex.map(lambda k: pack_range(int(cuts[k]), int(cuts[k + 1])), range(nthr)))
            packed.update(units=ua.ctypes.data, lens=lens, keep=pu)
            for _ in range(max(args.warmup, 0)):
                step("2bit")
            ms_2bit, _, _ = timed("2bit", args.steps)
            ck_2bit = allreduce_count_checksum(len(last["res"]), result_checksum(last["res"]), world)
            packed.clear()
        if rank != 0:
            return None
        expected = expected_pairs(N, G)
        return {"order": order, "value": total_pairs / (ms_val * 1e-3), "ms_per_step": ms_val, "launches": int(launches),
                "e2e_value": total_pairs / (ms_e2e * 1e-3), "e2e_ms_per_step": ms_e2e, "d2h": int(d2h), "host_gen_s": round(t_gen, 2),
                "host_pack_share": round(pack_share, 3), "step_ms_value": last.get("step_ms_value"), "step_ms_e2e": step_ms_e2e,
                "e2e_2bit_ms_per_step": ms_2bit, "step_ms_2bit": last.get("step_ms_2bit"), "units_bytes": int(((np.diff(off).astype(np.int64) + 31) // 32).sum() * 8),
                "checksum_2bit": (None if ck_2bit is None else "%016x" % ck_2bit[1]), "kept_2bit": (None if ck_2bit is None else int(ck_2bit[0])),
                "verify": {"kept_pairs_all_ranks": ck_e2e[0], "kept_pairs_expected": expected, "kept_ok": ck_e2e[0] == expected == ck_val[0],
                           "checksum_e2e": "%016x" % ck_e2e[1], "checksum_value_leg": "%016x" % ck_val[1],
                           "legs_agree": ck_e2e == ck_val, "oracle_spot_check": spot},
                "roof": roof, "roof_chain": roof_chain, "dumped": dumped}

    if rank == 0:
        clocks.start()
    m = measure("contiguous")
    shuf = None
    if (world > 1 or args.shuffle_order) and not args.no_shuffle:
        shuf = measure("shuffled")
    clk = clocks.stop() if rank == 0 else None

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        O, how = oracle_setup(native=True)
        cpu, _d = cpu_sample_baseline(O, how, args, host_threads()[0])
    if rank == 0:
        line = {"metric": cfg["metric"], "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic",
                "config": {"workload": workload_name(cfg), "genomes": N, "genome_len": L, "pairs": total_pairs, "order": "contiguous (clusters adjacent)",
                           "host_gen_s": m["host_gen_s"], "verify": m["verify"]},
                "step_ms_rank0": m["step_ms_value"],
                "e2e": {"value": m["e2e_value"], "unit": UNIT, "ms_per_step": m["e2e_ms_per_step"], "step_ms_rank0": m["step_ms_e2e"],
                        "h2d_bytes_per_step": int(N * L * (1.0 - 0.75 * m["host_pack_share"])), "d2h_bytes_per_step": m["d2h"],
                        "host_bytes_per_step": int(N * L), "host_pack_share": m["host_pack_share"],
                        "note": "inputs = ASCII in pinned host memory; host_pack_share of the bases is converted to 2-bit on the host "
                                "cores inside the timed call (0.25 B/base on the wire), the rest crosses PCIe as ASCII"},
                "gpu_launches": m["launches"], "clocks": clk, "roofline": m["roof"], "roofline_chain": m["roof_chain"], "cpu_baseline": cpu}
        if m["dumped"]:
            line["dumped_outputs"] = m["dumped"]
        if m.get("e2e_2bit_ms_per_step"):
            line["e2e_2bit"] = {"what": "the same call on genomes that are already 2-bit packed in pinned host memory (sk_triangle_2bit; SURVEY 8(d): "
                                        "'resident in host memory as ASCII/2-bit'); results on the host; the ASCII leg above stays the headline `e2e`",
                                "value": total_pairs / (m["e2e_2bit_ms_per_step"] * 1e-3), "unit": UNIT, "ms_per_step": m["e2e_2bit_ms_per_step"],
                                "step_ms_rank0": m["step_ms_2bit"], "h2d_bytes_per_step": m["units_bytes"] * (world if world > 1 else 1),
                                "kept_pairs_all_ranks": m["kept_2bit"], "checksum": m["checksum_2bit"],
                                "same_results_as_e2e": m["checksum_2bit"] == m["verify"]["checksum_e2e"] and m["kept_2bit"] == m["verify"]["kept_pairs_all_ranks"]}
        if shuf:
            line["shuffled"] = {"what": "same genomes, seeded random permutation of the genome order (perm seed %d): input order unrelated "
                                        "to relatedness" % args.perm_seed,
                                "value": shuf["value"], "ms_per_step": shuf["ms_per_step"], "e2e_value": shuf["e2e_value"],
                                "e2e_ms_per_step": shuf["e2e_ms_per_step"], "host_pack_share": shuf["host_pack_share"], "verify": shuf["verify"]}
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


def _peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def _ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per unit of work from THIS round's ncu --set full capture
    (profiles/r02_traffic.json, written by tools/profile_step.py + tools/summarize_ncu.py); None if absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[kernel]
    except Exception:
        return None


def measure_hashpass(ctx, dev_bases, off, goc, nloc, sp, L):
    """Roofline of the dominant seeding kernel (hashpass_kernel), timed live with CUDA events on the launch stream
    (sk_ctx_set_timing brackets every launch).  Algorithmic bytes: SURVEY.md section 8(d) seeding figure
    L/4 + L/8 + 12 L/c + 8 L/m per genome (2.395 MB at L = 5 Mbp), times the genomes one launch processes."""
    import skani_b200 as sk
    n = min(nloc, max(1, int(1.0e9 // L)))
    n_contigs = int(np.searchsorted(goc, n))
    o, g = off[:n_contigs + 1], goc[:n_contigs]
    sk.sketch_contigs(ctx, None, o, g, n, sp, device_ptr=dev_bases.data_ptr()).free()   # warm
    ctx.get_timing(reset=True)
    ctx.set_timing(True)
    reps = 3
    for _ in range(reps):
        sk.sketch_contigs(ctx, None, o, g, n, sp, device_ptr=dev_bases.data_ptr()).free()
    t = ctx.get_timing(reset=True)
    ctx.set_timing(False)
    ms, launches = t["hashpass_kernel"]
    bytes_per_genome = L / 4.0 + L / 8.0 + 12.0 * L / sp.c + 8.0 * L / sp.marker_c
    genomes_per_launch = n * reps / launches
    sec_per_launch = ms * 1e-3 / launches
    peak, peak_src = _peak()
    ach = genomes_per_launch * bytes_per_genome / sec_per_launch / 1e9
    stage_ms = sum(v[0] for v in t.values())
    tr = _ncu_traffic("hashpass_kernel")      # {"dram_bytes_per_base": ..., "issue_active_pct": ..., "inst_per_window": ..., "source": ...}
    traffic = tr["dram_bytes_per_base"] * L * genomes_per_launch if tr else None
    alu = None
    if tr and tr.get("inst_per_window"):
        # issue roofline: one warp instruction per cycle per SM sub-partition (4 per SM); windows/s at that rate
        sm, mhz = 148, 1965.0
        peak_windows = sm * 4 * 32 * mhz * 1e6 / tr["inst_per_window"]
        alu = {"inst_per_window": tr["inst_per_window"], "issue_active_pct": tr.get("issue_active_pct"),
               "busiest_pipe_pct": tr.get("sm_throughput_pct"),     # ncu sm__throughput: the integer ALU pipe (half-rate LOP3/SHF/IADD3)
               "windows_per_s": genomes_per_launch * L / sec_per_launch, "issue_peak_windows_per_s": peak_windows,
               "frac_of_issue_peak": genomes_per_launch * L / sec_per_launch / peak_windows}
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
            "traffic_source": tr["source"] if tr else None, "alu": alu,
            "kernel": "hashpass_kernel", "launch_ms": sec_per_launch * 1e3, "genomes_per_launch": genomes_per_launch,
            "algorithmic_bytes_per_genome": bytes_per_genome,
            "gbases_per_s": genomes_per_launch * L / sec_per_launch / 1e9,
            "kernel_ms": {k: round(v[0] / reps, 3) for k, v in t.items()}, "timed_kernels_ms_per_rep": round(stage_ms / reps, 3),
            "note": "nominal bound = HBM (north_star); the kernel is integer-issue bound (64-bit hash per base at 0.375 B/base), see `alu` and DESIGN.md",
            "peak_source": peak_src}


def measure_chain(ctx, dev_bases, off, goc, nloc, sp, mp, L, G):
    """Roofline block of the chaining stage: 0.96 MB algorithmic bytes per chained pair (SURVEY 8d: 12 B x (S_q + S_r) + 64) over
    the CUDA-event time of the chain kernels of one batch."""
    import skani_b200 as sk
    n = min(nloc, max(G, int(2.0e9 // L) // G * G))
    n_contigs = int(np.searchsorted(goc, n))
    gs = sk.sketch_contigs(ctx, None, off[:n_contigs + 1], goc[:n_contigs], n, sp, device_ptr=dev_bases.data_ptr())
    pairs = sk.screen_triangle(ctx, gs, mp)
    sk.chain_pairs(ctx, gs, gs, pairs, mp, as_array=True)    # warm
    ctx.get_timing(reset=True)
    ctx.set_timing(True)
    sk.chain_pairs(ctx, gs, gs, pairs, mp, as_array=True)
    t = ctx.get_timing(reset=True)
    ctx.set_timing(False)
    recs = sum(gs.info(g)["n_records"] for g in range(n)) / n
    gs.free()
    ms = sum(v[0] for v in t.values())
    if len(pairs) == 0 or ms <= 0:
        return None
    bpp = 12.0 * 2 * recs + 64
    peak, peak_src = _peak()
    ach = bpp * len(pairs) / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "pairs": int(len(pairs)),
            "us_per_pair": ms * 1e3 / len(pairs), "algorithmic_bytes_per_pair": bpp,
            "kernel_ms": {k: round(v[0], 3) for k, v in t.items()}, "peak_source": peak_src,
            "note": "chaining is latency / issue bound integer work (hash probes, banded DP, greedy selection), far from the HBM roofline"}


if __name__ == "__main__":
    sys.dont_write_bytecode = True   # the tree may be read-only: the modules main() imports from it leave no bytecode there
    sys.exit(main())
