#!/usr/bin/env python
"""bench.py — haystacks/sec of the match_list / match_list_parallel hot path on N B200s (DESIGN.md §5).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (restated)
    python bench.py ... --dump-outputs DIR                   # also writes the last timed step's match list (.npy)

A "step" is one blocking Matcher::match_list_parallel call (frz_match_list_parallel_rank; at N = 1 this is
Matcher::match_list) over one synthetic haystack list of BASELINE.json configs[2] shape per GPU — needle 'deadbeef',
10M haystacks, len <= 64 (mean 48), max_typos = 1 — weak scaling: rank r holds its own 10M-item shard with the indices
[r*10M, (r+1)*10M); a step is the local pipeline on every GPU, the k-way merge + exchange (host-out: ONE kernel per GPU that
stores its matches at their merged positions in the peers' slice buffers over NVLink; device-out: ONE NCCL all-gather of the
per-shard runs + the merge on every GPU), and every GPU copying its slice of the merged list into ONE pinned host buffer
shared by the ranks.

  value            whole-job haystacks/s, packed shards resident in HBM when the timed region starts, the ordered match
                   list LANDED IN PINNED HOST MEMORY when a step ends (SURVEY.md §8(d)); same definition at every N.
  value_device_out the same step without the final device->host copy (the merged list left in HBM).
  e2e              the same metric with the shard arriving as HOST Arrow buffers every step
                   (frz_match_list_parallel_rank_host: streamed H2D + pack + match + D2H inside the timed region).
Every loop runs a rank-identical, fixed number of steps (rank 0 decides the pre/post-roll length, everybody gets it by
broadcast): ranks never issue different numbers of collectives.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import datetime
import json
import os
import subprocess
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOAD = dict(needle="deadbeef", n=10_000_000, mu=48, max_len=64, max_typos=1, seed=12345)
PUBLISHED_CALIBRATION_MS = 1.85   # /root/reference/BENCHMARKS.md:124 — "Partial Match", median length 64, 100k items, `1 Typo`, 1 thread


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--haystacks-per-gpu", dest="n", type=int, default=WORKLOAD["n"],
                    help="haystacks per GPU (under torchrun spell it --haystacks-per-gpu: torchrun's own parser treats --n as an abbreviation)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="default: min(steps, 5)")
    ap.add_argument("--e2e-offsets", type=int, default=32, choices=[32, 64],
                    help="Arrow offset width of the e2e input (32 = Utf8, 64 = LargeUtf8)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="haystacks in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the full-shard parity leg (profiling runs)")
    ap.add_argument("--lanes", type=int, default=0, help="emulate_lanes (0 = what the reference picks on this CPU)")
    # the other BASELINE.json configs are parity-test cases; these flags let profiles/ record their numbers too
    ap.add_argument("--needle", default=WORKLOAD["needle"])
    ap.add_argument("--max-typos", type=int, default=WORKLOAD["max_typos"])
    ap.add_argument("--mu", type=int, default=WORKLOAD["mu"])
    ap.add_argument("--max-len", type=int, default=WORKLOAD["max_len"])
    ap.add_argument("--query", default=None, help="a multi-pattern query (Matcher::from_query), e.g. 'foo !^bar' (configs[4]); "
                                                  "the haystacks are generated around its first positive atom")
    ap.add_argument("--unicode-frac", type=float, default=0.0, help="fraction of haystacks with multibyte scalars spliced in")
    ap.add_argument("--prefix-frac", type=float, default=0.0, help="fraction of haystacks starting with 'bar'/'Bar'")
    ap.add_argument("--shards-per-gpu", type=int, default=1,
                    help="each GPU holds this many consecutive logical shards of --n haystacks (seeds consecutive): "
                         "`--gpus 1 --shards-per-gpu 8` matches the very list `--gpus 8` shards over 8 GPUs (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the ordered match list of the last timed step to DIR as .npy files "
                         "(see dump_outputs), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _gen_one(job):
    from frizbee_b200 import synth
    needle, n, mu, max_len, seed, ufrac, pfrac = job
    cache = os.environ.get("FRZ_BENCH_CACHE")   # A/B sweeps: generate a list once per box, reload it afterwards
    if cache:
        key = os.path.join(cache, f"synth_{needle}_{n}_{mu}_{max_len}_{seed}_{ufrac}_{pfrac}")
        if os.path.exists(key + "_o.npy"):
            return np.load(key + "_d.npy"), np.load(key + "_o.npy")
    data, off = synth.generate(needle, n, mu, max_len, seed, unicode_frac=ufrac, prefix_frac=pfrac)
    if cache:
        os.makedirs(cache, exist_ok=True)
        np.save(key + "_d.npy", data)
        np.save(key + "_o.npy", off)
    return data, off


def gen_needle(args) -> str:
    """The string the synthetic haystacks are built around: the needle, or the first positive atom of --query."""
    if not args.query:
        return WORKLOAD["needle"]
    for atom in args.query.split():
        if not atom.startswith("!"):
            return atom.strip("^$'")
    return "foo"


def make_rank_data(args, rank):
    """This rank's haystacks: `shards_per_gpu` logical shards of args.n items, logical shard j generated with seed + j
    (so the list does not depend on how many GPUs it is spread over).  Several shards are generated in parallel processes
    (called before torch / CUDA are initialised)."""
    S = args.shards_per_gpu
    jobs = [(gen_needle(args), args.n, WORKLOAD["mu"], WORKLOAD["max_len"], WORKLOAD["seed"] + rank * S + j, args.unicode_frac,
             args.prefix_frac) for j in range(S)]
    if S == 1:
        return _gen_one(jobs[0])
    import concurrent.futures as cf
    import multiprocessing as mp
    with cf.ProcessPoolExecutor(max_workers=min(S, 8), mp_context=mp.get_context("fork")) as ex:
        parts = list(ex.map(_gen_one, jobs))
    data = np.concatenate([p[0] for p in parts])
    offs = [parts[0][1]]
    base = int(parts[0][1][-1])
    for d, o in parts[1:]:
        offs.append(o[1:] + np.uint64(base))
        base += int(o[-1])
    return data, np.concatenate(offs)


def workload_patterns(args):
    """What the matcher is built from and what the CPU checker receives."""
    if args.query:
        import frizbee_b200 as F
        return F.parse_query(args.query)
    return [WORKLOAD["needle"]]


def workload_config(args):
    from frizbee_b200.types import Config
    return Config(max_typos=WORKLOAD["max_typos"], emulate_lanes=args.lanes)


def reference_lanes(args) -> int:
    """The lane width Matcher::get_backend (src/matcher/mod.rs:448-498) selects on THIS host for a u8-family needle —
    the oracle's own CPUID rule (no CUDA library involved)."""
    if args.lanes:
        return args.lanes
    from oracle import pyoracle as O
    return O.auto_lanes()


def config_block(args, world, extra=None):
    default = (WORKLOAD["needle"], WORKLOAD["max_typos"], WORKLOAD["mu"], WORKLOAD["max_len"], args.query, args.shards_per_gpu) == ("deadbeef", 1, 48, 64, None, 1)
    what = f"query '{args.query}'" if args.query else f"needle '{WORKLOAD['needle']}' (len {len(WORKLOAD['needle'])})"
    kind = "ASCII" if args.unicode_frac == 0 else f"mixed-unicode ({args.unicode_frac:.0%} with multibyte scalars, {args.prefix_frac:.0%} 'bar' prefixes)"
    c = {"workload": f"{what} vs {args.n * args.shards_per_gpu} synthetic {kind} haystacks per GPU, "
                     f"len<={WORKLOAD['max_len']} (mean {WORKLOAD['mu']}, sd {WORKLOAD['mu'] // 4}), max_typos={WORKLOAD['max_typos']}, "
                     f"5% full / 20% partial matches, seed 12345"
                     + (" (BASELINE.json configs[2], the configuration the 10x target is quoted on)" if default else ""),
         "haystacks_per_gpu": args.n * args.shards_per_gpu, "n_gpus": world, "sort": "ScoreThenIndexAsc",
         "l2": "inputs (~560 MB packed per GPU) are larger than the 126 MB L2; no explicit flush"}
    if extra:
        c.update(extra)
    return c


def pick_threads(cb, patterns, cfg, data, off, trials=3):
    """Thread count of the CPU arm: the reference's final k-way merge is single-threaded, so more threads is not always
    faster — the fastest of all / half / quarter of the host threads, decided on `trials` timed runs each."""
    threads = cb.host_threads()
    best = None
    for cand in sorted({threads, max(1, threads // 2), max(1, threads // 4)}, reverse=True):
        dt, _ = cb.timed(patterns, cfg, data, off, cand, repeats=trials)
        if best is None or dt < best[0]:
            best = (dt, cand)
    return best[1]


def calibration(cb, cfg):
    """BASELINE.md §2: the restated CPU path, ONE thread, on the reference's own published shape (100k haystacks, median
    length 64, needle 'deadbeef', max_typos 1: 1.85 ms on a Ryzen 9 9950X3D, BENCHMARKS.md:124)."""
    from frizbee_b200 import synth
    data, off = synth.generate("deadbeef", 100_000, 64, 128, 12345)
    c1 = cfg.with_(max_typos=1)
    dt, _ = cb.timed(["deadbeef"], c1, data, off, 1, repeats=7)
    return {"ours_ms_1thread": dt * 1e3, "published_ms": PUBLISHED_CALIBRATION_MS, "ratio_ours_over_published": dt * 1e3 / PUBLISHED_CALIBRATION_MS,
            "what": "100k haystacks, median len 64, 'deadbeef', max_typos=1, 1 thread, best of 7; published: Ryzen 9 9950X3D "
                    "(BENCHMARKS.md:124)"}


DUMP_BYTES = 64_000_000   # --dump-outputs: all files together stay below this


def dump_outputs(out_dir, matches):
    """Writes an ordered match list (MATCH_DTYPE) as DIR/matches_{index,score,exact}.npy (index float64, score and exact
    float32, all exact) and DIR/matches_count.npy (the list's length).  A list too long for DUMP_BYTES is replaced by a
    fixed, seeded sample of its rows, and DIR/matches_position.npy holds where the sampled rows sit in the full list."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(matches)
    max_rows = (DUMP_BYTES - 4096) // (8 + 4 + 4 + 8)   # index, score, exact, position; 4 KB for the .npy headers
    fields = {"count": np.array([n], dtype=np.float64)}
    if n > max_rows:
        pos = np.sort(np.random.default_rng(12345).choice(n, max_rows, replace=False))
        matches = matches[pos]
        fields["position"] = pos.astype(np.float64)
    fields.update(index=matches["index"].astype(np.float64), score=matches["score"].astype(np.float32),
                  exact=matches["exact"].astype(np.float32))
    for name, arr in fields.items():
        np.save(os.path.join(out_dir, f"matches_{name}.npy"), arr)


def run_reference(args):
    """The reference's own CPU implementation of the path (restated; no Rust toolchain here), all host threads,
    on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from frizbee_b200 import synth
    from oracle import cpu_baseline as cb
    cfg = workload_config(args)
    patterns = workload_patterns(args)
    sample = args.cpu_sample or args.n   # one logical shard of the workload: large enough to amortise thread start-up
    data, off = synth.generate(gen_needle(args), sample, WORKLOAD["mu"], WORKLOAD["max_len"], WORKLOAD["seed"],
                               unicode_frac=args.unicode_frac, prefix_frac=args.prefix_frac)
    lanes = reference_lanes(args)
    cfg = cfg.with_(emulate_lanes=lanes)
    threads = pick_threads(cb, patterns, cfg, data, off, trials=max(3, args.warmup))
    for _ in range(max(args.warmup, 3)):
        cb.match_list_parallel(patterns, cfg, data, off, threads)
    per_step = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        t1 = time.perf_counter()
        res = cb.match_list_parallel(patterns, cfg, data, off, threads)
        per_step.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {"impl": "reference", "metric": "haystacks/sec", "value": value, "unit": "haystacks/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * dt / args.steps,
            "ms_per_step_min": 1e3 * min(per_step), "ms_per_step_median": 1e3 * float(np.median(per_step)),
            "value_at_median_step": sample / float(np.median(per_step)),
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_block(args, args.gpus, {"sample_haystacks_per_step": sample, "matches_per_step": int(len(res))}),
            "cpu_baseline": {"value": value, "unit": "haystacks/s", "cores": threads, "kind": "port",
                             "sample": f"{sample} haystacks of the same workload per step; {cb.describe()}, "
                                       f"threaded like match_list_parallel (2048-item work claiming, workers pinned to "
                                       f"the process's CPUs round-robin), emulating the {lanes}-lane reference backend",
                             "calibration": calibration(cb, cfg)},
            "e2e": {"value": value, "unit": "haystacks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    print(json.dumps(line))


def check_parity(cb, O, patterns, cfg, data_np, off_np, index_offset, merged, rank, n_local, n_total):
    from frizbee_b200.types import SortStrategy
    """Full-shard parity: this rank's shard through the SIMD CPU restatement (validated bit-exact against the scalar
    oracle in tests/test_cpu_baseline.py) vs the entries of the MERGED list that fall into this rank's index range;
    rank 0 additionally checks the global order of the merged list and a 200k prefix against the scalar oracle."""
    threads = max(1, cb.host_threads() // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))))
    want = cb.match_list_parallel(patterns, cfg.with_(sort=SortStrategy.IndexAsc), data_np, off_np, threads)   # IndexAsc: the shard's matches in index order
    want = want.copy()
    want["index"] += np.uint32(index_offset)
    lo, hi = index_offset, index_offset + n_local
    mine = merged[(merged["index"] >= lo) & (merged["index"] < hi)]
    mine = mine[np.argsort(mine["index"], kind="stable")]
    if len(mine) != len(want):
        mism = max(1, abs(len(mine) - len(want)))
    else:
        mism = int(sum(int(np.count_nonzero(want[f] != mine[f])) for f in ("index", "score", "exact")))
    info = {"haystacks_checked": int(n_local), "matches_checked": int(len(want)), "mismatches": mism}
    if rank == 0:
        s = merged["score"].astype(np.int64)
        i = merged["index"].astype(np.int64)
        bad = int(np.count_nonzero((s[1:] > s[:-1]) | ((s[1:] == s[:-1]) & (i[1:] <= i[:-1]))))
        info["order_violations"] = bad
        info["index_out_of_range"] = int(np.count_nonzero(i >= n_total))
        sub = min(n_local, 200_000)
        w2 = O.match_list_packed(patterns, cfg.with_(sort=SortStrategy.IndexAsc), data_np[: int(off_np[sub])], off_np[: sub + 1])
        g2 = mine[mine["index"] < sub + index_offset]
        ok = len(w2) == len(g2) and all(np.array_equal(w2[f], g2[f] if f != "index" else g2[f] - np.uint32(index_offset))
                                        for f in ("index", "score", "exact"))
        info["scalar_oracle_prefix"] = {"haystacks": int(sub), "matches": int(len(w2)), "equal": bool(ok)}
        info["mismatches"] += bad + info["index_out_of_range"] + (0 if ok else 1)
    return info


def run_ours(args):
    rank0 = int(os.environ.get("RANK", "0"))
    RANK_DATA = make_rank_data(args, rank0)   # before torch / CUDA are initialised (may fork worker processes)
    import torch
    import torch.distributed as dist
    import frizbee_b200 as F
    from frizbee_b200 import parallel, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CUDA path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("FRZ_PARALLEL_TIMEOUT_S", "90")   # a missing peer fails the step with a message, not a hang
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "1")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def bcast_int(v: int) -> int:
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device=dev)
        dist.broadcast(t, 0)
        return int(t.item())

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: int) -> int:
        t = torch.tensor([int(x)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    cfg = workload_config(args)
    n = args.n * args.shards_per_gpu
    needle = WORKLOAD["needle"]
    patterns = workload_patterns(args)
    # each rank holds its own shard (weak scaling); rank r covers indices [r*n, (r+1)*n)
    data_np, off_np = RANK_DATA
    # pinned host buffers: the inputs of the e2e call
    data_pin = torch.empty(data_np.size, dtype=torch.uint8, pin_memory=True)
    off_pin = torch.empty(off_np.size, dtype=torch.int64, pin_memory=True)
    data_h = data_pin.numpy(); data_h[:] = data_np
    off_h = off_pin.numpy().view(np.uint64); off_h[:] = off_np
    if args.e2e_offsets == 32 and int(off_np[-1]) < 2 ** 31:   # Arrow Utf8: int32 offsets
        off32_pin = torch.empty(off_np.size, dtype=torch.int32, pin_memory=True)
        off_e2e = off32_pin.numpy(); off_e2e[:] = off_np
    else:
        off_e2e = off_h

    comm = parallel.Comm.from_torch_distributed(local)   # the data path's own NCCL communicator, behind the C ABI
    corpus = F.Corpus.from_arrow(data_h, off_h, device=local)
    matcher = F.Matcher.from_query(args.query, cfg) if args.query else F.Matcher(needle, cfg)
    info = matcher.backend_info()
    index_offset = rank * n

    # one device-only step sizes the shared host buffer (capacity = 1.25 x the observed total + slack)
    total0, _ = comm.match_list_parallel_rank(matcher, corpus, index_offset, None)
    cap = bcast_int(int(total0 * 1.25) + (1 << 20))
    out_h = comm.host_alloc_matches(cap)   # ONE pinned host buffer shared by all ranks (memfd segment for N > 1)

    def step():          # Matcher::match_list_parallel, the merged list landed in pinned host memory
        return comm.match_list_parallel_rank(matcher, corpus, index_offset, out_h)[0]

    def step_dev():      # the same without the final copy
        return comm.match_list_parallel_rank(matcher, corpus, index_offset, None)[0]

    def step_e2e():      # the shard arrives as host Arrow buffers
        return comm.match_list_parallel_rank_host(matcher, data_h, off_e2e, index_offset, out_h)

    for _ in range(max(args.warmup, 3)):
        n_matches = step()
    resident_result = np.array(out_h[:n_matches]) if rank == 0 else None   # the e2e call must land the very same list

    # ---- parity in the same run (outside the timed region): every rank checks its whole shard
    parity = None
    if not args.no_parity:
        from oracle import cpu_baseline as cb
        from oracle import pyoracle as O
        barrier()
        merged = np.array(out_h[:n_matches])   # every rank reads the whole shared buffer
        pcfg = cfg.with_(emulate_lanes=info["prefilter_lanes"])
        pi = check_parity(cb, O, patterns, pcfg, data_np, off_np, index_offset, merged, rank, n, n * world)
        mism = sum_over_ranks(pi["mismatches"])
        checked = sum_over_ranks(pi["matches_checked"])
        parity = dict(pi, mismatches=mism, matches_checked=checked, haystacks_checked=n * world,
                      matches_in_merged_list=int(n_matches),
                      checker=("oracle/cpu_baseline (SIMD restatement, bit-exact with the scalar oracle: tests/test_cpu_baseline.py)"
                               if (not args.query and WORKLOAD["max_typos"] in (0, 1)) else "the scalar oracle (oracle/frz_oracle.cpp), threaded over 2048-item chunks")
                              + ", every rank its whole shard; rank 0: global order + scalar-oracle 200k prefix")
        if checked != n_matches:
            parity["mismatches"] = mism + abs(checked - n_matches)
        del merged

    # ---- how many steps make 0.4 s (rank 0 decides, everybody runs the same number)
    barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        step()
    barrier()
    est = (time.perf_counter() - t0) / 5
    n_roll = bcast_int(min(4000, max(5, int(0.4 / max(est, 1e-5)))))

    def timed(fn, steps, clocks=False, last=None):
        """pre-roll, K timed steps between CUDA events, post-roll — all fixed counts; max over ranks.  `last` receives the
        last timed step's result before the post-roll runs."""
        sampler = ClockSampler(local) if clocks and rank == 0 else None
        barrier()
        if sampler:
            sampler.start()
            # nvidia-smi needs ~100 ms per sample: keep the GPU under the same load before (pre-roll) and after
            # (post-roll) the timed steps so that the samples describe the clocks the timed region ran at
            for _ in range(n_roll):
                fn()
        elif clocks:
            for _ in range(n_roll):
                fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = None
        for _ in range(steps):
            r = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if last is not None:
            last(r)
        if clocks:
            for _ in range(n_roll):
                fn()
            barrier()
        c = sampler.stop() if sampler else None
        return max_over_ranks(ms), r, c

    last_list = {}

    def keep_last(count):   # --dump-outputs: the merged list the last timed step landed in the shared host buffer
        if args.dump_outputs and rank == 0:
            last_list["matches"] = np.array(out_h[:count])

    ms, n_matches, clocks = timed(step, args.steps, clocks=True, last=keep_last)
    if clocks is not None:
        clocks["window"] = f"{n_roll} identical pre-roll steps + timed region + {n_roll} identical post-roll steps"
    value = n * world * args.steps / (ms / 1e3)
    ms_dev, _, _ = timed(step_dev, args.steps)

    # per-stage CUDA-event timings (recorded inside the library on the launching stream) from separate, identical steps
    stage_steps = 10
    stage = {k: 0.0 for k in ("prefilter_ms", "sw_ms", "sort_ms", "pipeline_ms", "local_ms", "gather_merge_ms", "d2h_ms", "total_ms")}
    launches = 0
    for _ in range(stage_steps):
        step()
        t = comm.last_timings(0)
        for k in stage:
            stage[k] += t.get(k, 0.0) / stage_steps
        launches += t.get("launches", 0)
    # kernels of this repo per step: the local pipeline + count publish + (N > 1: 3 merge kernels + copy-out flag)
    launches_per_step = launches / stage_steps + 1 + (4 if world > 1 else 0)

    # ---- timed region: end to end (host buffers in, host matches out)
    e2e_steps = args.e2e_steps or min(args.steps, 5)
    if e2e_steps > 0:
        step_e2e()   # warm
        e_ms, n_e2e, _ = timed(step_e2e, e2e_steps)
    else:            # --e2e-steps -1: profiling / large strong-scaling runs skip the end-to-end leg
        e_ms, n_e2e, e2e_steps = float("nan"), n_matches, 1
    e2e_equal = None
    if args.e2e_steps >= 0 and rank == 0 and resident_result is not None:
        e2e_equal = bool(n_e2e == n_matches and np.array_equal(np.array(out_h[:n_e2e]), resident_result))
    e2e_value = n * world * e2e_steps / (e_ms / 1e3)
    h2d = int(data_h.nbytes + off_e2e.nbytes)
    d2h_rank = int(n_e2e * 8 / world + 64)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        pf_ms = stage["prefilter_ms"]
        alg_bytes = int(corpus.total_bytes + 8 * n + 8 * n_matches / world)
        achieved = alg_bytes / (pf_ms / 1e3) / 1e9 if pf_ms > 0 else None
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if (needle, WORKLOAD["max_typos"], WORKLOAD["mu"], WORKLOAD["max_len"], n, args.query) == ("deadbeef", 1, 48, 64, 10_000_000, None):
                traffic = int(tj["dram_bytes_read"] + tj["dram_bytes_write"])   # from the committed ncu capture
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": "prefilter stage: k_sig_scan + k_window (+ tile rank/scan)", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                    "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": pf_ms,
                    "whole_step_frac": (alg_bytes / (ms / args.steps / 1e3) / 1e9 / peak),
                    "stage_ms_per_step": {"prefilter": pf_ms, "smith_waterman": stage["sw_ms"], "sort": stage["sort_ms"],
                                          "local_pipeline": stage["local_ms"], "all_gather_merge": stage["gather_merge_ms"],
                                          "d2h_slice": stage["d2h_ms"], "device_total": stage["total_ms"]}}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import cpu_baseline as cb
            sample = args.cpu_sample or n
            ccfg = cfg.with_(emulate_lanes=info["prefilter_lanes"])
            sd, so = data_np[: int(off_np[sample])], off_np[: sample + 1]
            threads = pick_threads(cb, patterns, ccfg, sd, so, trials=3)
            per = [cb.timed(patterns, ccfg, sd, so, threads, repeats=1)[0] for _ in range(7)]
            dt = float(np.median(per))
            cpu = {"value": sample / dt, "unit": "haystacks/s", "cores": threads, "kind": "port",
                   "value_best": sample / min(per),
                   "sample": f"first {sample} haystacks of the same list, median of 7 at the fastest of all/half/quarter "
                             f"of the {cb.host_threads()} host threads; {cb.describe()}, threaded like "
                             f"match_list_parallel; emulating the {info['prefilter_lanes']}-lane reference backend",
                   "calibration": calibration(cb, ccfg)}
        line = {"metric": "haystacks/sec", "value": value, "unit": "haystacks/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config_block(args, world, {"matches_per_step": int(n_matches),
                                                     "output": "ordered frz_match[] landed in ONE pinned host buffer "
                                                               "(shared by the ranks; every GPU copies its slice)",
                                                     "exchange": ("n/a (1 GPU)" if world == 1 else
                                                                  "all-gather of whole runs (FRZ_PARALLEL_EXCHANGE=allgather)"
                                                                  if os.environ.get("FRZ_PARALLEL_EXCHANGE") == "allgather" else
                                                                  "slice exchange: one grouped ncclSend/ncclRecv of exactly the ranges each rank copies out "
                                                                  "(value); all-gather of whole runs (value_device_out)"
                                                                  if os.environ.get("FRZ_PARALLEL_EXCHANGE") == "slices" or not comm.p2p_active() else
                                                                  "P2P placement: every GPU stores its matches at their merged positions in the peers' slice "
                                                                  "buffers over NVLink (k_place, cudaIpc-mapped peer memory), no NCCL kernel (value); "
                                                                  "all-gather of whole runs (value_device_out)" if comm.exchange_mode() == 2 else
                                                                  "direct placement: every GPU stores its matches at their merged positions straight into "
                                                                  "the shared pinned host buffer (k_place<DIRECT>, zero-copy over its own PCIe link; no "
                                                                  "NCCL kernel, no separate D2H copy) (value); all-gather of whole runs (value_device_out)"),
                                                     "emulated_reference_backend": info}),
                "clocks": clocks,
                "value_device_out": {"value": n * world * args.steps / (ms_dev / 1e3), "unit": "haystacks/s",
                                     "ms_per_step": ms_dev / args.steps, "what": "same step, merged list left in HBM"},
                "d2h_bytes_per_step": int(n_matches * 8),
                "e2e": {"value": e2e_value, "unit": "haystacks/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h_rank * world,
                        "steps": e2e_steps, "ms_per_step": e_ms / e2e_steps, "result_equals_resident_call": e2e_equal,
                        "streamed": os.environ.get("FRZ_E2E_STREAM", "1") != "0",
                        "input": f"Arrow {'Utf8 (int32' if off_e2e.dtype.itemsize == 4 else 'LargeUtf8 (int64'} offsets) "
                                 "value+offset buffers in pinned host memory, one shard per rank; H2D chunks overlap the pack kernels "
                                 "AND the match pipeline (tile ranges are matched as they land; only the sort waits for the last chunk)"},
                "gpu_launches": int(round(launches_per_step * args.steps)),
                "roofline": roofline, "cpu_baseline": cpu, "parity": parity}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_list["matches"])
        print(json.dumps(line), flush=True)
    barrier()
    comm.host_free(out_h)
    corpus.close()
    matcher.close()
    comm.close()
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and parity["mismatches"] != 0:
        raise SystemExit(f"bench.py: parity FAILED: {parity}")
    if e2e_equal is False:
        raise SystemExit("bench.py: the end-to-end call's list differs from the resident call's")


def main():
    args = parse_args()
    WORKLOAD.update(needle=args.needle, max_typos=args.max_typos, mu=args.mu, max_len=args.max_len)
    if args.impl == "reference":
        run_reference(args)
        return
    try:
        run_ours(args)
    except BaseException:
        # print the failing rank's traceback and leave at once: a rank that dies quietly would make its peers wait
        sys.stderr.write(f"[bench.py rank {os.environ.get('RANK', '0')}] failed:\n{traceback.format_exc()}\n")
        sys.stderr.flush()
        os._exit(1)


if __name__ == "__main__":
    main()
