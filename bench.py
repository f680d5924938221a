#!/usr/bin/env python
"""bench.py — kNN queries/sec of the knowledge-base search path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl ours|reference] [--no-extras]
                    [--dump-outputs DIR]
    python bench.py --gpus N --single-process      (no torchrun: ONE process, one rbk_group handle over N GPUs)

A "step" is one pass of the hot path (batched cosine scan + exact top-k) over one batch of
B synthetic queries against the resident synthetic corpus.  Workloads are BASELINE.json's
configs; the default is the one the target is quoted on (10M x 768 bf16, B=1024, k=16).
For N>1 (torchrun, one rank per GPU) the SAME corpus is row-sharded across the ranks
(strong scaling) and each step ends with the NCCL all-gather + merge of the per-rank lists.

Prints ONE JSON line (rank 0).  `value` = queries/s with the batch already resident in
HBM (steps are enqueued back to back, one synchronisation at the end of the timed region);
`e2e` = the same through the host-facing call (host query buffer in, host results out,
copies and one synchronisation per step inside the timed region).  `parity` = the first 64
queries of the batch re-answered by the CPU oracle over every rank's rows and compared
id for id and bit for bit.  `extra_workloads` carries the same measurements for the
hypothesis-branch batch (cfg5, every N) and the 50M x 1024 corpus (cfg4, N = 8).
`--impl reference` times the reference's CPU algorithm (oracle/, strict fp64 restatement;
Node is absent so the TypeScript itself cannot run) on the box's host cores on a bounded
sample of the same workload.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (N_docs, d, B, k, description)
    "cfg1": (10_000, 384, 1, 5, "10k x 384, B=1, k=5 (reference-scale, latency-bound)"),
    "cfg2": (1_000_000, 768, 256, 16, "1M x 768 bf16, B=256, k=16"),
    "cfg3": (10_000_000, 768, 1024, 16, "10M x 768 bf16, B=1024, k=16"),
    "cfg4": (50_000_000, 1024, 512, 32, "50M x 1024 bf16, B=512, k=32 (needs 8 GPUs)"),
    "cfg5": (5_000_000, 768, 256, 8, "5M x 768 bf16, 32 investigations x 8 queries, k=8"),
}
SEED = 0x5EED0003
GEN_CHUNK = 65536
PARITY_QUERIES = 64


def load_synth():
    """runbookai_b200/synth.py (numpy only) WITHOUT importing the package or its CUDA library."""
    spec = importlib.util.spec_from_file_location("rbk_synth", ROOT / "runbookai_b200" / "synth.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def dump_outputs(out_dir: str, arrays: dict):
    """--dump-outputs: `arrays` (what the timed call returned in its last step) as float64 DIR/<name>.npy.  Slots
    and counts are integers below 2**53, so float64 holds them exactly; the largest workload writes about 1 MB."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", np.asarray(a).astype(np.float64))


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return dict(hbm=j["hbm_gbs"], tf=j["bf16_tflops"], tf_sus=j.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm=6650.0, tf=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([time.monotonic()] + [x.strip() for x in line.split(",")])

    def window(self, t0: float, t1: float):
        """Keep only the samples taken inside [t0, t1] (monotonic clock); if the window was shorter than the
        sampling period, the sample nearest to it."""
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        if not inside and self.rows:
            inside = [min(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))]
        self.rows = inside

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        rows = [r[1:] for r in self.rows]   # drop the timestamp
        self.rows = rows
        sm = [float(r[1]) for r in rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        pw = [float(r[3]) for r in rows if len(r) >= 8 and r[3].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6),
                          ("sw_power_cap", 7)):
            if any(len(r) >= 8 and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": float(np.median(pw)) if pw else None, "reasons": reasons, "samples": len(sm)}


def gen_shard(ix, lo: int, hi: int, d: int, device):
    """Fill `ix` with global rows [lo, hi): N(0,1) rounded to bf16, generated on the device
    chunk by chunk from a per-chunk seed, so any sharding yields the same global corpus."""
    import torch
    c0 = lo // GEN_CHUNK
    c1 = -(-hi // GEN_CHUNK)
    g = torch.Generator(device=device)
    for c in range(c0, c1):
        g.manual_seed(SEED * 1_000_003 + c)
        t = torch.randn(GEN_CHUNK, d, device=device, generator=g, dtype=torch.float32).to(torch.bfloat16)
        a = max(lo, c * GEN_CHUNK) - c * GEN_CHUNK
        b = min(hi, (c + 1) * GEN_CHUNK) - c * GEN_CHUNK
        t = t[a:b].contiguous()
        torch.cuda.synchronize(device)
        ix.append_bf16_device(t.data_ptr(), b - a)
        del t


# ------------------------------------------------------------------------------------------ CPU legs (oracle/)
def cpu_allcores(oracle, corpus_bits, queries, k_fetch, threads):
    """ref-allcores: the literal per-pair loop (three accumulators per pair), rows split over the host threads."""
    t0 = time.perf_counter()
    oracle.search_batch_mt(corpus_bits, queries.astype(np.float64), k_fetch, None, n_threads=threads)
    return time.perf_counter() - t0


def cpu_one_thread(oracle, corpus_bits, queries, k_fetch):
    """ref-1T: the reference's real execution model - one thread, one query at a time, full stable sort
    (vector-store.ts:207-221 through oracle.search)."""
    t0 = time.perf_counter()
    for q in queries:
        oracle.search(corpus_bits, q.astype(np.float64), k_fetch, None)
    return time.perf_counter() - t0


def calibrate_sample(oracle, synth, d, k_fetch, threads, target_s, max_rows, max_q, min_rows=100_000):
    """(rows, queries) of the CPU sample so that one all-cores pass takes about target_s on THIS host."""
    probe_c = synth.random_corpus(50_000, d, SEED + 7)
    probe_q = synth.random_queries(8, d, SEED + 8)
    cpu_allcores(oracle, probe_c[:2000], probe_q, k_fetch, threads)            # page in, spin up
    dt = max(cpu_allcores(oracle, probe_c, probe_q, k_fetch, threads), 1e-4)
    pairs_per_s = 50_000 * 8 / dt
    want = pairs_per_s * target_s
    rows = int(min(max_rows, max(min_rows, want / max_q)))
    q = int(min(max_q, max(8, want / rows)))
    return rows, q, pairs_per_s


def run_reference(args, wl):
    """--impl reference: the reference's CPU algorithm on this box's cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    synth = load_synth()        # numpy only: the engine's CUDA library is never mapped on this arm
    import oracle
    oracle.build()
    n, d, B, k, desc = wl
    threads = oracle.host_threads()
    # >= 1M rows per step (or the whole corpus): small samples made this figure move 5x between boxes
    ns, bs, pps = calibrate_sample(oracle, synth, d, 2 * k, threads, target_s=3.0, max_rows=min(n, 1_000_000),
                                   max_q=B, min_rows=min(n, 1_000_000))
    corpus = synth.random_corpus(ns, d, SEED)
    queries = synth.random_queries(bs, d, SEED + 1)
    for _ in range(args.warmup):
        cpu_allcores(oracle, corpus, queries, 2 * k, threads)
    t_all, qps = 0.0, []
    for _ in range(args.steps):
        dt = cpu_allcores(oracle, corpus, queries, 2 * k, threads)
        qps.append(bs / dt * (ns / n))
        t_all += dt
    value = float(np.mean(qps))
    t1 = cpu_one_thread(oracle, corpus[:min(ns, 200_000)], queries[:4], 2 * k)
    v1 = 4 / t1 * (min(ns, 200_000) / n)
    sample = (f"{ns} rows x {bs} queries per step on {threads} host threads (cpu_count {os.cpu_count()}, "
              f"load {os.getloadavg()[0]:.1f}), literal 3-accumulator loop, scaled linearly to {n} rows")
    print(json.dumps({
        "impl": "reference", "metric": "knn_queries_per_sec", "value": value, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_all / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "n_docs": n, "dim": d, "batch": B, "k": k, "k_fetch": 2 * k},
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample,
                         "pairs_per_s": pps,
                         "ref_1T": {"value": v1, "unit": "queries/s", "cores": 1,
                                    "sample": f"{min(ns, 200_000)} rows x 4 queries, one thread, one query at a "
                                              f"time, full stable sort ({t1:.2f} s), scaled linearly to {n} rows"}},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------------ GPU legs
class Ctx:
    pass


def oracle_parity(ctx, ix, lo, hi, q_host_np, k_fetch, min_score, got, budget_s=150.0):
    """Re-answer the first PARITY_QUERIES queries with the CPU oracle over EVERY rank's rows (each rank reads its
    shard back from HBM chunk by chunk and runs the oracle on its share of the host threads; the per-rank lists are
    merged on rank 0) and compare with the engine's global answer `got` = (slots, scores, counts): ids identical,
    fp64 scores bit-identical."""
    import oracle
    import torch.distributed as dist
    oracle.build()
    nq = min(PARITY_QUERIES, q_host_np.shape[0])
    threads = max(1, oracle.host_threads() // ctx.world)
    q = q_host_np[:nq].astype(np.float64)
    n_local = hi - lo
    chunk = 1 << 19
    t0 = time.perf_counter()
    parts = []
    for i, r0 in enumerate(range(0, max(n_local, 1), chunk)):
        m = max(0, min(chunk, n_local - r0))
        if m > 0:
            rows = ix.read_rows_bf16(r0, m)
            parts.append(oracle.search_batch_verify(rows, q, k_fetch, min_score, n_threads=threads,
                                                    slot_base=lo + r0))
        if i == 0:
            # keep the default run inside a few minutes on a slow / shared host: fewer queries, never fewer rows
            # (every rank takes part in the decision, also one whose shard is empty)
            proj = (time.perf_counter() - t0) * (n_local / m) if m > 0 else 0.0
            nq_new = nq
            while proj * nq_new / nq > budget_s and nq_new > 8:
                nq_new //= 2
            if ctx.world > 1:
                import torch
                t = torch.tensor([nq_new], device=ctx.device)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                nq_new = int(t.item())
            if nq_new != nq:
                parts = [(p[0][:nq_new], p[1][:nq_new], p[2][:nq_new]) for p in parts]
                q, nq = q[:nq_new], nq_new
    local = oracle.merge_lists(parts, k_fetch) if parts else None
    secs = time.perf_counter() - t0
    if ctx.world > 1:
        gathered = [None] * ctx.world
        dist.all_gather_object(gathered, local)
        lists = [g for g in gathered if g is not None]
    else:
        lists = [local] if local is not None else []
    if ctx.rank != 0:
        return None
    es, ev, ec = oracle.merge_lists(lists, k_fetch)
    s, v, c = (np.asarray(a) for a in got)
    id_mis = score_mis = count_mis = 0
    max_abs = 0.0
    for b in range(nq):
        if c[b] != ec[b]:
            count_mis += 1
            continue
        m = ec[b]
        id_mis += int((s[b, :m] != es[b, :m]).sum())
        score_mis += int((v[b, :m] != ev[b, :m]).sum())
        if m:
            max_abs = max(max_abs, float(np.abs(v[b, :m] - ev[b, :m]).max()))
    return {"queries": int(nq), "rows_checked": int(ctx.n_total), "k_fetch": k_fetch,
            "id_mismatch": id_mis, "score_mismatch": score_mis, "count_mismatch": count_mis,
            "max_abs_score_diff": max_abs, "oracle": "oracle.search_batch_verify over every rank's rows, merged",
            "oracle_threads_per_rank": threads, "seconds": round(secs, 1)}


def run_workload(ctx, args, name, wl, main: bool, steps: int):
    """Build the (sharded) index of one workload, time it device-resident and end to end, check it."""
    import torch
    import torch.distributed as dist
    from runbookai_b200 import Index
    from runbookai_b200.sharded import ShardedSearcher, shard_bounds
    synth = ctx.synth
    n, d, B, k, desc = wl
    k_fetch = 2 * k   # the reference's over-fetch (vector-store.ts:221)
    world, rank, device = ctx.world, ctx.rank, ctx.device
    ctx.n_total = n
    lo, hi = shard_bounds(n, world, rank)
    ix = Index(d, device=ctx.local, capacity_hint=hi - lo)
    ix.set_slot_base(lo)
    gen_shard(ix, lo, hi, d, device)
    searcher = ShardedSearcher(ix)          # owns ONE stream for the engine, NCCL and the copies
    stream = searcher.stream
    q_np = synth.random_queries(B, d, SEED + 1)
    q_host = torch.from_numpy(q_np).pin_memory()
    with torch.cuda.stream(stream):
        q_dev = q_host.to(device, non_blocking=True)
    stream.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def max_over_ranks(x):
        t = torch.tensor([x], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- value: batch resident in HBM ----------------
    for _ in range(args.warmup):
        searcher.search_device(q_dev, k_fetch, args.min_score)
    barrier()
    st0 = ix.stats()
    t_region0 = time.monotonic()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # timing rule: inputs larger than L2, or L2 flushed between timed iterations.  A shard that could stay
    # (partly) resident in the 126 MB L2 is timed step by step with a 256 MB memset between steps (outside
    # the events); the large workloads stream far more than L2 per step and are timed as one region.
    l2_flush = 2.0 * (hi - lo) * d < 4 * 126e6
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=device) if l2_flush else None
    if l2_flush:
        ms = 0.0
        for _ in range(steps):
            with torch.cuda.stream(stream):
                flush_buf.zero_()
                ev0.record(stream)
                out = searcher.search_device_async(q_dev, k_fetch, args.min_score)
                ev1.record(stream)
            stream.synchronize()
            ms += ev0.elapsed_time(ev1)
        barrier()
    else:
        # steps are enqueued back to back (no host round trip inside a step); the exactness flags of every step
        # are accumulated on the device by the merge kernel and checked once after the region
        ev0.record(stream)
        for _ in range(steps):
            out = searcher.search_device_async(q_dev, k_fetch, args.min_score)
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
    flags = out[3]
    if main and rank == 0 and args.dump_outputs:
        # copied now: the same-box comparison below runs the search again into the same buffers
        dump_outputs(args.dump_outputs, {name: t.cpu().numpy() for name, t in zip(("slots", "scores", "counts", "flags"), out)})
    dirty = int(flags[-1].item()) - searcher._dirty_seen     # running count of unproven queries (merge kernel)
    searcher._dirty_seen += dirty
    st1 = ix.stats()
    n_scans = max(1, st1["scans_timed"] - st0["scans_timed"])
    scan_avg_ms = (st1["scan_ms_total"] - st0["scan_ms_total"]) / n_scans
    launches = (st1["kernel_launches"] - st0["kernel_launches"]) + steps + (steps if world > 1 else 0)
    # (index kernels: memset-free count of prep + scan + finalize) + merge kernel (+ NCCL all-gather kernel) per step
    ms = max_over_ranks(ms)
    clocks = None
    if main and rank == 0:
        t_region1 = time.monotonic()
        time.sleep(0.05)   # let the last sample of the region arrive
        ctx.sampler.window(t_region0, t_region1)
        clocks = ctx.sampler.stop()

    # ---------------- same box, same power state: the plain library GEMM of this shape ----------------
    same_box = None
    if main and world == 1 and not l2_flush and not args.no_cublas:
        try:
            same_box = cublas_same_box(ix, searcher, q_dev, k_fetch, args.min_score, hi - lo, d, B, steps)
        except Exception as e:   # a comparison must never cost the headline line
            same_box = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    # ---------------- e2e: host buffers through the public call ----------------
    def e2e_step():
        if world == 1:
            return ix.search(q_host.numpy(), k_fetch, args.min_score)[:3]      # rbk_index_search_f32: H2D + D2H inside
        return searcher.search(q_host, k_fetch, args.min_score, device)
    for _ in range(args.warmup):
        got = e2e_step()
    barrier()
    if l2_flush:
        e2e_s = 0.0
        for _ in range(steps):
            flush_buf.zero_()
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            got = e2e_step()                      # returns host results: the call has synchronised
            e2e_s += time.perf_counter() - t0
        barrier()
    else:
        t0 = time.perf_counter()
        for _ in range(steps):
            got = e2e_step()
        barrier()
        e2e_s = time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_s)
    st2 = ix.stats()

    # ---------------- parity: the same batch against the CPU oracle ----------------
    parity = None
    if not args.no_parity:
        parity = oracle_parity(ctx, ix, lo, hi, q_np, k_fetch, args.min_score, got)

    res = None
    if rank == 0:
        pk = ctx.pk
        n_local = hi - lo
        flops = 2.0 * B * n_local * d          # SURVEY §8d: dot products only
        bytes_ = 2.0 * n_local * d + 2.0 * B * d + 8.0 * B * k_fetch
        tensor_bound = B > pk["tf"] * 1e12 / (pk["hbm"] * 1e9)   # arithmetic intensity ~ B flop/byte vs ridge
        tf = flops / (scan_avg_ms * 1e-3) / 1e12
        gbs = bytes_ / (scan_avg_ms * 1e-3) / 1e9
        # ONE peak kind at every N: the burst figures of MEASURED_PEAKS.json (the sustained tensor peak alongside)
        if tensor_bound:
            roof = {"bound": "tensor", "achieved": tf, "peak": pk["tf"], "unit": "TFLOP/s", "frac": tf / pk["tf"],
                    "peak_kind": "burst", "frac_of_sustained": tf / pk["tf_sus"] if pk["tf_sus"] else None,
                    "hbm_gbs": gbs}
        else:
            roof = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                    "peak_kind": "burst", "tflops": tf, "frac_of_tensor_burst": tf / pk["tf"]}
        roof.update({"kernel": ("scan2_kernel: CTA-pair tcgen05 cta_group::2 QxC^T + fused top-k'" if B > 128
                                else "scan_kernel: tcgen05 QxC^T + fused top-k'"), "kernel_ms": scan_avg_ms,
                     "algorithmic_bytes": bytes_, "algorithmic_flops": flops, "peak_source": pk["src"],
                     # dram bytes per launch of the committed ncu --set full capture of this workload on ONE GPU;
                     # not measured by this run, and not meaningful for a 1/N shard
                     "traffic": _profiled_traffic(name) if world == 1 else None})
        res = {
            "value": B * steps / (ms * 1e-3), "unit": "queries/s", "steps": steps, "ms_per_step": ms / steps,
            "config": {"workload": desc + (" [REDUCED rows: debug run]" if ctx.reduced else ""), "n_docs": n, "dim": d,
                       "batch": B, "k": k, "k_fetch": k_fetch, "min_score": args.min_score,
                       "parallelism": (f"rows sharded over {world} GPUs, one NCCL all-gather of the packed top-k "
                                       "blocks + merge kernel per step" if world > 1 else "1 GPU"),
                       "pipelining": ("steps timed one by one (L2 flush between them)" if l2_flush else
                                      "value: steps enqueued back to back, exactness flags checked after the "
                                      "region; e2e: one host synchronisation per step"),
                       "l2": (f"corpus {2.0 * n_local * d / 1e6:.0f} MB per GPU could stay in the 126 MB L2: L2 flushed "
                              "(256 MB memset) before every timed step" if l2_flush else
                              f"corpus {2.0 * n_local * d / 1e9:.1f} GB per GPU >> 126 MB L2, no flush needed"),
                       "unproven_queries_in_timed_region": int(dirty),
                       "fallback_queries": int(st2["fallback_queries"]), "retry_batches": int(st2["retry_batches"])},
            "e2e": {"value": B * steps / e2e_s, "unit": "queries/s", "h2d_bytes_per_step": B * d * 4,
                    "d2h_bytes_per_step": B * k_fetch * 16 + B * 8, "ms_per_step": e2e_s / steps * 1e3},
            "gpu_launches": int(launches),
            "roofline": roof,
            "parity": parity,
        }
        if clocks is not None:
            res["clocks"] = clocks
        if same_box is not None:
            roof["same_box_cublas"] = same_box
        if main and not args.no_cpu_baseline and world == 1:
            res["cpu_baseline"] = cpu_baseline(ctx, ix, n, n_local, d, B, k_fetch, q_np)
    ix.close()
    del searcher, flush_buf
    torch.cuda.empty_cache()
    return res


def run_group(args, name, wl, pk, synth, reduced):
    """`--single-process`: the deployment one Node process would use - ONE host process, one `rbk_group` handle over
    `--gpus` devices (include/rbk_knn.h; per-GPU scans, one ncclAllGather, merge on the first device and one
    synchronisation inside every call).  The group's search takes host queries and returns host results, so the
    number measured here is the end-to-end one; the corpus is the same global corpus as the torchrun mode
    (generated on GPU 0 chunk by chunk, staged through host memory, dealt out by the library)."""
    import torch
    import oracle
    from runbookai_b200 import Group
    n, d, B, k, desc = wl
    k_fetch = 2 * k
    G = args.gpus
    dev0 = torch.device("cuda", 0)
    grp = Group(d, list(range(G)), capacity_hint=n)
    host = np.empty((n, d), dtype=np.uint16)
    gen = torch.Generator(device=dev0)
    t0 = time.perf_counter()
    for c in range(-(-n // GEN_CHUNK)):
        gen.manual_seed(SEED * 1_000_003 + c)
        t = torch.randn(GEN_CHUNK, d, device=dev0, generator=gen, dtype=torch.float32).to(torch.bfloat16)
        m = min(GEN_CHUNK, n - c * GEN_CHUNK)
        host[c * GEN_CHUNK:c * GEN_CHUNK + m] = t[:m].view(torch.int16).cpu().numpy().view(np.uint16)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    for r0 in range(0, n, 1 << 20):
        grp.append_bf16(host[r0:r0 + (1 << 20)])
    t_load = time.perf_counter() - t0
    q_np = synth.random_queries(B, d, SEED + 1)
    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        got = grp.search(q_np, k_fetch, args.min_score)
    st0 = grp.stats()
    t_r0 = time.monotonic()
    t0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(args.steps):
        got = grp.search(q_np, k_fetch, args.min_score)
        dev_ms += got[3]
    dt = time.perf_counter() - t0
    t_r1 = time.monotonic()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("slots", "scores", "counts"), got[:3])))
    st1 = grp.stats()
    time.sleep(0.05)
    sampler.window(t_r0, t_r1)
    clocks = sampler.stop()
    # parity: the first 64 queries against the oracle over all rows (host copy of the corpus)
    oracle.build()
    nq = min(PARITY_QUERIES, B)
    qd = q_np[:nq].astype(np.float64)
    t0 = time.perf_counter()
    parts = [oracle.search_batch_verify(host[r0:r0 + (1 << 19)], qd, k_fetch, args.min_score, slot_base=r0)
             for r0 in range(0, n, 1 << 19)]
    es, ev, ec = oracle.merge_lists(parts, k_fetch)
    s, v, c = got[0], got[1], got[2]
    id_mis = score_mis = count_mis = 0
    for b in range(nq):
        if c[b] != ec[b]:
            count_mis += 1
            continue
        m = ec[b]
        id_mis += int((s[b, :m] != es[b, :m]).sum())
        score_mis += int((v[b, :m] != ev[b, :m]).sum())
    per0, per1 = st0["per_device"], st1["per_device"]
    scan_ms = [(b_["scan_ms_total"] - a_["scan_ms_total"]) / max(1, b_["scans_timed"] - a_["scans_timed"])
               for a_, b_ in zip(per0, per1)]
    flops = 2.0 * B * n * d / G
    e2e = B * args.steps / dt
    out = {"metric": "knn_queries_per_sec", "value": e2e, "unit": "queries/s", "n_gpus": G, "steps": args.steps,
           "warmup": max(args.warmup, 3), "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": desc + (" [REDUCED rows: debug run]" if reduced else ""), "n_docs": n, "dim": d,
                      "batch": B, "k": k, "k_fetch": k_fetch, "min_score": args.min_score,
                      "parallelism": f"ONE process, rbk_group over {G} GPUs: rows dealt out in 4096-row blocks, per-GPU "
                                     "scans + one ncclAllGather + merge inside rbk_group_search_f32",
                      "value_is": "end to end (host queries in, host results out): the group call has no "
                                  "device-resident variant", "gen_s": round(t_gen, 1), "load_s": round(t_load, 1),
                      "redone_batches": st1["redone_batches"], "fallback_queries": st1["fallback_queries"]},
           "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": B * d * 4 * G,
                   "d2h_bytes_per_step": B * k_fetch * 16 + B * 4, "ms_per_step": dt / args.steps * 1e3,
                   "device_ms_per_step": dev_ms / args.steps},
           "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"] + args.steps * (1 + G)),
           "roofline": {"bound": "tensor" if B > pk["tf"] * 1e12 / (pk["hbm"] * 1e9) else "hbm",
                        "kernel_ms_per_device": scan_ms, "unit": "TFLOP/s", "peak": pk["tf"], "peak_kind": "burst",
                        "achieved": flops / (max(scan_ms) * 1e-3) / 1e12,
                        "frac": flops / (max(scan_ms) * 1e-3) / 1e12 / pk["tf"], "traffic": None},
           "parity": {"queries": nq, "rows_checked": n, "k_fetch": k_fetch, "id_mismatch": id_mis,
                      "score_mismatch": score_mis, "count_mismatch": count_mis,
                      "seconds": round(time.perf_counter() - t0, 1)},
           "clocks": clocks}
    grp.close()
    print(json.dumps(out), flush=True)


def cublas_same_box(ix, searcher, q_dev, k_fetch, min_score, n_local, d, B, steps):
    """What the library GEMM of the same shape does on THIS box in THIS power state: torch.matmul (cuBLAS, bf16 in,
    fp32 accumulate, bf16 out) of the B x d query block against n_local x d rows, in 1M-row pieces, interleaved with
    the scan in two rounds of `steps` passes each.  It only computes the score matrix (and writes it: 2*B bytes per
    row, which the scan never does) - no threshold, no top-k, no exact re-rank - so it is the roof a power-capped
    scan of this shape can be held against when boxes differ by 18 % on the identical kernel.  Measurement only:
    nothing the product runs goes through it."""
    import torch
    device, stream = q_dev.device, searcher.stream
    piece = -(-n_local // -(-n_local // (1 << 20)))      # ~1M-row pieces of equal size
    with torch.cuda.stream(stream):
        c = torch.randn(piece, d, device=device, dtype=torch.float32).to(torch.bfloat16)
        qb = q_dev.to(torch.bfloat16)
        out = torch.empty(B, piece, device=device, dtype=torch.bfloat16)
        full, rest = divmod(n_local, piece)

        def gemm_pass():
            for _ in range(full):
                torch.matmul(qb, c.t(), out=out)
            if rest:
                torch.matmul(qb, c[:rest].t(), out=out[:, :rest])
        gemm_pass()
        # the same flops as ONE GEMM with a `full` times deeper K: 1/full of the output bytes, cuBLAS at its best on
        # this box (what MEASURED_PEAKS.json's sustained figure measures elsewhere)
        deep = full >= 2 and rest == 0 and 2.0 * piece * d * full < 40e9
        if deep:
            c2 = torch.randn(piece, d * full, device=device, dtype=torch.bfloat16)
            q2 = torch.randn(B, d * full, device=device, dtype=torch.bfloat16)
            torch.matmul(q2, c2.t(), out=out)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
        st0 = ix.stats()
        e[0].record(stream)
        for r in range(2):
            for _ in range(steps):
                flags = searcher.search_device_async(q_dev, k_fetch, min_score)[3]
            e[2 * r + 1].record(stream)
            for _ in range(steps):
                gemm_pass()
            e[2 * r + 2].record(stream)
        if deep:
            for _ in range(steps):
                torch.matmul(q2, c2.t(), out=out)
            e[5].record(stream)
            for _ in range(steps):
                flags = searcher.search_device_async(q_dev, k_fetch, min_score)[3]
            e[6].record(stream)
    stream.synchronize()
    searcher._dirty_seen = int(flags[-1].item())
    st1 = ix.stats()
    step_ms = [e[0].elapsed_time(e[1]) / steps, e[2].elapsed_time(e[3]) / steps]
    gemm_ms = [e[1].elapsed_time(e[2]) / steps, e[3].elapsed_time(e[4]) / steps]
    scan_ms = (st1["scan_ms_total"] - st0["scan_ms_total"]) / max(1, st1["scans_timed"] - st0["scans_timed"])
    flops = 2.0 * B * n_local * d
    deep_ms = e[4].elapsed_time(e[5]) / steps if deep else None
    if deep:
        step_ms.append(e[5].elapsed_time(e[6]) / steps)
        del c2, q2
    del c, out, qb
    return {"gemm_ms": gemm_ms, "gemm_deep_k_ms": deep_ms,
            "gemm_deep_k_tflops": flops / (deep_ms * 1e-3) / 1e12 if deep else None, "search_step_ms": step_ms, "scan_kernel_ms": scan_ms,
            "gemm_tflops": flops / (min(gemm_ms) * 1e-3) / 1e12, "scan_tflops": flops / (scan_ms * 1e-3) / 1e12,
            "scan_over_gemm": min(gemm_ms) / scan_ms,
            "what": f"torch.matmul bf16 [{B}x{d}] x [{d}x{piece}] -> bf16, {full + (1 if rest else 0)} pieces per pass; "
                    f"2 rounds of {steps} search steps then {steps} GEMM passes, back to back on one stream"}


def cpu_baseline(ctx, ix, n, n_local, d, B, k_fetch, q_np):
    """The oracle timed on this box's host cores on a bounded sample of the same workload: rows read back from the
    index, the literal per-pair loop.  Both modes SURVEY §8d names: all cores, and one thread (the reference's
    real execution model: a single JS thread, one query at a time, full stable sort)."""
    import oracle
    oracle.build()
    threads = oracle.host_threads()
    ns, bs, pps = calibrate_sample(oracle, ctx.synth, d, k_fetch, threads, target_s=10.0,
                                   max_rows=min(n_local, 2_000_000), max_q=min(B, 64))
    ns = min(ns, n_local)
    bs = min(bs, B)
    rows = ix.read_rows_bf16(0, ns)
    dt = cpu_allcores(oracle, rows, q_np[:bs], k_fetch, threads)
    v = bs / dt * (ns / n)
    n1 = min(ns, 200_000)
    b1 = min(bs, 8)
    t1 = cpu_one_thread(oracle, rows[:n1], q_np[:b1], k_fetch)
    return {"value": v, "unit": "queries/s", "cores": threads, "kind": "port",
            "sample": (f"first {ns} rows x {bs} queries on {threads} host threads (cpu_count {os.cpu_count()}, load "
                       f"{os.getloadavg()[0]:.1f}; {dt:.2f} s), literal 3-accumulator loop, scaled linearly to {n} rows"),
            "ref_1T": {"value": b1 / t1 * (n1 / n), "unit": "queries/s", "cores": 1,
                       "sample": f"first {n1} rows x {b1} queries, one thread, one query at a time, full stable "
                                 f"sort ({t1:.2f} s), scaled linearly to {n} rows"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("RBK_BENCH_WORKLOAD", "cfg3"), choices=sorted(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="override N_docs (debug only; marks the run reduced)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check (debug only)")
    ap.add_argument("--no-cublas", action="store_true", help="skip the same-box library-GEMM comparison")
    ap.add_argument("--single-process", action="store_true",
                    help="ONE process, one rbk_group handle over --gpus devices (no torchrun): the deployment a single "
                         "Node process would use")
    ap.add_argument("--no-extras", action="store_true",
                    help="only the main workload (default: also cfg5 at every N and cfg4 at N=8, in `extra_workloads`)")
    ap.add_argument("--min-score", type=float, default=None,
                    help="cosine threshold (the reference's default is 0.5); default: none (-inf), the headline runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed search returned in its last step (slots, "
                         "scores, counts and, on the device-resident path, flags of the main workload) as "
                         "float64 DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference leg keeps no results")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = list(WORKLOADS[args.workload])
    reduced = bool(args.rows)
    if args.rows:
        wl[0] = args.rows
    if args.impl == "reference":
        run_reference(args, wl)
        return

    import torch
    import torch.distributed as dist

    ctx = Ctx()
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.rank = int(os.environ.get("RANK", "0"))
    ctx.local = int(os.environ.get("LOCAL_RANK", "0"))
    ctx.reduced = reduced
    ctx.synth = load_synth()
    ctx.pk = peaks()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this engine has no CPU path")
    if args.single_process:
        assert ctx.world == 1, "--single-process is not launched with torchrun"
        run_group(args, args.workload, wl, ctx.pk, ctx.synth, reduced)
        return
    torch.cuda.set_device(ctx.local)
    ctx.device = torch.device("cuda", ctx.local)
    if ctx.world > 1:
        dist.init_process_group("nccl", device_id=ctx.device)
    assert ctx.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={ctx.world} (launch with torchrun for N>1)"
    ctx.sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        ctx.sampler.start()   # nvidia-smi takes a second to start: launch it now, keep only the timed region's samples

    res = run_workload(ctx, args, args.workload, wl, main=True, steps=args.steps)
    extras = {}
    if not args.no_extras and not reduced and args.workload == "cfg3":
        names = ["cfg5"] + (["cfg4"] if ctx.world == 8 else [])
        for nm in names:
            try:
                extras[nm] = run_workload(ctx, args, nm, list(WORKLOADS[nm]), main=False, steps=args.steps)
            except Exception as e:   # an extra must never cost the headline line
                extras[nm] = {"error": f"{type(e).__name__}: {e}"}
    if ctx.rank == 0:
        n, d, B, k, desc = wl
        out = {"metric": "knn_queries_per_sec", "value": res["value"], "unit": "queries/s", "n_gpus": ctx.world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
               "data": "synthetic"}
        for key in ("config", "clocks", "e2e", "gpu_launches", "roofline", "parity", "cpu_baseline"):
            if key in res:
                out[key] = res[key]
        if extras:
            out["extra_workloads"] = extras
        print(json.dumps(out), flush=True)
    if ctx.world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _profiled_traffic(workload: str):
    """dram bytes per scan launch from the committed ncu --set full capture, if any."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        return json.loads(p.read_text()).get(workload)
    return None


if __name__ == "__main__":
    main()
