#!/usr/bin/env python
"""bench.py -- headline benchmark of the yams-b200 hot path (contract: see the task statement).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle/_ref or port)

Workloads (BASELINE.json):
  knn    C2: 10M x 768 fp16 corpus per GPU, 1024-query batch, cosine top-10  -> queries/s (headline)
         C4: at 8 GPUs the corpus is the named 100M x 768 (12.5M rows per GPU), value in 10M-row-equivalent queries/s
  ingest C3: 64 GiB synthetic byte stream per GPU, CDC (YAMS defaults) + SHA-256 per chunk -> GB/s
One JSON line is printed by rank 0; the ingest workload is reported in the "ingest" sub-object.
Multi-GPU: rows (knn) / independent streams (ingest) are sharded per rank -- weak scaling; the knn path all-gathers ONE
packed record of per-shard partial top-k (NCCL, 12*Q*k bytes per rank) and merges on the device, double-buffered so that
gather + merge of batch i overlap the scan of batch i+1.
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

METRIC = "queries/sec @10M x 768 brute-force kNN (cosine top-10)"
REF_ROWS = 10_000_000          # the row count the metric is quoted on


def load_traffic():
    """DRAM bytes per launch of the dominant kernels, copied from the committed ncu --set full captures."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "sm_mhz_min": min(sm) if sm else None, "power_w_median": float(np.median(pw)) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# reference / CPU arm (the ONLY code in this file that executes oracle/; never inside a GPU-timed region)
# ---------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm uses: every core of the box, whatever OMP_NUM_THREADS a launcher exported (torchrun sets 1)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except Exception:
        pass
    return n


def load_oracle(threads):
    """Imports the checker with its OpenMP runtime sized explicitly; returns (module, threads the runtime reports)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.pop("OMP_THREAD_LIMIT", None)
    from oracle import oracle as O
    O.build()
    O.lib()
    actual = threads
    try:
        import ctypes
        gomp = ctypes.CDLL("libgomp.so.1")
        gomp.omp_set_num_threads(int(threads))
        actual = int(gomp.omp_get_max_threads())
    except Exception:
        pass
    return O, actual


def median_of(fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def cpu_knn(O, threads, d, k, full_rows, kind, budget_s=8.0):
    """The CPU exact scan on a bounded sample (one warm-up + median of 3), extrapolated linearly to full_rows.
    Two arms, as BASELINE.md §3 lists them: the sqlite-vec-cpp batch operator (AVX, float accumulate) when oracle/_ref
    exists, and the R1 restatement of bruteForceSearchUnlocked (double accumulate)."""
    rows_sample = 500_000
    nq_sample = max(8, threads)
    rows32 = O.gen_rows_f32(42, 0, rows_sample, d)
    rows16 = O.f16_from_float(rows32).reshape(rows_sample, d)
    q = O.gen_rows_f32(43, 0, nq_sample, d)
    arms = {}
    if kind == "reference":
        R = O.ref()
        rows_up = O.f16_to_float(rows16).reshape(rows_sample, d)     # same fp16 values, upcast (the reference stores fp32)
        out_i = np.empty((nq_sample, k), dtype=np.uint64)
        out_d = np.empty((nq_sample, k), dtype=np.float32)

        def run_avx():
            R.ref_batch_top_k_queries(O._p(q, O.f32p), nq_sample, O._p(rows_up, O.f32p), rows_sample, d, O.METRIC_COSINE, k,
                                      O._p(out_i, O.u64p), O._p(out_d, O.f32p))
        dt, ts = median_of(run_avx)
        arms["avx_f32"] = {"queries_per_s": nq_sample / dt * rows_sample / full_rows, "sample_s": ts, "dtype": "f32 accumulate (AVX)",
                           "what": "sqlite-vec-cpp batch_distance_contiguous<cosine> + partial_sort compiled from /root/reference (oracle/_ref)"}
    del rows32

    def run_r1():
        O.exact_scan_cosine_batch(rows16, q, k, -1.0)
    dt, ts = median_of(run_r1)
    arms["r1_f64"] = {"queries_per_s": nq_sample / dt * rows_sample / full_rows, "sample_s": ts, "dtype": "f64 accumulate (scalar)",
                      "what": "oracle restatement of bruteForceSearchUnlocked (sqlite_vec_backend.cpp:4203-4331)"}
    head = "avx_f32" if "avx_f32" in arms else "r1_f64"    # the FASTER reference arm is the headline denominator
    if arms["r1_f64"]["queries_per_s"] > arms[head]["queries_per_s"]:
        head = "r1_f64"
    sample = (f"{nq_sample} queries x {rows_sample} rows x {d} (fp16 values), OpenMP over queries with {threads} threads, one warm-up + median of 3 "
              f"({', '.join('%.2f' % t for t in arms[head]['sample_s'])} s), extrapolated linearly to {full_rows} rows; headline arm: {head}")
    return arms[head]["queries_per_s"], arms, head, sample


def cpu_ingest(O, threads, kind):
    nbytes = int(min(8 << 30, max(1 << 30, threads * (64 << 20))))
    data = O.gen_bytes(12345, 0, nbytes)
    cfg = O.default_config()
    if kind == "reference":
        # the reference parallelises ingest only across files: one chunker per 64 MiB "file"
        from concurrent.futures import ThreadPoolExecutor
        piece = 64 << 20
        parts = [data[i:i + piece] for i in range(0, nbytes, piece)]

        def run():
            with ThreadPoolExecutor(max_workers=threads) as ex:
                list(ex.map(lambda p: O.ref_chunk(p, cfg, variant=1), parts))   # RabinChunker::chunkDataLazy (the fast arm)
        what = f"reference RabinChunker::chunkDataLazy + OpenSSL SHA-256 (oracle/_ref), {threads} threads over 64 MiB files"
    else:
        def run():
            O.cdc_chunk(data, cfg)
        what = f"oracle port: sequential CDC (1 thread) + OpenMP SHA-256 ({threads} threads)"
    dt, ts = median_of(run)
    return nbytes / dt / 1e9, f"{what}; {nbytes >> 20} MiB, one warm-up + median of 3 ({', '.join('%.2f' % t for t in ts)} s)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    O, omp_threads = load_oracle(threads)
    kind = "reference" if O.ref_available() else "port"
    value, arms, head, sample = cpu_knn(O, omp_threads, args.dim, args.k, args.rows, kind)
    ing_v, ing_sample = cpu_ingest(O, omp_threads, kind)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * args.queries / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": arms[head]["dtype"], "data": "synthetic",
        "config": knn_config(args, 1, args.rows),
        "cpu_baseline": {"value": value, "unit": "queries/s", "cores": omp_threads, "kind": kind, "sample": sample,
                         "omp_threads": omp_threads, "host_cpus": os.cpu_count(), "arms": arms},
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ingest": {"metric": "GB/s SHA-256+CDC", "value": ing_v, "unit": "GB/s",
                   "cpu_baseline": {"value": ing_v, "unit": "GB/s", "cores": omp_threads, "kind": kind, "sample": ing_sample}},
    }
    print(json.dumps(line))


def knn_config(args, world, rows_per_gpu):
    esz = 4 if args.corpus_dtype == "f32" else 2
    name = "C4" if world == 8 and rows_per_gpu * world == 100_000_000 else "C2"
    total = rows_per_gpu * world
    return {"workload": (f"{name}: {total} x {args.dim} {'fp32' if esz == 4 else 'fp16'} rows"
                         + (f" row-sharded over {world} GPUs ({rows_per_gpu} per GPU)" if world > 1 else "")
                         + f", {args.queries}-query batch, cosine top-{args.k}"),
            "rows_per_gpu": rows_per_gpu, "rows_total": total, "dim": args.dim, "queries": args.queries, "k": args.k,
            "parallelism": f"row-shard x{world}, one packed NCCL all-gather of partial top-k per batch" if world > 1 else "single GPU",
            "value_normalisation": f"queries/s x rows_total / {REF_ROWS} (the metric is quoted per 10M rows)",
            "l2_policy": f"corpus ({rows_per_gpu * args.dim * esz / 1e9:.1f} GB per GPU) >> 126 MB L2: every step re-streams it from HBM"}


def count_kernel_launches(fn):
    """Kernels one call of fn launches, counted by CUPTI through torch.profiler (None if the profiler is unavailable)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        from torch.autograd import DeviceType
        n = sum(1 for e in prof.events() if e.device_type == DeviceType.CUDA and not e.name.lower().startswith(("memcpy", "memset")))
        return n or None
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="both", choices=["both", "knn", "ingest"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (default: 10M; 12.5M at 8 GPUs = config C4 as named)")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--corpus-dtype", default="f16", choices=["f16", "f32"],
                    help="f16 = BASELINE config C2 (default); f32 = the reference's BLOB layout (tf32 tensor-core engine)")
    ap.add_argument("--ingest-gib", type=float, default=64.0)
    ap.add_argument("--e2e-ingest-gib", type=float, default=4.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the side measurements (q_sweep, c5, l2, small files, digest set)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.rows == 0:
        args.rows = 12_500_000 if (world == 8 and args.impl == "ours") else REF_ROWS
    if args.impl == "reference":
        args.rows = REF_ROWS
        return run_reference(args)

    import torch
    import yams_b200 as Y
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    assert Y.plugin_init({"device": local}) == 0, Y.health()
    peaks = load_peaks()

    def barrier_sync():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def over_ranks(x):
        """(min, max) of a per-rank scalar"""
        if not dist:
            return [x, x]
        t = torch.tensor([x, -x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(-t[1].item()), float(t[0].item())]

    out = {}
    W, K = max(args.warmup, 0), args.steps
    sampler = ClockSampler(local)
    side = {}          # work for after the GPU-timed regions (checker / CPU legs)
    dumps = {}         # --dump-outputs: name -> array

    # ------------------------------------------------------------------ knn -------------------------
    if args.workload in ("both", "knn"):
        n, d, nq, k = args.rows, args.dim, args.queries, args.k
        total_rows = n * world
        f32 = args.corpus_dtype == "f32"
        esz = 4 if f32 else 2
        corpus = Y.Corpus(d, Y.F32 if f32 else Y.F16, Y.COSINE, capacity_hint=n)
        step_rows = 1_000_000
        for r0 in range(0, n, step_rows):
            corpus.append_synthetic(42, rank * n + r0, min(step_rows, n - r0))
        q_dev = torch.empty((nq, d), dtype=torch.float32, device="cuda")
        Y.synth_rows_device(43, 0, nq, d, q_dev.data_ptr())          # the library's own generator (not the checker's)
        q_host = q_dev.cpu().pin_memory()
        S = torch.cuda.ExternalStream(corpus.stream)                 # the stream the scan is enqueued on
        comm = torch.cuda.Stream() if dist else None                 # gather + merge run here, behind the scan
        rec = nq * k * 12                                            # one rank's packed partial top-k record (SURVEY §8e)
        part = [torch.empty(rec, dtype=torch.uint8, device="cuda") for _ in range(2)]
        if dist:
            allp = [torch.empty(world * rec, dtype=torch.uint8, device="cuda") for _ in range(2)]
            fin_r = [torch.empty((nq, k), dtype=torch.int64, device="cuda") for _ in range(2)]
            fin_s = [torch.empty((nq, k), dtype=torch.float32, device="cuda") for _ in range(2)]
            ev_scan = [torch.cuda.Event() for _ in range(2)]
            ev_done = [torch.cuda.Event() for _ in range(2)]
            ev_c = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]   # per timed step: gather start / end, merge end
        gather_ms, merge_ms = [], []

        def scan_into(b, q_ptr):
            base = part[b].data_ptr()
            corpus.search_device(q_ptr, nq, k, -1.0, base, base + nq * k * 8)   # packed: [rowids][scores]; no host sync

        def gather_merge(b, evs=None):
            ev_scan[b].record(S)
            with torch.cuda.stream(comm):
                comm.wait_event(ev_scan[b])
                if evs:
                    evs[0].record(comm)
                dist.all_gather_into_tensor(allp[b], part[b])           # ONE packed all-gather per batch
                if evs:
                    evs[1].record(comm)
                corpus.merge_packed_device(allp[b].data_ptr(), world, nq, k, fin_r[b].data_ptr(), fin_s[b].data_ptr(), 0, comm.cuda_stream)
                if evs:
                    evs[2].record(comm)
                ev_done[b].record(comm)

        def step_resident(i, timed=False):
            b = i & 1
            if dist and i >= 2:
                S.wait_event(ev_done[b])                                # buffer b is free again (batch i-2 merged); device-side wait only
            scan_into(b, q_dev.data_ptr())
            if dist:
                gather_merge(b, ev_c[i] if timed else None)

        for i in range(max(W, 2)):
            step_resident(i)
        barrier_sync()
        sampler.start()                                                 # every rank samples its own GPU
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(S)
        for i in range(K):
            step_resident(i, timed=True)
        if dist:
            S.wait_stream(comm)
        e1.record(S)
        barrier_sync()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        if args.dump_outputs and rank == 0:       # the top-k the last timed step handed to its caller (merged over ranks at N > 1)
            b = (K - 1) & 1
            if dist:
                last_r, last_s = fin_r[b].cpu().numpy(), fin_s[b].cpu().numpy()
            else:
                packed = part[b].cpu().numpy()
                last_r, last_s = packed[:nq * k * 8].view(np.int64), packed[nq * k * 8:].view(np.float32)
            dumps["knn_rowids"] = last_r.reshape(nq, k).astype(np.float64)
            dumps["knn_scores"] = last_s.reshape(nq, k).astype(np.float32)
        if dist:
            gather_ms = [ev_c[i][0].elapsed_time(ev_c[i][1]) for i in range(K)]
            merge_ms = [ev_c[i][1].elapsed_time(ev_c[i][2]) for i in range(K)]
        resolved = corpus.search_device_finish()                      # status of the last batch: invalid queries / certificate failures
        tm = corpus.last_timings()
        ms_step = ms_total / K
        qps = nq / (ms_step / 1e3) * (total_rows / REF_ROWS)
        scan_ms_ranks = over_ranks(tm["scan_kernel_ms"] or tm["stage1_ms"])
        # ---- e2e through the public host API: pinned host queries in, host results out, every step ----
        q_dev2 = torch.empty_like(q_dev)

        def step_e2e():
            if not dist:
                return corpus.search(q_host.numpy(), k, threshold=-1.0)
            with torch.cuda.stream(S):   # H2D of the step's queries on the stream the scan runs on
                q_dev2.copy_(q_host, non_blocking=True)
            scan_into(0, q_dev2.data_ptr())
            corpus.search_device_finish()                              # a host-visible result must be a finished one
            gather_merge(0)
            with torch.cuda.stream(comm):
                r_host, s_host = fin_r[0].to("cpu", non_blocking=True), fin_s[0].to("cpu", non_blocking=True)
            comm.synchronize()
            return r_host.numpy(), s_host.numpy()

        step_e2e()
        barrier_sync()
        t0 = time.perf_counter()
        for _ in range(K):
            res = step_e2e()
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / K
        tm_e2e = corpus.last_timings()                                  # device timings of the last end-to-end call
        clocks_mine = sampler.stop()
        clocks = clocks_mine if rank == 0 else None
        e2e_qps = nq / (e2e_ms / 1e3) * (total_rows / REF_ROWS)
        launches_per_step = count_kernel_launches(lambda: (scan_into(0, q_dev.data_ptr()), corpus.sync())) if rank == 0 else None
        if dist:
            barrier_sync()

        # ---- parity of what was just timed, at EVERY N: the first 16 queries against the library's exhaustive pass over the
        #      full sharded corpus (exact score of every row + global sort on each shard, same all-gather + merge) ----
        parity_full = None
        if not args.no_parity:
            nchk = min(16, nq)
            fast_r, fast_s = res[0][:nchk].copy(), res[1][:nchk].copy()
            ex = corpus.search_exhaustive(q_host.numpy()[:nchk], k, threshold=-1.0)
            if dist:
                pr = torch.from_numpy(ex[0]).cuda()
                ps = torch.from_numpy(ex[1]).cuda()
                ar = torch.empty((world, nchk, k), dtype=torch.int64, device="cuda")
                as_ = torch.empty((world, nchk, k), dtype=torch.float32, device="cuda")
                dist.all_gather_into_tensor(ar, pr)
                dist.all_gather_into_tensor(as_, ps)
                mr = torch.empty((nchk, k), dtype=torch.int64, device="cuda")
                msc = torch.empty((nchk, k), dtype=torch.float32, device="cuda")
                torch.cuda.synchronize()
                corpus.merge_partials_device(ar.data_ptr(), as_.data_ptr(), world, nchk, k, mr.data_ptr(), msc.data_ptr())
                corpus.sync()
                want_r, want_s = mr.cpu().numpy(), msc.cpu().numpy()
            else:
                want_r, want_s = ex[0], ex[1]
            ok = bool(np.array_equal(fast_r, want_r) and np.array_equal(fast_s, want_s))
            parity_full = {"ok": ok, "queries_checked": nchk, "rows": total_rows,
                           "against": "yams_b200_search_exhaustive on every shard (exact fp64 score of every row + global sort), merged like the fast path",
                           "ids_equal": bool(np.array_equal(fast_r, want_r)), "scores_bit_equal": bool(np.array_equal(fast_s, want_s)),
                           "fast_path_queries_resolved_exhaustively": int(resolved)}
            side["oracle_window"] = (q_host.numpy()[:nchk].copy(), k, d, f32)

        flops = 2.0 * nq * n * d
        scan_s = (tm["scan_kernel_ms"] or tm["stage1_ms"]) / 1e3
        ach_tf = flops / scan_s / 1e12
        hbm_ach = n * d * esz / scan_s / 1e9
        tr = load_traffic()
        traffic = None if f32 else (tr.get("stage1_umma_kernel_per_row", 0) * n or tr.get("stage1_umma_kernel"))
        # which roof binds this batch size (SURVEY §8d: tensor above Q ~ 250, HBM below)
        # tf32 MMAs run at half the fp16/bf16 rate: the measured bf16 peak is halved for an fp32 corpus
        tensor_peak = peaks["bf16_tflops"] * (0.5 if f32 else 1.0)
        tensor_sus = peaks["bf16_tflops_sustained"] * (0.5 if f32 else 1.0)
        t_tensor = flops / (tensor_peak * 1e12)
        t_hbm = n * d * esz / (peaks["hbm_gbs"] * 1e9)
        tensor_view = {"achieved": ach_tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": ach_tf / tensor_peak,
                       "frac_of_sustained_peak": ach_tf / tensor_sus,
                       "note": "peak = burst cuBLAS bf16 (conservative); the kernel is timed inside a long back-to-back step, for which "
                               "the task's rule names the sustained figure (frac_of_sustained_peak)"}
        hbm_view = {"achieved": hbm_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_ach / peaks["hbm_gbs"]}
        roof = dict(bound="tensor", **tensor_view) if t_tensor >= t_hbm else dict(bound="hbm", **hbm_view)
        roof.update({"traffic": traffic, "traffic_source": "dram__bytes_read+write of the committed ncu --set full capture (profiles/traffic.json), scaled to this row count",
                     "peak_source": peaks["source"] + " (MEASURED_PEAKS.json: cuBLAS bf16 burst / sustained, copy bandwidth)",
                     "kernel": f"stage-1 filtered scan ({tm['engine']})", "kernel_ms": scan_s * 1e3,
                     "kernel_ms_over_ranks": scan_ms_ranks,
                     "algorithmic_flops": flops, "algorithmic_bytes": n * d * esz,
                     "tensor_view": tensor_view, "hbm_view": hbm_view})
        out.update({
            "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": world, "steps": K, "warmup": max(W, 2),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32" if f32 else "f16", "data": "synthetic", "config": knn_config(args, world, n),
            "roofline": roof,
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": nq * d * 4,
                    "d2h_bytes_per_step": nq * k * 12 + (nq * 12 if not dist else 0), "ms_per_step": e2e_ms,
                    "device_ms_last_call": tm_e2e["total_ms"], "scan_kernel_ms_last_call": tm_e2e["scan_kernel_ms"]},
            "gpu_launches": (launches_per_step + (1 if dist else 0)) * K if launches_per_step else (10 + (1 if dist else 0)) * K,
            "gpu_launches_source": "CUPTI (torch.profiler) count of one step's kernels x steps" if launches_per_step else "arithmetic (profiler unavailable)",
            "stage_ms": tm, "parity_full": parity_full,
        })
        if dist:
            gm, mm = (float(np.mean(gather_ms)) if gather_ms else 0.0), (float(np.mean(merge_ms)) if merge_ms else 0.0)
            out["multi_gpu"] = {"scan_kernel_ms_min_max": scan_ms_ranks, "allgather_ms_min_max": over_ranks(gm), "merge_ms_min_max": over_ranks(mm),
                                "allgather_bytes_per_rank": rec, "overlap": "gather + merge of batch i run on a side stream behind the scan of batch i+1",
                                "true_queries_per_s_against_full_corpus": nq / (ms_step / 1e3)}
            # per-rank kernel time and SM clock under load: the step runs at the pace of the slowest (most power-limited) GPU
            per_rank = [None] * world
            dist.all_gather_object(per_rank, {"rank": rank, "scan_kernel_ms": tm["scan_kernel_ms"], "sm_mhz": clocks_mine.get("sm_mhz"),
                                              "power_w": clocks_mine.get("power_w_median"), "reasons": clocks_mine.get("reasons")})
            out["multi_gpu"]["per_rank"] = per_rank
        if clocks is not None:
            out["clocks"] = clocks

        # ---- side measurements, N = 1 only, never allowed to break the line above ----
        if rank == 0 and world == 1 and not args.no_side and not f32:
            try:   # NS-2: the HBM-bound regime (sub-ridge batches) through the same entry point
                sweep = []
                for q_n in (1, 8, 64, 256):
                    for _ in range(3):
                        corpus.search_device(q_dev.data_ptr(), q_n, k, -1.0, part[0].data_ptr(), part[0].data_ptr() + q_n * k * 8)
                    corpus.sync()
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record(S)
                    reps = 10
                    kms = []
                    for _ in range(reps):
                        corpus.search_device(q_dev.data_ptr(), q_n, k, -1.0, part[0].data_ptr(), part[0].data_ptr() + q_n * k * 8)
                    a1.record(S)
                    corpus.sync()
                    kms = corpus.last_timings()["scan_kernel_ms"]
                    step = a0.elapsed_time(a1) / reps
                    sweep.append({"queries": q_n, "ms_per_step": step, "queries_per_s": q_n / step * 1e3, "scan_kernel_ms": kms,
                                  "hbm_gbs": n * d * esz / kms / 1e6, "hbm_frac": n * d * esz / kms / 1e6 / peaks["hbm_gbs"],
                                  "tensor_tflops": 2.0 * q_n * n * d / kms / 1e9})
                out["q_sweep"] = {"note": "same corpus, smaller query batches: HBM-bound below Q ~ 250 (SURVEY §8d); hbm_frac = algorithmic "
                                          "corpus bytes / scan kernel time / measured copy bandwidth", "points": sweep}
            except Exception as e:   # noqa: BLE001
                out["q_sweep"] = {"error": repr(e)[:200]}
        if rank == 0 and world == 1 and not args.no_side and not f32:
            try:   # N3: the SimeonPqAdc engine over the same corpus (32 B of codes per row) -- the latency engine
                rng = np.random.default_rng(1)
                m_pq, k_pq = 32, 256
                cb = (rng.normal(size=(m_pq, k_pq, d // m_pq)) / np.sqrt(d)).astype(np.float32)
                t0 = time.perf_counter()
                pq = Y.PqIndex(corpus, m_pq, k_pq, cb)
                build_s = time.perf_counter() - t0
                pts = []
                for q_n in (1, 16, 256):
                    qs = q_host.numpy()[:q_n]
                    pq.search(qs, k, rerank_factor=2, threshold=-1.0)
                    t0 = time.perf_counter()
                    for _ in range(5):
                        pq.search(qs, k, rerank_factor=2, threshold=-1.0)
                    pq_ms = (time.perf_counter() - t0) / 5 * 1e3
                    corpus.search(qs, k, threshold=-1.0)
                    t0 = time.perf_counter()
                    for _ in range(5):
                        corpus.search(qs, k, threshold=-1.0)
                    ex_ms = (time.perf_counter() - t0) / 5 * 1e3
                    pts.append({"queries": q_n, "pq_adc_ms_per_call": pq_ms, "exact_scan_ms_per_call": ex_ms,
                                "pq_code_gbs": n * m_pq * q_n / pq_ms / 1e6})
                out["pq_adc"] = {"workload": f"SimeonPqAdc over the same {n} x {d} corpus: m={m_pq}, k={k_pq} (defaults of VectorDatabaseConfig), rerank_factor 2, "
                                             "host call incl. query upload and result copy; random (untrained) codebooks -- timing only, parity is in tests/test_gpu_pq.py",
                                 "index_build_s": build_s, "code_bytes": n * m_pq, "points": pts}
                pq.close()
            except Exception as e:   # noqa: BLE001
                out["pq_adc"] = {"error": repr(e)[:200]}
        corpus.close()
        del corpus
        torch.cuda.empty_cache()

        keep5 = []
        if dist and not args.no_side and not f32:
            # e2 (SURVEY §8e): config C5 on a row-sharded corpus -- every rank keeps the part of each allowed list that falls into
            # its rowid range, re-ranks within it through the host entry point, the partial top-k are gathered and merged like the
            # unfiltered scan; rank 0 also answers the same batch on an unsharded copy and compares bit for bit.
            try:
                from yams_b200.dist import split_allowed
                c5n, c5q = 1_000_000, 256
                per = c5n // world
                lo5, hi5 = rank * per, (c5n if rank == world - 1 else (rank + 1) * per)
                c5 = Y.Corpus(d, Y.F16, Y.COSINE, capacity_hint=hi5 - lo5)
                c5.append_synthetic(42, lo5, hi5 - lo5)
                q5 = q_host.numpy()[:c5q]
                rec5 = c5q * k * 12
                p5 = torch.empty(rec5, dtype=torch.uint8, device="cuda")
                a5 = torch.empty(world * rec5, dtype=torch.uint8, device="cuda")
                f5r = torch.empty((c5q, k), dtype=torch.int64, device="cuda")
                f5s = torch.empty((c5q, k), dtype=torch.float32, device="cuda")
                pts = []
                for frac in (0.001, 0.01, 0.1):
                    rng5 = np.random.default_rng(int(frac * 1e6))      # the same lists on every rank
                    m5 = int(c5n * frac)
                    allowed = [np.sort(rng5.choice(c5n, size=m5, replace=False)).astype(np.int64) for _ in range(c5q)]
                    mine = split_allowed(allowed, lo5, hi5)

                    def one():
                        r, sc, _, _ = c5.search(q5, k, threshold=-1.0, allowed=mine)
                        p5[:c5q * k * 8].copy_(torch.from_numpy(np.ascontiguousarray(r)).view(torch.uint8).reshape(-1), non_blocking=True)
                        p5[c5q * k * 8:].copy_(torch.from_numpy(np.ascontiguousarray(sc)).view(torch.uint8).reshape(-1), non_blocking=True)
                        dist.all_gather_into_tensor(a5, p5)
                        c5.merge_packed_device(a5.data_ptr(), world, c5q, k, f5r.data_ptr(), f5s.data_ptr(), 0, torch.cuda.current_stream().cuda_stream)
                        return f5r.cpu().numpy(), f5s.cpu().numpy()

                    one()
                    barrier_sync()
                    t0 = time.perf_counter()
                    for _ in range(3):
                        rr, ss = one()
                    dt = max_over_ranks((time.perf_counter() - t0) / 3)
                    keep5.append((allowed, rr, ss))
                    pts.append({"candidate_fraction": frac, "rows_per_list": m5, "ms_per_batch": dt * 1e3, "queries_per_s": c5q / dt})
                if rank == 0:
                    out["c5_sharded"] = {"workload": f"C5 on {world} row shards: {c5n} x {d} fp16, {c5q} queries, cosine top-{k}; host call per rank "
                                                     "(list upload included) + packed all-gather + device merge + result copy", "points": pts}
                c5.close()
            except Exception as e:   # noqa: BLE001  (every rank runs the same code: a failure is symmetric, no collective is left half-entered)
                if rank == 0:
                    out["c5_sharded"] = {"error": repr(e)[:300]}
            barrier_sync()
            if rank == 0 and keep5:   # rank-local check, after the last collective of this block
                try:
                    whole = Y.Corpus(d, Y.F16, Y.COSINE, capacity_hint=1_000_000)
                    whole.append_synthetic(42, 0, 1_000_000)
                    same = True
                    for allowed, rr, ss in keep5:
                        wr, ws, _, _ = whole.search(q_host.numpy()[:256], k, threshold=-1.0, allowed=allowed)
                        same = same and bool(np.array_equal(rr, wr) and np.array_equal(ss.view(np.uint32), ws.view(np.uint32)))
                    whole.close()
                    out["c5_sharded"]["equals_unsharded_bit_for_bit"] = same
                except Exception as e:   # noqa: BLE001
                    out["c5_sharded"]["check_error"] = repr(e)[:300]
        if rank == 0 and world == 1 and not args.no_side and not f32:
            try:   # C5: candidate-set re-rank within 1M x 768, 256 queries, host call incl. the rowid-list upload
                c5n, c5q = 1_000_000, 256
                c5 = Y.Corpus(d, Y.F16, Y.COSINE, capacity_hint=c5n)
                c5.append_synthetic(42, 0, c5n)
                q5 = q_host.numpy()[:c5q]
                rng = np.random.default_rng(5)
                pts = []
                for frac in (0.001, 0.01, 0.1):
                    m = int(c5n * frac)
                    allowed = [np.sort(rng.choice(c5n, size=m, replace=False)).astype(np.int64) for _ in range(c5q)]
                    c5.search(q5, k, threshold=-1.0, allowed=allowed)
                    t0 = time.perf_counter()
                    reps = 3
                    for _ in range(reps):
                        r5 = c5.search(q5, k, threshold=-1.0, allowed=allowed)
                    dt = (time.perf_counter() - t0) / reps
                    pts.append({"candidate_fraction": frac, "rows_per_list": m, "ms_per_batch_host_call": dt * 1e3,
                                "device_ms": c5.last_timings()["total_ms"], "queries_per_s": c5q / dt})
                t0 = time.perf_counter()
                c5.search(q5, k, threshold=-1.0)
                pts.append({"candidate_fraction": 1.0, "rows_per_list": c5n, "ms_per_batch_host_call": (time.perf_counter() - t0) * 1e3,
                            "note": "unfiltered, for scale"})
                out["c5"] = {"workload": f"C5: candidate re-rank within {c5n} x {d} fp16, {c5q} queries, cosine top-{k}; lists as numpy arrays through the ctypes mirror", "points": pts}
                side["c5_last"] = (r5, allowed, q5)
                c5.close()
            except Exception as e:   # noqa: BLE001
                out["c5"] = {"error": repr(e)[:200]}
            try:   # NS-1: the L2 metric over the same kind of corpus through the same tensor-core pipeline
                ln = 2_000_000
                cl = Y.Corpus(d, Y.F16, Y.L2, capacity_hint=ln)
                for r0 in range(0, ln, step_rows):
                    cl.append_synthetic(42, r0, min(step_rows, ln - r0))
                for _ in range(2):
                    cl.search_device(q_dev.data_ptr(), nq, k, -1.0, part[0].data_ptr(), part[0].data_ptr() + nq * k * 8)
                cl.sync()
                Sl = torch.cuda.ExternalStream(cl.stream)
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record(Sl)
                for _ in range(5):
                    cl.search_device(q_dev.data_ptr(), nq, k, -1.0, part[0].data_ptr(), part[0].data_ptr() + nq * k * 8)
                a1.record(Sl)
                cl.sync()
                resolved_l2 = cl.search_device_finish()
                step = a0.elapsed_time(a1) / 5
                out["l2"] = {"workload": f"L2 (vec0 surface) {ln} x {d} fp16, {nq}-query batch, top-{k}", "ms_per_step": step,
                             "queries_per_s_10M_equiv": nq / step * 1e3 * ln / REF_ROWS, "scan_kernel_ms": cl.last_timings()["scan_kernel_ms"],
                             "tensor_tflops": 2.0 * nq * ln * d / cl.last_timings()["scan_kernel_ms"] / 1e9, "resolved_exhaustively": int(resolved_l2)}
                cl.close()
            except Exception as e:   # noqa: BLE001
                out["l2"] = {"error": repr(e)[:200]}

    # ------------------------------------------------------------------ ingest ----------------------
    if args.workload in ("both", "ingest"):
        nbytes = int(args.ingest_gib * (1 << 30))
        buf = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        Y.synth_bytes_device(12345 + rank, 0, nbytes, buf.data_ptr())
        cfg = Y.default_config()
        Wi, Ki = min(max(W, 1), 3), K
        for _ in range(Wi):
            ch = Y.chunk_and_hash_device(buf.data_ptr(), nbytes, cfg)
        barrier_sync()
        tot, sha, scan, sel = [], [], [], []
        for _ in range(Ki):
            ch = Y.chunk_and_hash_device(buf.data_ptr(), nbytes, cfg)
            t = Y.ingest_last_timings()
            tot.append(t["total_ms"]); sha.append(t["sha256_ms"]); scan.append(t["scan_ms"]); sel.append(t["select_ms"])
        barrier_sync()
        ms = max_over_ranks(float(np.mean(tot)))
        if args.dump_outputs and rank == 0:       # the chunk table of the last timed step: its size and a fixed, seeded sample of rows
            pick = np.sort(np.random.default_rng(0).choice(len(ch), size=min(len(ch), 1 << 16), replace=False))
            dumps["ingest_chunk_count"] = np.array([len(ch)], dtype=np.float64)
            dumps["ingest_offset"] = ch["offset"][pick].astype(np.float64)
            dumps["ingest_size"] = ch["size"][pick].astype(np.float64)
            dumps["ingest_digest_words"] = np.ascontiguousarray(ch["digest"][pick]).view(">u4").astype(np.float64)   # 8 big-endian words
        gbs = nbytes / (ms / 1e3) / 1e9 * world
        sha_gbs = nbytes / (float(np.mean(sha)) / 1e3) / 1e9
        scan_gbs = nbytes / (float(np.mean(scan)) / 1e3) / 1e9
        ing_launches = count_kernel_launches(lambda: Y.chunk_and_hash_device(buf.data_ptr(), nbytes, cfg)) if rank == 0 else None   # one whole step
        # e2e: pinned host buffer through the host C-ABI call (H2D inside the timed region)
        e2e_bytes = int(min(args.e2e_ingest_gib, args.ingest_gib) * (1 << 30))
        hbuf = torch.empty(e2e_bytes, dtype=torch.uint8).pin_memory()
        hbuf.copy_(buf[:e2e_bytes])
        Y.chunk_and_hash(hbuf.numpy(), cfg)
        barrier_sync()
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            che = Y.chunk_and_hash(hbuf.numpy(), cfg)
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / reps
        alu = load_traffic().get("sha256_alu_ceiling_gbs", 1103.0)
        ing = {
            "metric": "GB/s SHA-256+CDC", "value": gbs, "unit": "GB/s", "ms_per_step": ms, "steps": Ki,
            "config": {"workload": f"C3: {args.ingest_gib:g} GiB synthetic stream per GPU, StreamingChunker defaults "
                                   "(window 48, min 16 KiB, max 1 MiB, mask 0x1FFF) + SHA-256 per chunk",
                       "chunks": int(len(ch)), "l2_policy": "input >> L2"},
            "stage_ms": {"candidate_scan": float(np.mean(scan)), "cut_selection": float(np.mean(sel)),
                         "sha256": float(np.mean(sha)), "total": float(np.mean(tot))},
            "roofline": {"bound": "hbm", "achieved": sha_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": sha_gbs / peaks["hbm_gbs"], "traffic": load_traffic().get("sha256_chunks_kernel_per_gib"),
                         "kernel": "sha256_chunks_kernel",
                         "note": "SHA-256 is INT32-ALU bound, not HBM bound: ALU-pipe instructions per 64-B block counted in SASS and the "
                                 "INT32 issue rate calibrated on the device (profiles/r2_sha256_alu_ceiling.md) give the ceiling; alu_frac is the binding fraction",
                         "alu_ceiling_gbs": alu, "alu_frac": sha_gbs / alu,
                         "candidate_scan": {"achieved": scan_gbs, "frac": scan_gbs / peaks["hbm_gbs"],
                                            "note": "single pass over the input (cdc_scan_single_pass_kernel)"}},
            "e2e": {"value": e2e_bytes / (e2e_ms / 1e3) / 1e9 * world, "unit": "GB/s", "h2d_bytes_per_step": e2e_bytes,
                    "d2h_bytes_per_step": int(len(che)) * 48, "sample": f"{e2e_bytes / (1 << 30):g} GiB pinned host buffer"},
            "gpu_launches": (ing_launches if ing_launches else (int((nbytes + (1 << 34) - 1) // (1 << 34)) * 14 + 3)) * Ki,
            "gpu_launches_source": "CUPTI (torch.profiler) count of one step's kernels x steps" if ing_launches else "arithmetic",
        }
        if args.workload == "ingest":
            out.update({"metric": "GB/s SHA-256+CDC", "value": gbs, "unit": "GB/s", "n_gpus": world, "steps": Ki,
                        "warmup": Wi, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                        "vs_baseline": None, "dtype": "u8/u32", "data": "synthetic", "config": ing["config"],
                        "roofline": ing["roofline"], "e2e": ing["e2e"], "gpu_launches": ing["gpu_launches"]})
        # side measurement, N=1 only, never allowed to break the line above: many small files through the batch entry
        # (host buffers in ordinary pageable memory, chunk tables out) -- the shape of `yams add -r`
        if rank == 0 and world == 1 and not args.no_side:
            try:
                nfiles, fsz = 4096, 64 << 10
                pool = buf[: 64 * fsz].cpu().numpy().reshape(64, fsz)
                files = [np.array(pool[i % 64], copy=True) for i in range(nfiles)]
                Y.chunk_and_hash_batch(files, cfg)            # sizes the pooled pinned / device staging buffers
                t0 = time.perf_counter()
                tables = Y.chunk_and_hash_batch(files, cfg)
                dt = time.perf_counter() - t0
                ing["small_files_batch"] = {"files": nfiles, "file_bytes": fsz, "files_per_s": nfiles / dt, "gb_per_s": nfiles * fsz / dt / 1e9,
                                            "chunks": int(sum(len(t) for t in tables)),
                                            "note": "one chunk_and_hash_batch call through the ctypes mirror, pageable host buffers, wall clock incl. upload and result copy"}
            except Exception as e:   # noqa: BLE001
                ing["small_files_batch"] = {"error": repr(e)[:200]}
            # the step after chunking: exists/store over the whole chunk table as one digest-set call
            try:
                ds = Y.DigestSet(capacity_hint=len(ch))
                t0 = time.perf_counter()
                existed, fresh = ds.insert(ch)
                dt = time.perf_counter() - t0
                dev_ms = ds.last_ms()
                t0 = time.perf_counter()
                again = ds.contains(ch)
                dt2 = time.perf_counter() - t0
                ing["digest_set"] = {"digests": int(len(ch)), "new": int(fresh), "insert_ms_host_call": dt * 1e3, "insert_ms_device": dev_ms,
                                     "contains_ms_host_call": dt2 * 1e3, "contains_ms_device": ds.last_ms(),
                                     "all_found_afterwards": bool(again.all()),
                                     "note": "exists-then-store over the C3 chunk table (content_store_impl.cpp:245-288 as one call)"}
                ds.close()
            except Exception as e:   # noqa: BLE001
                ing["digest_set"] = {"error": repr(e)[:200]}
            if not args.no_parity:
                side["ingest_windows"] = (ch, nbytes)
                side["ingest_buf"] = buf
        out["ingest"] = ing
        if "ingest_buf" not in side:
            del buf

    # ------------------------------------------------------------------ checker / CPU legs ----------
    # Everything below executes oracle/ (the CPU restatement, or the reference compiled in place): after every GPU-timed region.
    if rank == 0 and (side or (world == 1 and not args.no_cpu_baseline)):
        threads = host_threads()
        O, omp_threads = load_oracle(threads)
        kind = "reference" if O.ref_available() else "port"
        if "oracle_window" in side and "parity_full" in out and out["parity_full"]:
            try:   # the exhaustive pass itself, cross-checked by the CPU oracle on a 1M-row window of shard 0
                qs, k_, d_, f32_ = side["oracle_window"]
                wn = 1_000_000
                cw = Y.Corpus(d_, Y.F32 if f32_ else Y.F16, Y.COSINE, capacity_hint=wn)
                cw.append_synthetic(42, 0, wn)
                ex = cw.search_exhaustive(qs, k_)
                fast = cw.search(qs, k_)
                rows = np.empty((wn, d_), dtype=np.float32 if f32_ else np.uint16)
                for r0 in range(0, wn, 100_000):
                    g = O.gen_rows_f32(42, r0, 100_000, d_)
                    rows[r0:r0 + 100_000] = g if f32_ else O.f16_from_float(g).reshape(100_000, d_)
                rc, wr, ws, wc = O.exact_scan_cosine_batch(rows, qs, k_)
                out["parity_full"]["oracle_window"] = {
                    "rows": wn, "queries": int(len(qs)),
                    "exhaustive_equals_oracle": bool(np.array_equal(ex[0], wr) and np.array_equal(ex[1], ws)),
                    "fast_path_equals_oracle": bool(np.array_equal(fast[0], wr) and np.array_equal(fast[1], ws)),
                    "oracle": "yo_exact_scan_cosine_batch (restatement of sqlite_vec_backend.cpp:4203-4331)"}
                out["parity_full"]["ok"] = bool(out["parity_full"]["ok"] and out["parity_full"]["oracle_window"]["exhaustive_equals_oracle"]
                                                and out["parity_full"]["oracle_window"]["fast_path_equals_oracle"])
                cw.close()
                del rows
            except Exception as e:   # noqa: BLE001
                out["parity_full"]["oracle_window"] = {"error": repr(e)[:200]}
        if "c5_last" in side:
            try:   # C5 results of the last (10 %) batch: 8 queries against the oracle with the same allowed lists
                r5, allowed, q5 = side["c5_last"]
                rows = np.empty((1_000_000, args.dim), dtype=np.uint16)
                for r0 in range(0, 1_000_000, 100_000):
                    rows[r0:r0 + 100_000] = O.f16_from_float(O.gen_rows_f32(42, r0, 100_000, args.dim)).reshape(100_000, args.dim)
                ok = True
                for qi in range(8):
                    rc, wr, ws = O.exact_scan_cosine(rows, q5[qi], args.k, threshold=-1.0, allowed=allowed[qi])
                    ok = ok and list(r5[0][qi][:len(wr)]) == list(wr) and np.array_equal(r5[1][qi][:len(wr)], ws)
                out["c5"]["parity_vs_oracle"] = {"queries_checked": 8, "ok": bool(ok)}
                del rows
            except Exception as e:   # noqa: BLE001
                out["c5"]["parity_vs_oracle"] = {"error": repr(e)[:200]}
        if "ingest_windows" in side:
            try:   # C3 parity gate (SURVEY §8d): >= 1 GiB prefix + two interior 1 GiB windows, bit-compared with the reference chunker
                ch, nbytes = side["ingest_windows"]
                buf = side["ingest_buf"]
                cfg_o = O.default_config()
                offs = ch["offset"].astype(np.uint64)
                win = 1 << 30
                rng = np.random.default_rng(17)
                starts = [0] + ([int(rng.integers(nbytes // 8, nbytes - 2 * win)) for _ in range(2)] if nbytes > 4 * win else [])
                jobs = []
                for s0 in starts:
                    # An interior window starts at a cut of the device's own table: the rolling hash at p depends on the 48 bytes
                    # before p only and candidates closer than min_chunk (16 KiB) to the window start are never cuts, so chunking
                    # stream[s0 : s0 + 1 GiB] on its own must reproduce the table from that cut on (all but the truncated last chunk).
                    i0 = 0 if s0 == 0 else int(np.searchsorted(offs, s0))
                    s0 = int(offs[i0]) if len(offs) else 0
                    jobs.append((s0, i0, buf[s0: s0 + win].cpu().numpy()))
                del side["ingest_buf"], buf

                def check(job):
                    s0, i0, host = job
                    if kind == "reference":
                        o_off, o_sz, o_dg = O.ref_chunk(host, cfg_o, variant=0)      # the reference's own StreamingChunker + OpenSSL SHA-256
                    else:
                        o_off, o_sz, o_dg = O.cdc_chunk(host, cfg_o)
                    m = len(o_off) - 1                                              # the last chunk is cut short by the window end
                    got = ch[i0:i0 + m]
                    ok = bool(m > 0 and len(got) == m and np.array_equal(got["offset"] - np.uint64(s0), o_off[:m])
                              and np.array_equal(got["size"], o_sz[:m]) and np.array_equal(got["digest"], o_dg[:m]))
                    return {"start": s0, "bytes": int(len(host)), "chunks_compared": int(m), "ok": ok}
                from concurrent.futures import ThreadPoolExecutor
                with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
                    reports = list(ex.map(check, jobs))
                out["ingest"]["parity_windows"] = {"ok": bool(all(r["ok"] for r in reports)), "windows": reports,
                                                   "checker": "reference StreamingChunker::chunkData + SHA256Hasher compiled from /root/reference (oracle/_ref)"
                                                   if kind == "reference" else "oracle restatement (oracle/yams_oracle.c)"}
            except Exception as e:   # noqa: BLE001
                out["ingest"]["parity_windows"] = {"error": repr(e)[:300]}
        if world == 1 and not args.no_cpu_baseline:   # cpu_baseline: rank 0 at N=1 only, bounded samples
            if args.workload in ("both", "knn"):
                v, arms, head, sample = cpu_knn(O, omp_threads, args.dim, args.k, args.rows, kind)
                out["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": omp_threads, "kind": kind, "sample": sample, "arms": arms}
            if args.workload in ("both", "ingest"):
                v, sample = cpu_ingest(O, omp_threads, kind)
                out["ingest"]["cpu_baseline"] = {"value": v, "unit": "GB/s", "cores": omp_threads, "kind": kind, "sample": sample}
                if args.workload == "ingest":
                    out["cpu_baseline"] = out["ingest"]["cpu_baseline"]

    if dumps:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if rank == 0:
        print(json.dumps(out), flush=True)
    if dist:
        # all ranks are done; leave without running NCCL / CUDA teardown (the external-stream communicator
        # segfaults in destroy_process_group on this torch build after the line above is already out)
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
