#!/usr/bin/env python
"""Headline benchmark of the dense-retrieval hot path (BASELINE.json):

  metric  : queries/sec, top-1000 over an 8.8M x 768 corpus (configs[1]: bert-base 768-d, 6 980 queries,
            brute force on 1 x B200); with --gpus N the same corpus is row-sharded over N GPUs and searched through
            om_index_search_sharded (collectives inside the library, NCCL over NVLink) -> strong scaling.
  also    : passages encoded/sec (bert-base / t5-base / bert-large, L=128, batch 256 per GPU), the contrastive loss,
            the C4 train step, the C5-sized shard (2.625 M x 1024), the streaming regime, and the eager-PyTorch GPU
            comparators of BASELINE.md section 2 ("gpu_eager_baseline").

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      # CPU arm: faiss if importable, else the oracle port, on a bounded sample
  python bench.py --workload c5 --gpus 8    # configs[4]: 21 M x 1024 row-sharded 8-way (2.625 M rows per GPU)

A step = one search of the whole query batch against the HBM-resident corpus (value: inputs resident in HBM;
e2e: host fp32 queries in, host (D, I) out, copies inside the timed region).  Synthetic data: corpus and
queries i.i.d. N(0,1) fp32 (seeded), random-init weights.  Timed with CUDA events, max over ranks.  After the
timed region the result of the run is verified ("parity"): sampled queries against the library's exact fp32 scan
(bit-exact expected) and against an independent chunked torch.matmul(fp32) + topk path (eps-aware).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (corpus rows, dim, encoder spec name, scaling, description)
    "c2": dict(corpus=8_800_000, dim=768, scaling="strong", metric="queries/sec top-1000 over 8.8M x 768 corpus",
               name="configs[1] search"),
    "c5": dict(corpus=2_625_000, dim=1024, scaling="weak", metric="queries/sec top-1000 over (2.625M x n_gpus) x 1024 corpus",
               name="configs[4] search (21M x 1024 at 8 GPUs, 2.625M rows per GPU)"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--corpus", type=int, default=None, help="c2: total rows (row-sharded); c5: rows PER GPU")
    ap.add_argument("--nq", type=int, default=6980)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--k", type=int, default=1000)
    ap.add_argument("--encode-batch", type=int, default=256)
    ap.add_argument("--skip-encode", action="store_true", help="search line only (no encoder / loss / train / extra legs)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-train", action="store_true")
    ap.add_argument("--skip-eager", action="store_true")
    ap.add_argument("--skip-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's search result to DIR/D.npy (scores, float32) and "
                         "DIR/I.npy (ids, float64): every query, or a fixed seeded sample of them beyond 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the result of --impl ours")
    w = WORKLOADS[args.workload]
    args.corpus = args.corpus or w["corpus"]
    args.dim = args.dim or w["dim"]
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"tflops": float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0))), "hbm": float(p["hbm_gbs"]),
                "burst": float(p.get("bf16_tflops", 0.0)) or None,
                "source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"}
    return {"tflops": 1400.0, "hbm": 6650.0, "burst": None, "source": "B200_PROFILING.md fallback (of fallback)"}


class ClockSampler:
    """SM clock / throttle reasons sampled every 100 ms while the timed region runs: NVML in-process (pynvml; a polling
    `nvidia-smi -lms` child stalls CUDA launches for tens of ms per query on these boxes), nvidia-smi only as fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, enabled=True):
        self.rows, self.proc, self.gpu, self.stop, self.thread, self.how = [], None, gpu_index, False, None, None
        self.enabled = enabled  # rank 0 only: concurrent NVML pollers on every rank stalled a step by ~100 ms at N = 2

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            max_sm = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

            def pump():
                while not self.stop:
                    try:
                        r = int(get_reasons(h))
                        self.rows.append([str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(max_sm), "0",
                                          "Active" if r & bits["hw_slowdown"] else "Not Active",
                                          "Active" if r & bits["hw_thermal_slowdown"] else "Not Active",
                                          "Active" if r & bits["sw_thermal_slowdown"] else "Not Active",
                                          "Active" if r & bits["sw_power_cap"] else "Not Active"])
                    except Exception:
                        pass
                    time.sleep(0.2)

            self.thread = threading.Thread(target=pump, daemon=True)
            self.thread.start()
            self.how = "nvml"
            return self
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "500"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            self.how = "nvidia-smi"
        except OSError:
            self.proc = None
        return self

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except (ValueError, IndexError):
                pass
        return self.gpu

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        self.stop = True
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
        elif self.thread:
            self.thread.join(timeout=1.0)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "via": self.how}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons, "samples": len(sm),
                "via": self.how}


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own path for this step is faiss IndexFlatIP.search on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_search(args, steps, warmup):
    """faiss-cpu if importable (kind "reference"), else the oracle port (blocked fp32 SGEMM + exact top-k): `nq_s`
    queries against a 1 M-row slice (BASELINE.md section 2), extrapolated linearly in rows to the full corpus.
    torchrun exports OMP_NUM_THREADS=1: the thread count is set explicitly here, before numpy / torch are imported."""
    cores = os.cpu_count() or 1
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = str(cores)
    import numpy as np
    import torch
    torch.set_num_threads(cores)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    total_rows = args.corpus * (args.gpus if WORKLOADS[args.workload]["scaling"] == "weak" else 1)
    n_s, nq_s = min(total_rows, 1_000_000), min(args.nq, 256)
    k = min(args.k, n_s)
    rng = np.random.default_rng(1234)
    x = rng.standard_normal((n_s, args.dim), dtype=np.float32)
    q = rng.standard_normal((nq_s, args.dim), dtype=np.float32)
    kind, what = "port", "oracle.flat_ip_search (numpy BLAS SGEMM + exact top-%d)" % k
    try:
        import faiss  # noqa: F401
        index = faiss.IndexFlatIP(args.dim)
        index.add(x)
        faiss.omp_set_num_threads(cores)
        run = lambda: index.search(q, k)  # noqa: E731
        kind, what = "reference", "faiss.IndexFlatIP.search (top-%d)" % k
    except ImportError:
        import oracle
        run = lambda: oracle.flat_ip_search(q, x, k)  # noqa: E731
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    qps_full = nq_s / t * (n_s / total_rows)
    return {"value": qps_full, "unit": "queries/s", "cores": cores, "kind": kind, "threads_torch": torch.get_num_threads(),
            "sample": "%s, %d queries x %d rows x %d dims per step, %.2f s/step, %d warm-up + %d timed steps, extrapolated "
                      "linearly in rows to %d" % (what, nq_s, n_s, args.dim, t, warmup, steps, total_rows),
            "ms_per_step": t * 1e3, "warmup_run": warmup, "total_rows": total_rows}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]

    if args.impl == "reference":
        if rank != 0:
            return
        wu = max(0, min(args.warmup, 2))
        base = cpu_reference_search(args, max(1, min(args.steps, 5)), wu)
        line = {"impl": "reference", "metric": wl["metric"], "value": base["value"],
                "unit": "queries/s", "n_gpus": args.gpus, "steps": max(1, min(args.steps, 5)), "warmup": wu,
                "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": "%s: top-%d over %d x %d, %d queries (CPU sample extrapolated)" % (
                    wl["name"], args.k, base["total_rows"], args.dim, args.nq), "corpus_rows": base["total_rows"],
                    "dim": args.dim, "k": args.k},
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the one JSON line
    import torch
    import torch.distributed as dist

    from openmatch_b200 import synthetic
    from openmatch_b200.encoder import CudaEncoder
    from openmatch_b200.index import FlatIPIndex, comm_for

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    assert world == args.gpus or world == 1, "--gpus must match WORLD_SIZE under torchrun"
    comm = comm_for(None) if world > 1 else None
    peaks = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    def fill_index(d, lo, hi, seed_base):
        idx_ = FlatIPIndex(d)
        chunk = 550_000
        for c0 in range(lo, hi, chunk):
            n = min(chunk, hi - c0)
            rows = idx_.reserve_rows(n)
            g = torch.Generator(device=dev).manual_seed(seed_base + c0 // chunk + 7919 * rank)
            rows.normal_(generator=g)
            idx_.commit_rows(n)
        return idx_

    # ---------------- corpus shard: rows [lo, hi) of the global corpus, generated straight into HBM ----------------
    d, k, nq = args.dim, args.k, args.nq
    if wl["scaling"] == "strong":
        total_rows = args.corpus
        per = (total_rows + world - 1) // world
        lo, hi = rank * per, min(total_rows, (rank + 1) * per)
    else:
        total_rows = args.corpus * world
        lo, hi = rank * args.corpus, (rank + 1) * args.corpus
    idx = fill_index(d, lo, hi, 1234)
    gq = torch.Generator(device=dev).manual_seed(99)
    q_dev = torch.randn(nq, d, generator=gq, device=dev)
    q_host = q_dev.cpu().pin_memory()
    if rank == 0:
        D_out = torch.empty((nq, k), dtype=torch.float32).pin_memory()
        I_out = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    else:  # only rank 0 ships the merged result to the host (the reference's rank 0 owns the result, :200-203)
        D_out = torch.empty((nq, k), dtype=torch.float32, device=dev)
        I_out = torch.empty((nq, k), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()

    # device results go into tensors allocated ONCE: a fresh [nq, k] pair per step made the caching allocator call
    # cudaMalloc inside the second timed step (the first pair still being referenced): a 15 - 100 ms stall in every run
    D_dev = torch.empty((nq, k), dtype=torch.float32, device=dev)
    I_dev = torch.empty((nq, k), dtype=torch.int64, device=dev)

    def search_step(q):
        if world == 1:
            return idx.search_device(q, k, id_offset=lo, out=(D_dev, I_dev))
        return idx.search_sharded_device(comm, q, k, lo, out=(D_dev, I_dev))

    def e2e_step():
        if world == 1:
            idx.search_pinned(q_host, k, D_out, I_out, id_offset=lo)  # C-ABI call with HOST buffers: H2D + search + D2H
        else:
            idx.search_sharded_pinned(comm, q_host, k, D_out, I_out, lo)

    # ---------------- device-resident search (value) + per-kernel device time for the roofline ----------------
    idx.set_param("profile", 1)
    acc = {"scan_ns": 0, "select_ns": 0, "finalize_ns": 0, "other_ns": 0, "launches": 0, "uncertified": 0, "exact_queries": 0,
           "overflow_retries": 0}
    rounds = 0
    last = {}

    def value_step():
        nonlocal rounds
        last["D"], last["I"] = search_step(q_dev)
        for key in acc:
            acc[key] += idx.stat(key)
        rounds = idx.stat("rounds")

    step_wall = []

    def value_step_timed():
        t0 = time.perf_counter()
        value_step()
        step_wall.append((time.perf_counter() - t0) * 1e3)  # host wall per step (diagnostic; every step ends synchronised)

    with ClockSampler(local_rank, enabled=(rank == 0)) as clocks:  # started before the warm-up: nvidia-smi's start-up lands outside the timed steps
        for _ in range(args.warmup):
            search_step(q_dev)
        total_ms = timed(value_step_timed, args.steps, 0)
    idx.set_param("profile", 0)
    ms_per_step = total_ms / args.steps
    qps = nq / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, last["D"], last["I"])

    e2e_ms = timed(e2e_step, args.steps, min(args.warmup, 2)) / args.steps
    e2e_qps = nq / (e2e_ms * 1e-3)

    # ---------------- parity of THIS run's result (sampled queries; every rank takes part) ----------------
    parity = None
    if not args.skip_parity:
        parity = check_search_parity(torch, dist, idx, comm, q_dev, last["D"], last["I"], k, lo, rank, world, dev)
        # the e2e call must have produced the same ranking
        if rank == 0:
            parity["e2e_equals_device_result"] = bool(torch.equal(I_out, last["I"].cpu()) and torch.equal(D_out, last["D"].cpu()))
            parity["ok"] = bool(parity["ok"] and parity["e2e_equals_device_result"])

    # ---------------- streaming regime (SURVEY 8(d)): few queries per pass -> one sweep of the fp16 shard is
    # HBM-bound.  Local shard only (no exchange), k = 100; roofline = rows_local * d * 2 B per sweep / measured HBM
    streaming = None
    if not args.skip_encode:
        try:
            streaming = {"unit": "ms per search over this GPU's shard", "k": 100, "cases": {}}
            sweep_bytes = (hi - lo) * d * 2.0
            for snq in (1, 16, 64):
                qs = q_dev[:snq].contiguous()
                sms_ = timed(lambda: idx.search_device(qs, 100), 10, 3) / 10
                case = {"ms": sms_, "queries_per_s": world * snq / (sms_ * 1e-3), "achieved_gbs": sweep_bytes / (sms_ * 1e-3) / 1e9}
                case["frac_of_hbm_peak"] = case["achieved_gbs"] / peaks["hbm"]
                streaming["cases"]["nq=%d" % snq] = case
        except Exception as e:  # informational leg
            streaming = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---------------- eager-PyTorch search comparator on the same GPU (BASELINE.md section 2) ----------------
    eager = {}
    if not args.skip_eager and not args.skip_encode:
        try:
            eager["search"] = eager_search(torch, idx, q_dev, k, hi - lo, total_rows, timed)
        except Exception as e:
            eager["search"] = {"error": "%s: %s" % (type(e).__name__, e)}

    n_local = hi - lo
    del idx
    last.clear()
    torch.cuda.empty_cache()

    encode = loss_obj = train_obj = c5_obj = None
    if not args.skip_encode:
        encode = encoder_legs(torch, synthetic, CudaEncoder, args, timed, world, rank, dev, peaks, eager if not args.skip_eager else None)
        loss_obj = loss_leg(torch, timed, dev, eager if not args.skip_eager else None)
        if not args.skip_train:
            train_obj = train_leg(torch, synthetic, timed, world, rank, dev)
        if args.workload == "c2" and world == 1:
            try:
                c5_obj = c5_shard_leg(torch, fill_index, timed, nq, k, dev, peaks)
            except Exception as e:
                c5_obj = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    scan_flops = 2.0 * nq * n_local * d * args.steps
    scan_s = acc["scan_ns"] * 1e-9
    achieved = scan_flops / scan_s / 1e12 if scan_s > 0 else None
    traffic = traffic_note = None
    tpath = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if os.path.exists(tpath) and world == 1 and args.workload == "c2":
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj.get("dram_bytes_per_launch")
        traffic_note = "%s: %.3g B DRAM vs %.3g B algorithmic (x%.3f); %s (constant from that ncu capture, not measured in this run)" % (
            tj.get("launch"), traffic, tj.get("algorithmic_bytes_per_launch"), tj.get("ratio_traffic_over_algorithmic"),
            tj.get("source"))
    phase = {p: acc[p + "_ns"] / 1e6 / args.steps for p in ("scan", "select", "finalize", "other")}
    line = {
        "metric": wl["metric"], "value": qps, "unit": "queries/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "%s: top-%d over %d x %d fp32 corpus resident in HBM, %d queries per step"
                               % (wl["name"], k, total_rows, d, nq), "corpus_rows": total_rows, "rows_per_gpu": n_local, "dim": d,
                   "k": k, "nq": nq, "candidate_stage": "fp16 tensor-core scan on CTA pairs (tcgen05 cta_group::2, fp32 accumulate) + fp32 re-score + exactness "
                   "certificate (escalation: 4096-wide list, then exact fp32 scan)", "rounds": rounds,
                   "parallelism": ("index row-sharded x%d, om_index_search_sharded: shard-sized candidate lists, ONE packed NCCL "
                                   "all-gather per query chunk (scores | ids | floors | error norms), merge + certificate on "
                                   "every rank" % world)
                   if world > 1 else "single shard",
                   "l2_policy": "inputs_exceed_l2 (fp16 scan copy %.1f GB per GPU)" % (n_local * d * 2 / 1e9)},
        "e2e": {"value": e2e_qps, "unit": "queries/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": nq * d * 4,
                "d2h_bytes_per_step": nq * k * 12, "note": "host result on rank 0 only" if world > 1 else None},
        "gpu_launches": acc["launches"],
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                     "frac": achieved / peaks["tflops"] if achieved else None, "traffic": traffic,
                     "traffic_note": traffic_note, "frac_of_burst_peak": achieved / peaks["burst"] if achieved and peaks["burst"] else None,
                     "kernel": "gemm2_tn_kernel<5,1,8,EpiScan,F16> (CTA pairs, cta_group::2; fused Q*X^T + top-k filter)",
                     "note": "2*nq*rows*d FLOPs per sweep / CUDA-event time of the scan launches on the launching "
                             "stream; " + peaks["source"],
                     "phase_ms_per_step": {"scan": phase["scan"], "select": phase["select"], "finalize_rescore": phase["finalize"],
                                           "exchange_merge_certify": phase["other"]},
                     "non_scan_ms_per_step": ms_per_step - phase["scan"]},
        "certificate": {"uncertified_queries_per_step": acc["uncertified"] / args.steps,
                        "exact_scan_queries_per_step": acc["exact_queries"] / args.steps,
                        "overflow_retries": acc["overflow_retries"]},
        "clocks": clocks.summary(),
        "step_wall_ms": step_wall,
    }
    if parity is not None:
        line["parity"] = parity
    if encode:
        line["encode"] = encode
    if loss_obj:
        line["loss"] = loss_obj
    if train_obj:
        line["train"] = train_obj
    if streaming:
        line["streaming"] = streaming
    if c5_obj:
        line["c5_shard"] = c5_obj
    if eager:
        line["gpu_eager_baseline"] = eager
    if world == 1 and not args.skip_cpu:
        base = cpu_reference_search(args, 1, 1)
        line["cpu_baseline"] = {k_: base[k_] for k_ in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(torch, out_dir, D, I):
    """Writes the [nq, k] result of the last timed step as D.npy (float32) and I.npy (int64 ids as float64, exact below
    2^53).  Rows beyond DUMP_BYTES are dropped by a fixed seeded sample of queries (ascending), so that two builds run
    with the same arguments, hence the same seeded inputs, can be compared output for output."""
    import numpy as np
    nq, k = D.shape
    fit = (DUMP_BYTES - 4096) // (k * (4 + 8))  # 4096: headroom for the two .npy headers
    rows = np.arange(nq) if nq <= fit else np.sort(np.random.default_rng(0).choice(nq, fit, replace=False))
    sel = torch.from_numpy(rows).to(D.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "D.npy"), D[sel].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "I.npy"), I[sel].cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------------------------
# parity of the timed run
# ------------------------------------------------------------------------------------------------------------------
def check_search_parity(torch, dist, idx, comm, q_dev, D, I, k, lo, rank, world, dev, n_sample=32):
    """Sampled queries of the run just timed, checked two ways (every rank takes part; verdict on rank 0):
      exact : the library's exact fp32 CUDA-core scan of each shard (no candidate stage), merged with torch ops —
              expected bit-identical ids AND scores (same summation order as the re-score);
      torch : independent chunked torch.matmul (fp32, TF32 off) + topk over the fp32 master rows — eps-aware: every id we
              return must be within eps of the torch k-th score, scores within eps (eps = 2e-5 |q| |x|max)."""
    nq = q_dev.shape[0]
    sel = torch.linspace(0, nq - 1, min(n_sample, nq), device=dev).round().long().unique()
    qs = q_dev[sel].contiguous()
    x = idx.master_rows()
    # (1) exact scan of the local shard
    idx.set_param("exact_only", 1)
    De, Ie = idx.search_device(qs, k, id_offset=lo)
    idx.set_param("exact_only", 0)
    # (2) torch fp32 path over the local shard
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        best_s = torch.full((qs.shape[0], k), float("-inf"), device=dev)
        best_i = torch.full((qs.shape[0], k), -1, dtype=torch.int64, device=dev)
        step = 1 << 20
        for c0 in range(0, x.shape[0], step):
            s = qs @ x[c0:c0 + step].T
            kk = min(k, s.shape[1])
            v, i = torch.topk(s, kk, dim=1)
            cat_s, cat_i = torch.cat([best_s, v], 1), torch.cat([best_i, i + (lo + c0)], 1)
            v2, p = torch.topk(cat_s, k, dim=1)
            best_s, best_i = v2, torch.gather(cat_i, 1, p)
        xmax = float(x.norm(dim=1).max())
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev

    def merge_over_ranks(Dl, Il):
        if world == 1:
            return Dl, Il
        Dp = [torch.empty_like(Dl) for _ in range(world)]
        Ip = [torch.empty_like(Il) for _ in range(world)]
        dist.all_gather(Dp, Dl.contiguous())
        dist.all_gather(Ip, Il.contiguous())
        Dc, Ic = torch.cat(Dp, 1), torch.cat(Ip, 1)
        Dc = torch.where(Ic >= 0, Dc, torch.full_like(Dc, float("-inf")))
        # (score desc, id asc): stable sort by id first, then stable sort by score
        o1 = torch.argsort(Ic, dim=1, stable=True)
        Dc, Ic = torch.gather(Dc, 1, o1), torch.gather(Ic, 1, o1)
        o2 = torch.argsort(Dc, dim=1, descending=True, stable=True)[:, :k]
        return torch.gather(Dc, 1, o2), torch.gather(Ic, 1, o2)

    De, Ie = merge_over_ranks(De, Ie)
    best_s, best_i = merge_over_ranks(best_s, best_i)
    if world > 1:
        t = torch.tensor([xmax], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        xmax = float(t.item())
    got_D, got_I = D[sel], I[sel]
    ids_exact = bool(torch.equal(got_I, Ie))
    scores_exact = bool(torch.equal(got_D, De))
    eps = 2e-5 * qs.norm(dim=1, keepdim=True) * xmax
    kth = best_s[:, k - 1:k]
    eps_valid = bool(((got_D >= kth - eps).all()) and ((got_D - best_s).abs() <= eps).all())
    same_ids_frac = float((got_I == best_i).float().mean())
    set_overlap = float(sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(got_I, best_i)) / got_I.numel())
    out = {"queries_checked": int(sel.numel()), "k": k,
           "vs_exact_fp32_scan": {"ids_identical": ids_exact, "scores_identical": scores_exact},
           "vs_torch_matmul_topk_fp32": {"eps_valid": eps_valid, "ids_equal_frac": same_ids_frac, "set_overlap": set_overlap,
                                         "max_abs_score_diff": float((got_D - best_s).abs().max()),
                                         "eps_rule": "2e-5 * |q| * |x|max (fp32 summation-order noise)"},
           "ok": bool(ids_exact and scores_exact and eps_valid)}
    return out


def eager_search(torch, idx, q_dev, k, n_local, total_rows, timed):
    """Chunked torch.matmul + topk over a bounded slice of the fp32 master rows (TF32 on = what a PyTorch user gets
    with torch.set_float32_matmul_precision('high')), extrapolated linearly in rows."""
    x = idx.master_rows()
    rows = min(n_local, 1 << 20)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    chunk = 65536

    def step():
        best_s = best_i = None
        for c0 in range(0, rows, chunk):
            s = q_dev @ x[c0:c0 + chunk].T
            v, i = torch.topk(s, min(k, s.shape[1]), dim=1)
            i = i + c0
            if best_s is None:
                best_s, best_i = v, i
            else:
                v2, p = torch.topk(torch.cat([best_s, v], 1), k, dim=1)
                best_s, best_i = v2, torch.gather(torch.cat([best_i, i], 1), 1, p)
        return best_s, best_i

    try:
        ms = timed(step, 2, 1) / 2
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    full_ms = ms * (total_rows / rows)
    return {"what": "chunked torch.matmul (fp32 master rows, TF32 allowed) + torch.topk(%d) + running merge, chunk %d rows" % (k, chunk),
            "sample_rows": rows, "ms_per_step_sample": ms, "queries_per_s_extrapolated": q_dev.shape[0] / (full_ms * 1e-3),
            "note": "single GPU, extrapolated linearly in rows to %d" % total_rows}


# ------------------------------------------------------------------------------------------------------------------
# encoder legs
# ------------------------------------------------------------------------------------------------------------------
def encoder_legs(torch, synthetic, CudaEncoder, args, timed, world, rank, dev, peaks, eager):
    B, L = args.encode_batch, 128
    steps = max(args.steps, 5)

    def flops(spec):
        H = spec["hidden"]
        return spec["layers"] * L * (24 * H * H + 4 * L * H) * B

    spec = dict(synthetic.BERT_BASE)
    sd = synthetic.bert_state_dict(spec, seed=0)
    enc = CudaEncoder(spec, sd, pooling="first", max_batch_tokens=B * L)
    ids, mask = synthetic.token_batch(B, L, spec["vocab"], seed=1234 + rank, device=dev)
    out = torch.empty((B, 768), dtype=torch.float32, device=dev)
    ids_h, mask_h = ids.cpu().pin_memory(), mask.cpu().pin_memory()
    out_h = torch.empty((B, 768), dtype=torch.float32).pin_memory()

    def enc_e2e():
        i, m = ids_h.to(dev, non_blocking=True), mask_h.to(dev, non_blocking=True)
        enc.encode(i, m, out=out)
        out_h.copy_(out, non_blocking=True)
        torch.cuda.synchronize()

    enc_ms = timed(lambda: enc.encode(ids, mask, out=out), steps, 3) / steps
    enc_e2e_ms = timed(enc_e2e, steps, 2) / steps
    fl = flops(spec)
    encode = {"metric": "passages encoded/sec (bert-base, L=128)", "value": world * B / (enc_ms * 1e-3),
              "unit": "passages/s", "ms_per_step": enc_ms, "batch_per_gpu": B,
              "e2e": {"value": world * B / (enc_e2e_ms * 1e-3), "unit": "passages/s",
                      "h2d_bytes_per_step": 2 * B * L * 8, "d2h_bytes_per_step": B * 768 * 4},
              "roofline": {"bound": "tensor", "achieved": fl / (enc_ms * 1e-3) / 1e12, "peak": peaks["tflops"],
                           "unit": "TFLOP/s", "frac": fl / (enc_ms * 1e-3) / 1e12 / peaks["tflops"],
                           "note": "whole encoder step (22.35 GFLOP/passage algorithmic) / step time; " + peaks["source"]}}
    # parity of THIS batch (B = 256, 32 768 tokens, all 12 layers) against the HF module in fp32 on the same GPU, and the
    # eager comparator (HF bf16 autocast + SDPA) timed on the same batch
    if rank == 0:
        try:
            from transformers import BertConfig, BertModel
            lm = BertModel(BertConfig(), add_pooling_layer=False)
            missing, _ = lm.load_state_dict(sd, strict=False)
            assert not [m for m in missing if "position_ids" not in m], missing
            lm = lm.to(dev).eval()
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            with torch.no_grad():
                ref = lm(input_ids=ids, attention_mask=mask).last_hidden_state[:, 0].float()
            torch.backends.cuda.matmul.allow_tf32 = prev
            got = enc.encode(ids, mask).float()
            rel = float((got - ref).norm() / ref.norm())
            cos = float(torch.nn.functional.cosine_similarity(got, ref, dim=1).min())
            encode["parity"] = {"vs": "HF BertModel fp32 (TF32 off) on the same GPU, same weights, B=%d x L=%d" % (B, L),
                                "rel_l2": rel, "min_cosine": cos, "tolerance": "rel_l2 <= 1e-2, cosine >= 0.9999",
                                "ok": bool(rel <= 1e-2 and cos >= 0.9999)}
            if eager is not None:
                def hf_step():
                    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                        lm(input_ids=ids, attention_mask=mask).last_hidden_state[:, 0]
                hf_ms = timed_local(torch, hf_step, steps, 3)
                eager["encoder_bert_base"] = {"what": "HF BertModel, bf16 autocast, SDPA attention, no_grad, B=%d L=%d" % (B, L),
                                              "passages_per_s_per_gpu": B / (hf_ms * 1e-3), "ms_per_step": hf_ms}
            del lm
        except Exception as e:
            encode["parity"] = {"error": "%s: %s" % (type(e).__name__, e)}
    del enc
    torch.cuda.empty_cache()
    # C3's encoder: t5-base (GTR) + masked mean pooling + bias-free 768x768 head + L2 normalisation
    try:
        tspec = dict(synthetic.T5_BASE)
        tenc = CudaEncoder(tspec, synthetic.t5_state_dict(tspec, seed=0),
                           head_weight=torch.randn(768, 768, generator=torch.Generator().manual_seed(3)) * 0.03,
                           pooling="mean", normalize=True, max_batch_tokens=B * L)
        tids, tmask = synthetic.token_batch(B, L, tspec["vocab"], seed=4321 + rank, bert=False, device=dev)
        t5_ms = timed(lambda: tenc.encode(tids, tmask, out=out), steps, 3) / steps
        encode["t5_base_gtr"] = {"value": world * B / (t5_ms * 1e-3), "unit": "passages/s", "ms_per_step": t5_ms,
                                 "frac_of_peak": fl / (t5_ms * 1e-3) / 1e12 / peaks["tflops"]}
        del tenc
    except Exception as e:  # informational leg
        encode["t5_base_gtr"] = {"error": "%s: %s" % (type(e).__name__, e)}
    # C5's encoder: bert-large (24 x 1024, 16 heads)
    try:
        lspec = dict(synthetic.BERT_LARGE)
        lenc = CudaEncoder(lspec, synthetic.bert_state_dict(lspec, seed=1), pooling="first", max_batch_tokens=B * L)
        lout = torch.empty((B, 1024), dtype=torch.float32, device=dev)
        l_ms = timed(lambda: lenc.encode(ids, mask, out=lout), steps, 3) / steps
        lfl = flops(lspec)
        encode["bert_large"] = {"value": world * B / (l_ms * 1e-3), "unit": "passages/s", "ms_per_step": l_ms,
                                "frac_of_peak": lfl / (l_ms * 1e-3) / 1e12 / peaks["tflops"],
                                "gflop_per_passage": lfl / B / 1e9}
        del lenc
    except Exception as e:
        encode["bert_large"] = {"error": "%s: %s" % (type(e).__name__, e)}
    torch.cuda.empty_cache()
    return encode


def timed_local(torch, fn, steps, warmup):
    """Single-rank CUDA-event timing (comparator legs that only rank 0 runs)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def loss_leg(torch, timed, dev, eager):
    """contrastive loss fwd+bwd (C4): local negatives [64, 768] x [512, 768] and the cross-device-at-8 shape
    [512, 768] x [4096, 768]; one cooperative tcgen05 kernel per call (latency-bound: reported in microseconds)"""
    from openmatch_b200 import _lib as om_lib
    lib = om_lib.load()
    loss_obj = {"metric": "contrastive loss fwd+bwd latency", "unit": "us", "kernel_launches_per_call": 1, "shapes": {}}
    for name, (bq, bp) in {"local_64x512": (64, 512), "xdevice8_512x4096": (512, 4096)}.items():
        g = torch.Generator(device="cpu").manual_seed(1234)
        xq = (torch.randn(bq, 768, generator=g) * 0.5).to(torch.bfloat16).to(dev)
        xp = (torch.randn(bp, 768, generator=g) * 0.5).to(torch.bfloat16).to(dev)
        lo_t = torch.empty((), dtype=torch.float32, device=dev)
        dxq, dxp = torch.empty(bq, 768, device=dev), torch.empty(bp, 768, device=dev)
        reps = 50

        def loss_step():
            for _ in range(reps):
                om_lib.check(lib.om_contrastive_loss_fwd_bwd(
                    xq.data_ptr(), xp.data_ptr(), om_lib.OM_BF16, bq, bp, 768, None, om_lib.OM_REDUCE_MEAN, 1.0,
                    lo_t.data_ptr(), dxq.data_ptr(), dxp.data_ptr(), None, om_lib.current_stream_ptr()))

        us = timed(loss_step, 3, 3) / 3 / reps * 1e3
        import ctypes
        ph = (ctypes.c_uint64 * 4)()
        om_lib.check(lib.om_debug_loss_phase_ns(ph))
        loss_obj["shapes"][name] = {"us": us, "tflops": 6.0 * bq * bp * 768 / (us * 1e-6) / 1e12,
                                    "phase_us": dict(zip(("prep", "logits", "softmax", "grads"),
                                                         [round(v / 1e3, 2) for v in ph]))}
        if eager is not None:
            a, b = xq.clone().requires_grad_(), xp.clone().requires_grad_()
            tgt = torch.arange(bq, device=dev) * (bp // bq)

            def eager_step():
                for _ in range(reps):
                    a.grad = b.grad = None
                    s = a @ b.T
                    torch.nn.functional.cross_entropy(s.float(), tgt).backward()

            eus = timed_local(torch, eager_step, 3, 3) / reps * 1e3
            eager.setdefault("loss", {})[name] = {"us": eus, "what": "bf16 matmul + F.cross_entropy(fp32) + autograd backward (eager)"}
    return loss_obj


def train_leg(torch, synthetic, timed, world, rank, dev):
    """contrastive training step (C4): bert-base, 64 queries (L=32) x 8 passages (L=128) per GPU, bf16 autocast.
    Encoder forward/backward = the HF torch module under autograd (our encoder kernels are forward-only, DESIGN
    section 6); loss forward+backward = loss_fused_kernel; AdamW step included; DDP all-reduce when world > 1; with
    world > 1 a second line runs --negatives_x_device (all-gather of reps + fused loss on the gathered batch)."""
    try:
        import types
        from transformers import BertConfig, BertModel
        from openmatch_b200.modeling import DRModel
        flop = 3 * (64 * 12 * 32 * (24 * 768 * 768 + 4 * 32 * 768) + 512 * 12 * 128 * (24 * 768 * 768 + 4 * 128 * 768))
        qi, qm = synthetic.token_batch(64, 32, 30522, seed=77 + rank, device=dev)
        pi, pm = synthetic.token_batch(512, 128, 30522, seed=177 + rank, device=dev)
        qb_ = {"input_ids": qi, "attention_mask": qm, "token_type_ids": torch.zeros_like(qi)}
        pb_ = {"input_ids": pi, "attention_mask": pm, "token_type_ids": torch.zeros_like(pi)}
        out = None
        for xdev in ([False, True] if world > 1 else [False]):
            torch.manual_seed(0)
            lm = BertModel(BertConfig(), add_pooling_layer=False).to(dev)
            model = DRModel(lm, lm, tied=True, pooling="first",
                            data_args=types.SimpleNamespace(train_n_passages=8),
                            train_args=types.SimpleNamespace(negatives_x_device=xdev)).to(dev).train()
            net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[dev.index]) if world > 1 else model
            opt = torch.optim.AdamW(net.parameters(), lr=5e-6, fused=True)

            def train_step():
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    loss = net(qb_, pb_).loss
                loss.backward()
                opt.step()
                opt.zero_grad(set_to_none=True)

            tr_ms = timed(train_step, 5, 3) / 5
            obj = {"value": world * 64 / (tr_ms * 1e-3), "unit": "queries/s", "ms_per_step": tr_ms,
                   "tflops_per_gpu": flop / (tr_ms * 1e-3) / 1e12}
            if not xdev:
                out = {"metric": "train queries/sec (bert-base, 64 q x 8 psg per GPU, bf16)", **obj,
                       "note": "encoder fwd/bwd: HF torch module under autograd (cuBLAS/SDPA); loss fwd+bwd: "
                               "loss_fused_kernel; fused AdamW; DDP all-reduce when n_gpus > 1"}
            else:
                out["negatives_x_device"] = {**obj, "loss_shape": "[%d, 768] x [%d, 768]" % (64 * world, 512 * world)}
            del model, net, opt, lm
            torch.cuda.empty_cache()
        return out
    except Exception as e:  # informational leg: never take the search line down with it
        return {"error": "%s: %s" % (type(e).__name__, e)}


def c5_shard_leg(torch, fill_index, timed, nq, k, dev, peaks):
    """One C5 shard on this GPU: 2.625 M x 1024 (= 21 M / 8), 6 980 queries, top-1000 (configs[4] per-GPU work;
    `bench.py --workload c5 --gpus 8` runs the whole 21 M corpus)."""
    n, d = 2_625_000, 1024
    idx = fill_index(d, 0, n, 4321)
    q = torch.randn(nq, d, generator=torch.Generator(device=dev).manual_seed(5), device=dev)
    idx.set_param("profile", 1)
    scan_ns = 0
    unc = 0

    out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int64, device=dev))

    def step():
        nonlocal scan_ns, unc
        idx.search_device(q, k, out=out)
        scan_ns += idx.stat("scan_ns")
        unc += idx.stat("uncertified")

    for _ in range(2):
        idx.search_device(q, k, out=out)
    ms = timed(step, 3, 0) / 3
    ach = 2.0 * nq * n * d * 3 / (scan_ns * 1e-9) / 1e12
    out = {"rows": n, "dim": d, "nq": nq, "k": k, "ms_per_step": ms, "queries_per_s": nq / (ms * 1e-3),
           "roofline": {"bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                        "scan_ms_per_step": scan_ns / 1e6 / 3},
           "uncertified_queries_per_step": unc / 3,
           "ceiling_note": "compute ceiling for 21M x 1024 on 8 GPUs at this per-shard time: %.0f queries/s" % (nq / (ms * 1e-3))}
    del idx
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
