#!/usr/bin/env python3
"""bench.py -- pgvector's distance hot path on B200, one JSON line per run (BASELINE.json metric and configs).

  python bench.py [--config B] [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]

--config selects the BASELINE.json configuration (default B = configs[1], the one the metric is quoted on):

  A  exact L2 <-> scan, 10k x 128 fp32, k = 10                      (no index; the CPU-runnable parity case)
  B  IVFFlat L2 1M x 1536 fp32, lists = 1000, probes = 10, k = 10   (HEADLINE: queries/s, 2048-query batches)
  C  HNSW cosine 1M x 768 halfvec, ef_search = 100                  (graph built on the GPU by vb_hnsw_build)
  D  IVFFlat k-means build 10M x 1536, lists = 4096                 (rows sharded over the ranks; k-means++ + Lloyd + assign)
  E  HNSW Hamming 10M x bit(1024), ef_search = 200

A "step" is one pass of the hot path over one batch of synthetic input (D: one complete build).

  value    whole-job throughput with inputs resident in HBM (device pointers, the C ABI's *_dev calls)
  e2e      the same through the host-buffer C ABI call (pinned host queries in, host results out, copies timed)
  roofline the dominant kernel: bytes the launch moves (computed live from the launch's own job list, see
           vb_ivf_tc_traffic) / its CUDA-event time vs the measured HBM peak -- always a physical fraction (<= ~1);
           SURVEY 8(d)'s per-query algorithmic bytes are reported next to it as `algorithmic`
  cpu_baseline / --impl reference   the oracle port of the reference's CPU path on the host cores (bounded sample)

Config B's line also carries: the second synthetic law (`laws`), a batch sweep incl. single-query latency through
vb_ivf_scan_lists + vb_ivf_scan_items (`batch_sweep`), and the per-query fused-scan formulation of north_star
(`north_star_kernel`, scan_impl 1) with its own roofline.  Under torchrun the lists are sharded over the ranks
(`scaling: strong`, exchanges inside the library over NCCL) and the replica mode is measured beside it.

Both arms share ONE index: whichever arm runs first writes centres + assignment to a cache under /tmp; the other
loads it (`config.index_build` says which happened)."""
from __future__ import annotations

import argparse
import hashlib
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

try:    # the metric is BASELINE.json's, verbatim
    METRIC = json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
except Exception:
    METRIC = "IVFFlat 1M×1536d queries/sec at 1/2/4/8 GPU; recall@10; HBM GB/s vs roofline"

CACHE_DIR = os.environ.get("VB_BENCH_CACHE", "/tmp/pgvector_b200_bench")
D_METRIC = "IVFFlat k-means build (BASELINE.json configs[3]): rows indexed per second (k-means++ seeding + k-means on the samples + assign of all rows)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="B", choices=["A", "B", "C", "D", "E"])
    ap.add_argument("--rows", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--lists", type=int, default=None)
    ap.add_argument("--probes", type=int, default=10)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--law", default="both", choices=["rank16", "mixture", "both"],
                    help="config B: synthetic law of the headline (rank16) and/or SURVEY 8(d)'s Gaussian mixture")
    ap.add_argument("--latent-dim", type=int, default=16)
    ap.add_argument("--components", type=int, default=1000)
    ap.add_argument("--ef", type=int, default=None)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--ef-construction", type=int, default=64)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-recall", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="config B: skip batch sweep / north-star kernel / second law")
    ap.add_argument("--scan-impl", type=int, default=int(os.environ.get("VB_SCAN_IMPL", "2")),
                    help="0 = per-query LDG.128 scan, 1 = per-query cp.async.bulk (TMA) scan, 2 = library default "
                         "(query batches: tensor-core filter + exact re-score), 3 = list-major fp32, 4 = tensor-core filter")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="config B, product arm: write the ids and distances of the last timed step to DIR/*.npy")
    a = ap.parse_args()
    if a.dump_outputs is not None and (a.config != "B" or a.impl != "ours"):
        ap.error("--dump-outputs is implemented for config B, product arm")
    d = {"A": dict(rows=10_000, dim=128, lists=0, batch=1000, steps=100, warmup=3),
         "B": dict(rows=1_000_000, dim=1536, lists=1000, batch=2048, steps=100, warmup=3),
         "C": dict(rows=1_000_000, dim=768, lists=0, batch=10_000, steps=20, warmup=3),
         "D": dict(rows=10_000_000, dim=1536, lists=4096, batch=0, steps=3, warmup=1),
         "E": dict(rows=10_000_000, dim=1024, lists=0, batch=10_000, steps=20, warmup=3)}[a.config]
    for key, v in d.items():
        if getattr(a, key) is None:
            setattr(a, key, v)
    if a.ef is None:
        a.ef = 200 if a.config == "E" else 100
    if a.config == "A":
        a.queries = min(a.queries, 1000)
    return a


# ----------------------------------------------------------------------------- plumbing

def host_threads():
    """cores this process may use (cgroup / affinity aware), not the machine's"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


_NEAR = {}


class near_gpu:
    """Run the pinned host allocations of the end-to-end legs on the CPUs NVML calls ideal for the GPU, so the pages are
    first touched (and pinned) on the GPU's NUMA node: on a two-socket box a far-node staging buffer halves the H2D rate
    (measured between boxes of this pool: 52 vs ~17 GB/s for the same 12.6 MB copy).  No-op when NVML is not usable."""

    def __init__(self, index):
        self.index, self.saved = index, None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            ncpu = os.cpu_count() or 1
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
            ideal = {w * 64 + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
            cur = os.sched_getaffinity(0)
            near = ideal & cur
            _NEAR[self.index] = {"gpu_ideal_cpus": len(ideal), "usable": len(near), "of": len(cur)}
            if near and near != cur:
                self.saved = cur
                os.sched_setaffinity(0, near)
        except Exception as e:      # noqa: BLE001 -- a hint, never a failure
            _NEAR[self.index] = {"error": str(e)[:80]}
        return self

    def __exit__(self, *exc):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)
        return False


class ClockSampler:
    # Sampled every 200 ms (the period of the profiling recipe).  A query is not free: with `-lms 20` and power.draw in
    # the list the end-to-end step of config B measured 1.69 ms under the sampler against 0.98 ms without it
    # (profiles/r2_diag_e2e.json) -- the driver serialises the query with the process's copies and synchronisations.
    # power.draw (the slow sensor read) is not used by the line, so it is not queried; the placeholder keeps the columns.
    FIELDS = ("clocks.sm,clocks.max.sm,clocks.mem,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 200

    def __init__(self, index=0):
        self.samples = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1417.3)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1417.3, "fallback (B200_PROFILING.md)"


class Env:
    """ranks, device, the library, its communicator"""

    def __init__(self, args, need_gpu=True):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        self.pv = None
        if not need_gpu:
            self.dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
            return
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import torch.distributed as dist
            # rank 0 prints exactly one JSON line on stdout; NCCL writes its banner to fd 1 when a communicator is created
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                warm = torch.zeros(1, device=self.dev)
                dist.all_reduce(warm)
                torch.cuda.synchronize()
                self.dist = dist
                import pgvector_b200 as pv
                pv.init(self.local)
                ident = [pv.comm_unique_id() if self.rank == 0 else None]
                dist.broadcast_object_list(ident, src=0)
                pv.comm_init(ident[0], self.rank, self.world)      # the library's own communicator (NCCL from C)
                pv.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        import pgvector_b200 as pv
        pv.init(self.local)
        pv.set_option("scan_impl", args.scan_impl)
        if os.environ.get("VB_FUSED_REFINE") is not None:       # A/B switch of the fused select / re-score / certify kernel
            pv.set_option("fused_refine", int(os.environ["VB_FUSED_REFINE"]))
        if os.environ.get("VB_HNSW_L2") is not None:            # A/B switch of the persisting-L2 window over the HNSW visited tables
            pv.set_option("hnsw_l2_persist", int(os.environ["VB_HNSW_L2"]))
        if os.environ.get("VB_SLAB_SELECT") is not None:        # A/B switch of the selection from slab minima
            pv.set_option("slab_select", int(os.environ["VB_SLAB_SELECT"]))
        self.pv = pv
        self.stream = torch.cuda.ExternalStream(pv.stream_handle(), device=self.dev)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.dist is None:
            return x
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            if self.pv is not None:
                self.pv.comm_free()
            self.dist.destroy_process_group()


def timed_steps(env, step, steps, warmup, extra_load=0):
    """W untimed steps, `extra_load` more while nvidia-smi spins up, then exactly K steps between events on the library
    stream, barrier + synchronize on both sides, max over ranks."""
    torch = env.torch
    for i in range(warmup):
        step(i)
    env.barrier()
    for i in range(extra_load):
        step(i)
    env.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(env.stream)
    for i in range(steps):
        step(warmup + i)
    e1.record(env.stream)
    env.barrier()
    return env.max_over_ranks(e0.elapsed_time(e1))


def dump_outputs(out_dir, arrays, budget=64 << 20):
    """Write each array (rows = queries) as out_dir/<name>.npy in float32 / float64.  Above `budget` bytes in all, a
    fixed seeded sample of the rows is written, with the sampled row numbers in row_index.npy."""
    arrays = {name: np.asarray(a, dtype=np.float32 if a.dtype == np.float32 else np.float64) for name, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_row = sum(a[:1].nbytes for a in arrays.values()) + 8
    if n * per_row > budget:
        keep = np.sort(np.random.default_rng(0).choice(n, budget // per_row, replace=False))
        arrays = {name: a[keep] for name, a in arrays.items()}
        arrays["row_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- config B: data, index (shared between the arms)

def law_name(args, law):
    return (f"x = Q z + 0.02 eps, z ~ N(0, I_{args.latent_dim}), Q random {args.dim}x{args.latent_dim} orthonormal frame, seeds 3/4"
            if law == "rank16" else
            f"mixture of {args.components} Gaussians (centres N(0,1), sigma 0.3), seeds 3/4 (SURVEY 8d)")


def make_dataset(args, law, device, n_rows=None, row_offset=0):
    """rows (seed 3) and queries (seed 4), generated in slabs.  rank16: 1536-d vectors of intrinsic dimension 16
    (k-means gives balanced lists, ~10 k candidates per query at probes = 10 -- the scan BASELINE's config describes);
    mixture: SURVEY 8(d)'s law, on which the reference's own k-means++/Lloyd leaves ~11 % of the components without a
    centre and merges them into a few giant lists (DESIGN.md section 5)."""
    import torch
    n = args.rows if n_rows is None else n_rows
    g = torch.Generator(device=device).manual_seed(3)
    slab = 65536
    rows = torch.empty((n, args.dim), device=device, dtype=torch.float32)
    if law == "rank16":
        frame = torch.linalg.qr(torch.randn((args.dim, args.latent_dim), generator=g, device=device, dtype=torch.float32))[0]
        for lo in range(0, n, slab):
            hi = min(n, lo + slab)
            z = torch.randn((hi - lo, args.latent_dim), generator=g, device=device)
            rows[lo:hi] = z @ frame.T + 0.02 * torch.randn((hi - lo, args.dim), generator=g, device=device)
        g2 = torch.Generator(device=device).manual_seed(4)
        zq = torch.randn((args.queries, args.latent_dim), generator=g2, device=device)
        queries = zq @ frame.T + 0.02 * torch.randn((args.queries, args.dim), generator=g2, device=device)
        return rows, queries.contiguous()
    comp = torch.randn((args.components, args.dim), generator=g, device=device, dtype=torch.float32)
    for lo in range(0, n, slab):
        hi = min(n, lo + slab)
        which = torch.randint(0, args.components, (hi - lo,), generator=g, device=device)
        rows[lo:hi] = comp[which] + 0.3 * torch.randn((hi - lo, args.dim), generator=g, device=device)
    g2 = torch.Generator(device=device).manual_seed(4)
    which = torch.randint(0, args.components, (args.queries,), generator=g2, device=device)
    queries = comp[which] + 0.3 * torch.randn((args.queries, args.dim), generator=g2, device=device)
    return rows, queries


def torch_assign(rows, centers, slab=32768):
    import torch
    out = torch.empty(rows.shape[0], dtype=torch.int64, device=rows.device)
    cn = (centers * centers).sum(1)
    for lo in range(0, rows.shape[0], slab):
        x = rows[lo:lo + slab]
        out[lo:lo + slab] = (cn[None, :] - 2.0 * (x @ centers.T)).argmin(1)
    return out


def index_cache_path(args, law):
    key = json.dumps([args.rows, args.dim, args.lists, law, args.latent_dim, args.components, "v2"])
    return os.path.join(CACHE_DIR, "ivf_" + hashlib.sha1(key.encode()).hexdigest()[:16] + ".npz")


def build_index_arrays(args, law, rows, pv):
    """centres + assignment: from the cache another arm wrote, else k-means on a sample + assign -- with the library
    (k-means++ / Lloyd / tensor-core assign) in the product arm, with a torch fp32 k-means++ / Lloyd in the reference
    arm (setup only; neither is inside a timed region).  Returns (centres, offsets, grouped rows, heap ids, how)."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    n = rows.shape[0]
    path = index_cache_path(args, law)
    centers = assign = None
    if os.path.exists(path):
        try:
            z = np.load(path)
            centers = torch.from_numpy(z["centers"]).to(rows.device)
            assign = torch.from_numpy(z["assign"]).to(rows.device).to(torch.int64)
            how = f"shared index cache written by the {str(z['arm'])} arm ({str(z['how'])})"
        except Exception:
            centers = assign = None
    if centers is None:
        g = torch.Generator(device=rows.device).manual_seed(42)
        ns = min(n, max(args.lists * 50, 10000))          # src/ivfbuild.c:448-452
        samp = rows[torch.randperm(n, generator=g, device=rows.device)[:ns]]
        t0 = time.perf_counter()
        if pv is not None:
            torch.cuda.synchronize()
            t = pv.Table(pv.VECTOR, args.dim).append(samp)
            init = pv.kmeans_pp_init(t, pv.L2, args.lists, seed=42)       # InitCenters (src/ivfkmeans.c:23-91)
            c_host, iters = pv.kmeans(t, pv.L2, init, max_iter=500)
            centers = torch.from_numpy(c_host).to(rows.device)
            t.free()
            tr = pv.Table(pv.VECTOR, args.dim).append(rows)
            assign = pv.assign(tr, pv.L2_SQUARED, centers).to(torch.int64)
            pv.synchronize()
            tr.free()
            arm, how = "product", f"vb_kmeans_pp_init + vb_kmeans ({iters} it) + vb_assign, {time.perf_counter() - t0:.2f} s"
        else:
            centers = samp[:args.lists].clone()
            w = torch.full((ns,), float("inf"), device=rows.device)
            cur = int(torch.randint(0, ns, (1,), generator=g, device=rows.device).item())
            sn = (samp * samp).sum(1)
            for i in range(args.lists):
                centers[i] = samp[cur]
                d2 = (sn - 2.0 * (samp @ samp[cur]) + sn[cur]).clamp_(min=0)
                w = torch.minimum(w, d2)
                cur = int(torch.multinomial(w.clamp(min=0) + 1e-30, 1, generator=g).item())
            for _ in range(10):
                a = torch_assign(samp, centers)
                sums = torch.zeros_like(centers).index_add_(0, a, samp)
                cnt = torch.bincount(a, minlength=args.lists).clamp(min=1).to(torch.float32)
                centers = sums / cnt[:, None]
            assign = torch_assign(rows, centers)
            arm, how = "reference", f"torch fp32 k-means++ + 10 Lloyd iterations + assign (setup), {time.perf_counter() - t0:.2f} s"
        try:
            os.makedirs(CACHE_DIR, exist_ok=True)
            tmp = path + f".{os.getpid()}.tmp.npz"
            np.savez(tmp, centers=centers.cpu().numpy(), assign=assign.to(torch.int32).cpu().numpy(), arm=arm, how=how)
            os.replace(tmp, path)
        except OSError:
            pass
        how = f"built by this ({arm}) arm: {how}"
    order = torch.argsort(assign, stable=True)
    counts = torch.bincount(assign, minlength=args.lists)
    offsets = torch.zeros(args.lists + 1, dtype=torch.int64)
    offsets[1:] = torch.cumsum(counts.cpu(), 0)
    grouped = torch.empty_like(rows)
    for lo in range(0, n, 65536):
        grouped[lo:lo + 65536] = rows[order[lo:lo + 65536]]
    lens = counts.cpu().numpy()
    how += f"; list sizes min/mean/max = {int(lens.min())}/{float(lens.mean()):.0f}/{int(lens.max())}"
    return centers.contiguous(), offsets.numpy(), grouped, order.contiguous(), how


def workload_b(args, law, how, extra=None):
    cfg = {"workload": f"IVFFlat L2 {args.rows}x{args.dim} fp32, lists={args.lists}, probes={args.probes}, k={args.k} "
                       f"(BASELINE.json configs[1])",
           "data_law": law_name(args, law), "queries": args.queries, "batch": args.batch, "index_build": how}
    if extra:
        cfg.update(extra)
    return cfg


# ----------------------------------------------------------------------------- CPU arm (oracle port), config B

def cpu_arm_b(args, oix, queries, steps, warmup, budget_s):
    """oracle port of GetScanLists + GetScanItems + sort on the cores this process may use, one query per thread.
    A step is a bounded sample of S queries (stated), sized from a calibration so W + K steps take about budget_s."""
    cores = host_threads()
    t0 = time.perf_counter()
    oix.search_batch(queries[:cores], args.probes, args.k, threads=cores)
    per_round = max(time.perf_counter() - t0, 1e-4)              # one query on every thread
    total_q = max(cores, int(budget_s / per_round) * cores)
    s = max(cores, min(len(queries), total_q // max(1, steps + warmup)))
    s -= s % cores if s > cores else 0
    nq = len(queries)

    def batch(i):
        lo = (i * s) % max(1, nq - s + 1)
        return queries[lo:lo + s]

    for i in range(warmup):
        oix.search_batch(batch(i), args.probes, args.k, threads=cores)
    t0 = time.perf_counter()
    for i in range(steps):
        oix.search_batch(batch(warmup + i), args.probes, args.k, threads=cores)
    dt = time.perf_counter() - t0
    n1 = max(2, min(32, int(1.0 / max(per_round, 1e-4))))
    t1 = time.perf_counter()
    oix.search_batch(queries[:n1], args.probes, args.k, threads=1)
    dt1 = time.perf_counter() - t1
    return {"value": steps * s / dt, "unit": "queries/s", "cores": cores, "kind": "port",
            "sample": f"{steps} steps of {s} queries of the same workload, one query per thread on {cores} threads "
                      f"(sched_getaffinity; oracle port of src/ivfscan.c:47-187 with the reference's compiler flags; no "
                      f"PostgreSQL buffer-manager / fmgr / tuplesort overhead => optimistic)",
            "queries_per_step": s, "ms_per_step": 1000.0 * dt / steps, "single_thread_qps": n1 / dt1}


# ----------------------------------------------------------------------------- config B, product arm

def measure_ivf(env, args, law, centers, offsets, grouped, order, full, queries):
    """device-resident throughput, end-to-end throughput and the list-scan roofline of one index"""
    torch, pv = env.torch, env.pv
    dev, world, rank = env.dev, env.world, env.rank
    B, k = min(args.batch, args.queries), args.k
    nb = max(1, args.queries // B)
    qbatches = [queries[i * B:(i + 1) * B].contiguous() for i in range(nb)]
    ids_dev = torch.empty((B, k), dtype=torch.int64, device=dev)
    dist_dev = torch.empty((B, k), dtype=torch.float32, device=dev)

    if world > 1:
        # list l lives on rank l % world; the other ranks keep it empty under the same number
        keep = (torch.arange(args.lists) % world) == rank
        lens = np.diff(offsets)
        sel = torch.zeros(grouped.shape[0], dtype=torch.bool)
        for l in range(args.lists):
            if keep[l]:
                sel[offsets[l]:offsets[l + 1]] = True
        sel = sel.to(dev)
        g_local, o_local = grouped[sel].contiguous(), order[sel].contiguous()
        off_local = np.zeros(args.lists + 1, dtype=np.int64)
        off_local[1:] = np.cumsum(np.where(keep.numpy(), lens, 0))
    else:
        g_local, o_local, off_local = grouped, order, offsets
    ix = pv.IvfflatIndex("vector_l2_ops", args.dim, args.lists)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ix.load(centers, off_local, g_local, o_local)
    pv.synchronize()
    upload_s = time.perf_counter() - t0

    def step_dev(i):
        if world > 1:
            ix.search_sharded_into(qbatches[i % nb], k, args.probes, ids_dev, dist_dev)
        else:
            ix.search_into(qbatches[i % nb], k, args.probes, ids_dev, dist_dev)

    sampler = ClockSampler(env.local)
    if rank == 0 and full:
        sampler.start()
    for i in range(args.warmup):
        step_dev(i)
    env.barrier()
    for i in range(600 if args.scan_impl >= 2 and full else 3):     # load for the clock sampler (nvidia-smi reports every 200 ms)
        step_dev(i)
    env.barrier()
    # The timed region carries the per-kernel event brackets (the roofline's kernel time is measured over it); the
    # traffic accounting -- an extra kernel per filter launch that walks the launch's job list -- runs over two
    # identical steps AFTER it (it cost 4-7 % of `value` inside, profiles/r2_diag_e2e_v2.json).
    pv.prof_enable(True)
    for p in (pv.PROF_SCAN_ITEMS, pv.PROF_SCAN_LISTS, pv.PROF_TOPK, pv.PROF_LIST_TC, pv.PROF_CENTRE_TC):
        pv.prof_read(p)
    l0 = pv.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(env.stream)
    for i in range(args.steps):
        step_dev(args.warmup + i)
    e1.record(env.stream)
    env.barrier()
    ms = env.max_over_ranks(e0.elapsed_time(e1))
    launches = pv.launch_count() - l0
    last_step = (ids_dev.cpu().numpy(), dist_dev.cpu().numpy()) if args.dump_outputs is not None else None    # the last timed step's result
    prof = {name: pv.prof_read(p) for name, p in (("scan_items", pv.PROF_SCAN_ITEMS), ("scan_lists", pv.PROF_SCAN_LISTS),
                                                   ("topk", pv.PROF_TOPK), ("list_tc", pv.PROF_LIST_TC), ("centre_tc", pv.PROF_CENTRE_TC))}
    pv.prof_enable(False)
    pv.tc_traffic(True, read=True)
    for i in range(2):
        step_dev(args.warmup + args.steps - 1 - i)      # the last batches of the timed region again
    pv.synchronize()
    traffic = pv.tc_traffic(False, read=True)
    cand_last = ix.last_candidates()                    # this rank's candidates in the last step
    cand_all = int(env.sum_over_ranks(cand_last))
    qps = args.steps * B / (ms / 1000.0)

    # ---- end to end through the host-buffer C ABI call
    with near_gpu(env.local):
        q_host = [torch.empty((B, args.dim), dtype=torch.float32).pin_memory().copy_(qb.cpu()).numpy() for qb in qbatches[:4]]
        ids_h = torch.empty((B, k), dtype=torch.int64).pin_memory().numpy()
        dist_h = torch.empty((B, k), dtype=torch.float64).pin_memory().numpy()
    # the host -> device copy of one batch alone (explains the end-to-end number on boxes with a slow link)
    h2d_dst = torch.empty((B, args.dim), dtype=torch.float32, device=dev)
    q_pin_t = torch.from_numpy(q_host[0])
    for _ in range(3):
        h2d_dst.copy_(q_pin_t, non_blocking=True)
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(10):
        h2d_dst.copy_(q_pin_t, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    h2d_alone_ms = c0.elapsed_time(c1) / 10
    del h2d_dst
    pipelined = world == 1 and args.dim % 4 == 0 and os.environ.get("VB_BENCH_NO_PIPELINE") != "1"
    n_e2e = [0]
    if pipelined:
        ix.prefetch_queries(q_host[0], 0)

    def step_host(_):
        i = n_e2e[0]
        n_e2e[0] += 1
        if world > 1:
            ix.search_sharded_host_into(q_host[i % len(q_host)], k, args.probes, ids_h, dist_h)
        elif pipelined:
            ix.prefetch_queries(q_host[(i + 1) % len(q_host)], (i + 1) % 2)
            ix.search_prefetched_into(i % 2, k, args.probes, ids_h, dist_h)
        else:
            ix.search_host_into(q_host[i % len(q_host)], k, args.probes, ids_h, dist_h)

    ms_h = timed_steps(env, step_host, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 and full else None
    e2e_matches = None
    if world == 1:
        last = (n_e2e[0] - 1) % len(q_host)
        got_ids, got_dist = ids_h.copy(), dist_h.copy()
        chk_ids, chk_dist = np.empty_like(ids_h), np.empty_like(dist_h)
        ix.search_host_into(q_host[last], k, args.probes, chk_ids, chk_dist)
        e2e_matches = bool(np.array_equal(got_ids, chk_ids) and np.array_equal(got_dist, chk_dist))
    e2e = {"value": args.steps * B / (ms_h / 1000.0), "unit": "queries/s", "h2d_bytes_per_step": B * args.dim * 4,
           "d2h_bytes_per_step": B * k * 16, "ms_per_step": ms_h / args.steps,
           "call": ("vb_ivf_search_sharded (host buffers; NCCL exchanges inside)" if world > 1 else
                    "vb_ivf_prefetch_queries (next batch) + vb_ivf_search_prefetched" if pipelined else "vb_ivf_search"),
           "last_step_equals_plain_call": e2e_matches, "h2d_alone_ms": h2d_alone_ms,
           "h2d_gbs": B * args.dim * 4 / (h2d_alone_ms / 1000.0) / 1e9, "pinned_near_gpu": _NEAR.get(env.local)}

    # ---- roofline of the dominant kernel, from live CUDA events and the launch's own job list
    peak, _, peak_src = measured_peaks()
    roofline = roofline_ivf(args, ix, prof, traffic, cand_last, cand_all, B, ms, peak, peak_src, world)
    return dict(ix=ix, qps=qps, ms=ms, launches=int(launches), e2e=e2e, roofline=roofline, clocks=clocks, upload_s=upload_s,
                cand_all=cand_all, qbatches=qbatches, last_step=last_step)


def roofline_ivf(args, ix, prof, traffic, cand_last, cand_all, B, ms, peak, peak_src, world):
    elem_bytes = 4
    alg_per_query_bytes = (B * args.lists + cand_all) * args.dim * elem_bytes      # SURVEY 8(d): per query, not amortised
    path = {0: "ldg", 1: "bulk", 3: "tile"}.get(args.scan_impl, "tc" if args.k <= 40 else "tile")
    tc_ms, tc_n = prof["list_tc"]
    if path == "tc" and tc_n > 0:
        kern_ms = tc_ms / tc_n
        n = max(int(traffic[3]), 1)
        a_once, b_once, issued = traffic[1] / n, traffic[2] / n, traffic[0] / n
        out_bytes = cand_last * 4
        moved = a_once + b_once + out_bytes
        level = 1 if ix.tc_level1_fallbacks() == 0 else 2
        achieved = moved / (kern_ms / 1000.0) / 1e9
        r = {"bound": "hbm", "kernel": "list_tc_kernel (GetScanItems list scan, tcgen05 filter level %d)" % level,
             "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
             "traffic": moved, "traffic_source": "computed live from the launch's job list (vb_ivf_tc_traffic): distinct "
                        "row-plane tiles + distinct query tiles + candidate distances written; the ncu capture is the cross-check",
             "traffic_detail": {"row_planes": a_once, "query_tiles": b_once, "distances_written": out_bytes,
                                "bulk_copy_bytes_requested": issued},
             "avg_launch_ms": kern_ms, "launches_timed": int(tc_n), "share_of_step": tc_ms / ms if ms > 0 else None,
             "filter_level": level, "certificate_fallback_queries": ix.tc_fallbacks(),
             "level1_fallback_queries": ix.tc_level1_fallbacks(),
             "bf16_mma_tflops_issued": (level + 1) * 2.0 * cand_last * args.dim / (kern_ms / 1000.0) / 1e12}
        ncu = os.path.join(ROOT, "profiles", "listtc_traffic.json")
        default_shape = (args.rows, args.dim, args.lists, args.probes, args.batch) == (1_000_000, 1536, 1000, 10, 2048)
        r["traffic_ncu"] = json.load(open(ncu))["traffic_bytes"] if (os.path.exists(ncu) and default_shape and world == 1 and level == 1) else None
    else:
        it_ms, it_n = prof["scan_items"]
        kern_ms = it_ms / max(it_n, 1)
        moved = cand_last * args.dim * elem_bytes if path in ("ldg", "bulk") else None
        name = {"ldg": "scan_kernel", "bulk": "scan_bulk_kernel", "tile": "list_tile_kernel", "tc": "list_tile_kernel"}[path]
        achieved = (moved / (kern_ms / 1000.0) / 1e9) if moved and kern_ms > 0 else None
        r = {"bound": "hbm" if path != "tile" else "fp32-fma", "kernel": name + "<vector,L2^2> (GetScanItems list scan)",
             "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
             "frac": achieved / peak if achieved else None, "traffic": moved,
             "traffic_source": "every candidate row read once per query (per-query formulation)" if moved else None,
             "avg_launch_ms": kern_ms, "share_of_step": it_ms / ms if ms > 0 else None}
    step_s = ms / args.steps / 1000.0
    r["algorithmic"] = {"definition": "SURVEY 8(d): (lists + candidates) x dim x 4 B per query, NOT amortised over the batch",
                        "bytes_per_step": alg_per_query_bytes, "gbs": alg_per_query_bytes / step_s / 1e9,
                        "over_traffic": (alg_per_query_bytes / r["traffic"]) if r.get("traffic") else None,
                        "note": "list-major kernels read each probed list once per BATCH; the ratio is the reuse across the batch "
                                "(x the bytes per element the filter level reads), not a bandwidth"}
    r["other_kernels_ms_per_step"] = {"probe_selection": prof["scan_lists"][0] / max(prof["scan_lists"][1], 1),
                                      "select_rescore_certify": prof["topk"][0] / max(prof["topk"][1], 1),
                                      "grouping_and_query_packing": (prof["scan_items"][0] - tc_ms) / max(prof["scan_items"][1], 1) if path == "tc" else None}
    return r


def recall_and_parity(env, args, ix, grouped, order, queries, oix, n_par):
    """recall@10 vs the exact scan (GPU exact top-k over the same rows) and id / distance agreement with the oracle"""
    torch, pv = env.torch, env.pv
    out = {}
    k = args.k
    nq_r = min(256, args.queries)
    t = pv.Table(pv.VECTOR, args.dim).append(grouped)
    ex_ids, _ = t.exact_topk(pv.L2_SQUARED, queries[:nq_r].contiguous(), k)
    ex_heap = order[ex_ids.clamp(min=0)]
    got, _ = ix.search(queries[:nq_r].contiguous(), k=k, probes=args.probes)
    hit = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(got.cpu(), ex_heap.cpu()))
    out["recall_at_10"] = hit / (nq_r * k)
    t.free()
    if oix is not None:
        qh = queries[:n_par].cpu().numpy()
        wi, wd = oix.search_batch(qh, args.probes, k, threads=host_threads())
        gi, gd = ix.search(queries[:n_par].contiguous(), k=k, probes=args.probes)
        gi, gd = gi.cpu().numpy(), gd.cpu().numpy()
        out["parity"] = {"queries": int(n_par), "id_agreement": float((gi == wi).mean()),
                         "max_rel_dist_err": float(np.max(np.abs(gd - wd) / np.maximum(np.abs(wd), 1e-30))),
                         "oracle_recall_at_10": None}
        o_hit = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(wi[:nq_r], ex_heap.cpu().numpy()[:len(wi[:nq_r])]))
        out["parity"]["oracle_recall_at_10"] = o_hit / (min(nq_r, n_par) * k)
    return out


def batch_sweep(env, args, ix, queries):
    """queries/s of the device-resident call at several batch sizes, and single-query latency through the two host calls
    the extension glue makes per scan (vb_ivf_scan_lists + vb_ivf_scan_items, INTEGRATION.md)"""
    torch, pv = env.torch, env.pv
    out = []
    k = args.k
    # the oracle legs before this ran on the CPU: bring the GPU back to its working clocks first (a batch-1 loop is all
    # launch latency and never loads the GPU enough to do that by itself: it measured 0.51 ms per call right after the CPU legs)
    wb = min(2048, args.queries)
    w_ids = torch.empty((wb, k), dtype=torch.int64, device=env.dev)
    w_dist = torch.empty((wb, k), dtype=torch.float32, device=env.dev)
    for _ in range(300):
        ix.search_into(queries[:wb].contiguous(), k, args.probes, w_ids, w_dist)
    pv.synchronize()
    for b in (1, 8, 64, 512, 2048, 8192):
        if b > args.queries:
            continue
        qb = queries[:b].contiguous()
        ids = torch.empty((b, k), dtype=torch.int64, device=env.dev)
        dist = torch.empty((b, k), dtype=torch.float32, device=env.dev)
        reps = int(max(5, min(200, 40000 // b)))
        for _ in range(3):
            ix.search_into(qb, k, args.probes, ids, dist)
        pv.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(env.stream)
        for _ in range(reps):
            ix.search_into(qb, k, args.probes, ids, dist)
        e1.record(env.stream)
        pv.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out.append({"batch": b, "queries_per_s": b / (ms / 1000.0), "ms_per_batch": ms})
    # one query per scan, host buffers, synchronous: what a single backend sees (amcanparallel = false)
    qh = queries[:200].cpu().numpy()
    lat = []
    for i in range(len(qh)):
        t0 = time.perf_counter()
        lists, _ = ix.scan_lists(qh[i], args.probes)
        ix.scan_items(qh[i], lists[0], cap=k)
        lat.append(time.perf_counter() - t0)
    lat = np.sort(np.array(lat[20:])) * 1e6
    t0 = time.perf_counter()
    for i in range(100):
        ix.search(qh[i:i + 1], k=k, probes=args.probes)
    one_call = (time.perf_counter() - t0) / 100 * 1e6
    # the same two calls through the general path (nine launches, three memsets, four copies) for comparison
    pv.set_option("one_query", 0)
    try:
        lat0 = []
        for i in range(120):
            t0 = time.perf_counter()
            lists, _ = ix.scan_lists(qh[i], args.probes)
            ix.scan_items(qh[i], lists[0], cap=k)
            lat0.append(time.perf_counter() - t0)
        lat0 = np.sort(np.array(lat0[20:])) * 1e6
        t0 = time.perf_counter()
        for i in range(100):
            ix.search(qh[i:i + 1], k=k, probes=args.probes)
        one_call0 = (time.perf_counter() - t0) / 100 * 1e6
    finally:
        pv.set_option("one_query", 1)
    return {"device_resident": out,
            "single_query": {"calls": "vb_ivf_scan_lists + vb_ivf_scan_items (host buffers, synchronous, timed around the Python wrappers)",
                             "kernels": "one_probe_kernel + one_scan_kernel (fused distance + select, csrc/vb_ivf_one.cu)",
                             "latency_us_p50": float(lat[len(lat) // 2]), "latency_us_p90": float(lat[int(len(lat) * 0.9)]),
                             "latency_us_mean": float(lat.mean()), "queries_per_s": float(1e6 / lat.mean()),
                             "one_call_vb_ivf_search_latency_us": one_call,
                             "general_path": {"latency_us_p50": float(lat0[len(lat0) // 2]), "one_call_vb_ivf_search_latency_us": one_call0}}}


def north_star_kernel(env, args, ix, qbatches, cand_per_step_hint):
    """north_star's formulation: one query against its candidates, fused distance kernel with TMA (cp.async.bulk) tiles
    into shared memory + per-query top-k select (scan_impl 1), every candidate row read once per query"""
    torch, pv = env.torch, env.pv
    B, k = qbatches[0].shape[0], args.k
    ids = torch.empty((B, k), dtype=torch.int64, device=env.dev)
    dist = torch.empty((B, k), dtype=torch.float32, device=env.dev)
    res = {}
    for impl, name in ((1, "scan_bulk_kernel (cp.async.bulk + mbarrier ring)"), (0, "scan_kernel (LDG.128 streaming)")):
        pv.set_option("scan_impl", impl)
        try:
            for i in range(2):
                ix.search_into(qbatches[i % len(qbatches)], k, args.probes, ids, dist)
            pv.synchronize()
            pv.prof_enable(True)
            pv.prof_read(pv.PROF_SCAN_ITEMS)
            steps = 5
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(env.stream)
            cand = 0
            for i in range(steps):
                ix.search_into(qbatches[i % len(qbatches)], k, args.probes, ids, dist)
            e1.record(env.stream)
            pv.synchronize()
            ms = e0.elapsed_time(e1)
            it_ms, it_n = pv.prof_read(pv.PROF_SCAN_ITEMS)
            pv.prof_enable(False)
            cand = ix.last_candidates()
            peak, _, _ = measured_peaks()
            moved = cand * args.dim * 4
            achieved = moved / (it_ms / max(it_n, 1) / 1000.0) / 1e9
            res[f"scan_impl_{impl}"] = {"kernel": name, "value": steps * B / (ms / 1000.0), "unit": "queries/s", "ms_per_step": ms / steps,
                                        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                                     "traffic": moved, "traffic_source": "candidates x dim x 4 B: every candidate row read once per query",
                                                     "avg_launch_ms": it_ms / max(it_n, 1), "share_of_step": it_ms / ms}}
        finally:
            pv.set_option("scan_impl", args.scan_impl)
            pv.prof_enable(False)
    return res


def run_b_ours(args):
    env = Env(args)
    torch, pv = env.torch, env.pv
    laws = ["rank16", "mixture"] if args.law == "both" else [args.law]
    if args.no_extras or env.world > 1:
        laws = laws[:1]
    primary = None
    second = {}
    for li, law in enumerate(laws):
        rows, queries = make_dataset(args, law, env.dev)
        torch.cuda.synchronize()
        centers, offsets, grouped, order, how = build_index_arrays(args, law, rows, pv)
        del rows
        torch.cuda.empty_cache()
        full = li == 0
        saved_steps = args.steps
        if not full:
            args.steps = max(10, args.steps // 4)
        m = measure_ivf(env, args, law, centers, offsets, grouped, order, full, queries)
        args.steps = saved_steps
        extras = {}
        oix = None
        if env.world == 1 and env.rank == 0 and not args.no_cpu:
            import oracle as O
            oix = O.Ivf(O.VECTOR, O.L2_SQUARED, centers.cpu().numpy(), offsets, grouped.cpu().numpy(), order.cpu().numpy())
        if env.world == 1 and not args.no_recall:
            extras.update(recall_and_parity(env, args, m["ix"], grouped, order, queries, oix, n_par=min(2048, args.queries)))
        if full:
            if env.world == 1 and not args.no_extras:
                extras["batch_sweep"] = batch_sweep(env, args, m["ix"], queries)
                extras["north_star_kernel"] = north_star_kernel(env, args, m["ix"], m["qbatches"], m["cand_all"])
            if oix is not None:
                cpu = cpu_arm_b(args, oix, queries.cpu().numpy(), steps=8, warmup=1, budget_s=args.cpu_seconds)
                extras["cpu_baseline"] = cpu
            replica = None
            if env.world > 1:
                replica = measure_replica(env, args, centers, offsets, grouped, order, queries)
            primary = dict(m=m, law=law, how=how, extras=extras, replica=replica)
        else:
            second[law] = {"data_law": law_name(args, law), "index_build": how, "value": m["qps"], "unit": "queries/s",
                           "ms_per_step": m["ms"] / max(10, saved_steps // 4), "steps": max(10, saved_steps // 4),
                           "e2e": m["e2e"], "roofline": m["roofline"], "candidates_per_query": m["cand_all"] / min(args.batch, args.queries),
                           **extras}
        m["ix"].free()
        del grouped, order, centers
        torch.cuda.empty_cache()
    if env.rank == 0:
        m, ex = primary["m"], primary["extras"]
        if args.dump_outputs is not None:
            dump_outputs(args.dump_outputs, {"ids": m["last_step"][0], "distances": m["last_step"][1]})
        B = min(args.batch, args.queries)
        cfg = workload_b(args, primary["law"], primary["how"], dict(
            index_upload_s=m["upload_s"], candidates_per_query=m["cand_all"] / B,
            l2_policy="inputs larger than L2: every step reads the probed lists of a %d MB table once" % (args.rows * args.dim * 4 // env.world // 2**20),
            scan_kernel={0: "per-query LDG.128 streaming (all scans)", 1: "per-query cp.async.bulk + mbarrier staged (all scans)",
                         3: "list-major fp32x2 register tiles (rows read once per batch)"}.get(
                args.scan_impl, "query batches: tcgen05 split-bf16 filter over packed row planes (each probed list read once per batch; level 1 = "
                                "hi plane, level 2 = both planes on certificate failure) + exact fp32 re-score + certificate; exact kernel last"),
            parallelism=("lists sharded l % N; probe selection sharded over the queries; two NCCL all-gathers inside libvecb200 "
                         "(probe lists, per-rank top-k) + k-way merge kernel" if env.world > 1 else "single GPU")))
        line = {"metric": METRIC, "value": m["qps"], "unit": "queries/s", "n_gpus": env.world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": m["ms"] / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "recall_at_10": ex.get("recall_at_10"), "parity": ex.get("parity"), "roofline": m["roofline"],
                "cpu_baseline": ex.get("cpu_baseline"), "e2e": m["e2e"], "gpu_launches": m["launches"], "clocks": m["clocks"],
                "laws": second or None, "batch_sweep": ex.get("batch_sweep"), "north_star_kernel": ex.get("north_star_kernel"),
                "replica_mode": primary["replica"]}
        print(json.dumps(line))
    env.close()
    return 0


def measure_replica(env, args, centers, offsets, grouped, order, queries):
    """query-sharded replicas: every rank holds the whole index and serves its own batches (no exchange)"""
    torch, pv = env.torch, env.pv
    B, k = min(args.batch, args.queries), args.k
    ix = pv.IvfflatIndex("vector_l2_ops", args.dim, args.lists).load(centers, offsets, grouped, order)
    nb = max(1, args.queries // B)
    qb = [queries[i * B:(i + 1) * B].contiguous() for i in range(nb)]
    ids = torch.empty((B, k), dtype=torch.int64, device=env.dev)
    dist = torch.empty((B, k), dtype=torch.float32, device=env.dev)
    ms = timed_steps(env, lambda i: ix.search_into(qb[(i + env.rank) % nb], k, args.probes, ids, dist), args.steps, args.warmup, extra_load=50)
    ix.free()
    return {"value": env.world * args.steps * B / (ms / 1000.0), "unit": "queries/s", "ms_per_step": ms / args.steps, "scaling": "weak",
            "note": "every rank holds the full 6 GB index (+ 6 GB of packed planes) and serves its own 2048-query batches; no exchange"}


def run_b_reference(args):
    env = Env(args, need_gpu=False)
    if env.rank != 0:
        return 0
    import oracle as O
    law = "rank16" if args.law in ("both", "rank16") else "mixture"
    rows, queries = make_dataset(args, law, env.dev)
    centers, offsets, grouped, order, how = build_index_arrays(args, law, rows, None)
    del rows
    oix = O.Ivf(O.VECTOR, O.L2_SQUARED, centers.cpu().numpy(), offsets, grouped.cpu().numpy(), order.cpu().numpy())
    cb = cpu_arm_b(args, oix, queries.cpu().numpy(), steps=args.steps, warmup=args.warmup, budget_s=max(args.cpu_seconds * 5, 30.0))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_b(args, law, how, {"batch": cb["queries_per_step"],
                                                  "note": "a step of this arm is a bounded sample of `batch` queries of the same workload"}),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- config A: exact scan

def run_a(args):
    ref = args.impl == "reference"
    env = Env(args, need_gpu=not ref)
    if ref and env.rank != 0:
        return 0
    torch = env.torch
    import oracle as O
    g = torch.Generator().manual_seed(1)
    rows = torch.randn((args.rows, args.dim), generator=g, dtype=torch.float32)
    g2 = torch.Generator().manual_seed(2)
    queries = torch.randn((args.queries, args.dim), generator=g2, dtype=torch.float32)
    rows_h, q_h = rows.numpy(), queries.numpy()
    k = args.k
    cores = host_threads()

    def cpu_pass(qs):
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(cores) as ex:
            return list(ex.map(lambda q: O.exact_topk(O.VECTOR, O.L2, q, rows_h, k), qs))

    workload = {"workload": f"exact L2 <-> scan, {args.rows}x{args.dim} fp32, k={k}, {args.queries} queries per step (BASELINE.json configs[0])",
                "data_law": "iid N(0,1), seeds 1/2", "queries": args.queries, "batch": args.queries}
    if ref:
        for _ in range(args.warmup):
            cpu_pass(q_h)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_pass(q_h)
        dt = time.perf_counter() - t0
        v = args.steps * len(q_h) / dt
        cb = {"value": v, "unit": "queries/s", "cores": cores, "kind": "port",
              "sample": f"{args.steps} steps of all {len(q_h)} queries, one query per thread (oracle port of src/vector.c:579-589 + top-N sort)"}
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload, "cpu_baseline": cb,
                          "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return 0
    pv = env.pv
    t = pv.Table(pv.VECTOR, args.dim).append(rows_h)
    q_dev = queries.to(env.dev)
    torch.cuda.synchronize()
    nq = args.queries
    ids = torch.empty((nq, k), dtype=torch.int64, device=env.dev)
    dist = torch.empty((nq, k), dtype=torch.float32, device=env.dev)
    lib = pv.load()
    import ctypes as C

    def step_dev(_):
        pv._lib.check(lib.vb_exact_topk_dev(t.h, pv.L2, C.c_void_p(q_dev.data_ptr()), nq, k, C.c_void_p(ids.data_ptr()), C.c_void_p(dist.data_ptr())))

    sampler = ClockSampler(env.local)
    sampler.start()
    l0 = pv.launch_count()
    ms = timed_steps(env, step_dev, args.steps, args.warmup, extra_load=2000)
    launches = (pv.launch_count() - l0)
    with near_gpu(env.local):
        q_pin = torch.empty((nq, args.dim), dtype=torch.float32).pin_memory().copy_(queries).numpy()
    ids_h = np.empty((nq, k), dtype=np.int64)
    dist_h = np.empty((nq, k), dtype=np.float64)

    def step_host(_):
        pv._lib.check(lib.vb_exact_topk(t.h, pv.L2, q_pin.ctypes.data_as(C.c_void_p), nq, k, ids_h.ctypes.data_as(C.c_void_p), dist_h.ctypes.data_as(C.c_void_p)))

    ms_h = timed_steps(env, step_host, args.steps, args.warmup)
    clocks = sampler.stop()
    want = cpu_pass(q_h)
    wi = np.stack([w[0] for w in want])
    wd = np.stack([w[1] for w in want])
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        cpu_pass(q_h)
    cpu_qps = reps * nq / (time.perf_counter() - t0)
    peak, _, peak_src = measured_peaks()
    per_launch = ms / args.steps
    moved = args.rows * args.dim * 4 * ((nq + 127) // 128) + nq * args.dim * 4 + nq * args.rows * 4 * 2
    line = {"metric": METRIC, "value": args.steps * nq / (ms / 1000), "unit": "queries/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_launch, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload, l2_policy="table (5 MB) is L2-resident by construction of this config; nothing to flush"),
            "parity": {"queries": nq, "id_agreement": float((ids_h == wi).mean()),
                       "max_rel_dist_err": float(np.max(np.abs(dist_h - wd) / np.maximum(np.abs(wd), 1e-30)))},
            "roofline": {"bound": "hbm", "kernel": "distance_matrix (128x128 fp32 tiles) + segment_topk", "achieved": moved / (per_launch / 1000) / 1e9,
                         "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": moved / (per_launch / 1000) / 1e9 / peak, "traffic": moved,
                         "traffic_source": "table re-read per 128-query tile (L2 hits) + queries + the nq x rows distance matrix written and re-read by the select",
                         "note": "a 5 MB table against 1000 queries is L2 / FMA bound, not HBM bound; the fraction is reported for completeness",
                         "algorithmic": {"definition": "SURVEY 8(d): rows x dim x 4 B per query", "bytes_per_step": nq * args.rows * args.dim * 4}},
            "cpu_baseline": {"value": cpu_qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": f"{reps} passes over all {nq} queries, one query per thread"},
            "e2e": {"value": args.steps * nq / (ms_h / 1000), "unit": "queries/s", "h2d_bytes_per_step": nq * args.dim * 4, "d2h_bytes_per_step": nq * k * 16,
                    "ms_per_step": ms_h / args.steps, "call": "vb_exact_topk"},
            "gpu_launches": int(launches), "clocks": clocks}
    print(json.dumps(line))
    env.close()
    return 0


# ----------------------------------------------------------------------------- configs C / E: HNSW

def hnsw_dataset(args, cfg, dev, torch):
    dim, comps = args.dim, 1000
    g = torch.Generator(device=dev).manual_seed(3 if cfg == "C" else 6)
    centres = torch.randn((comps, dim), generator=g, device=dev)

    def draw(count, gen):
        out = []
        for lo in range(0, count, 1 << 18):
            m = min(1 << 18, count - lo)
            which = torch.randint(0, comps, (m,), generator=gen, device=dev)
            x = centres[which] + (0.3 if cfg == "C" else 1.0) * torch.randn((m, dim), generator=gen, device=dev)
            if cfg == "C":
                # halfvec_cosine_ops stores l2_normalize'd rows (HnswFormIndexValue); normalise, round to half, normalise again
                x = torch.nn.functional.normalize(x, dim=1).to(torch.float16)
                x = torch.nn.functional.normalize(x.float(), dim=1).to(torch.float16)
                out.append(x.view(torch.int16))
            else:
                bits = (x > 0).to(torch.uint8).reshape(m, dim // 8, 8)       # binary_quantize (src/vector.c:952-978), MSB first
                w = torch.tensor([128, 64, 32, 16, 8, 4, 2, 1], device=dev, dtype=torch.uint8)
                out.append((bits * w).sum(dim=2).to(torch.uint8))
        return torch.cat(out)

    rows = draw(args.rows, g)
    queries = draw(args.queries, torch.Generator(device=dev).manual_seed(4 if cfg == "C" else 7))
    return rows, queries


def run_hnsw(args):
    cfg = args.config
    ref = args.impl == "reference"
    env = Env(args, need_gpu=True)      # the graph is built on the GPU in both arms (setup); the reference arm then searches it on the CPU
    torch, pv = env.torch, env.pv
    opclass = "halfvec_cosine_ops" if cfg == "C" else "bit_hamming_ops"
    elem, metric = pv.OPCLASSES[opclass][:2]
    law = ("Gaussian mixture (1000 components, sigma 0.3), l2-normalised, rounded to half, seeds 3/4" if cfg == "C" else
           "binary_quantize of a 1024-d Gaussian mixture (1000 components, sigma 1.0), seeds 6/7")
    rows, queries = hnsw_dataset(args, cfg, env.dev, torch)
    torch.cuda.synchronize()
    ix = pv.HnswIndex(opclass, args.dim, m=args.m)
    t0 = time.perf_counter()
    ix.build(rows, ef_construction=args.ef_construction, seed=42)
    pv.synchronize()
    build_s = time.perf_counter() - t0
    k, ef = args.k, args.ef
    B = min(args.batch, args.queries)
    workload = {"workload": (f"HNSW cosine {args.rows}x{args.dim} halfvec, m={args.m}, ef_construction={args.ef_construction}, ef_search={ef}, k={k} (BASELINE.json configs[2])"
                             if cfg == "C" else
                             f"HNSW Hamming {args.rows} x bit({args.dim}), m={args.m}, ef_construction={args.ef_construction}, ef_search={ef}, k={k} (BASELINE.json configs[4])"),
                "data_law": law, "queries": args.queries, "batch": B,
                "index_build": f"vb_hnsw_build on the GPU: {build_s:.2f} s ({args.rows / build_s:.0f} rows/s), shared by both arms",
                "parallelism": "replicas only (north_star: HNSW search stays single-GPU)"}
    row_bytes = args.dim * 2 if cfg == "C" else args.dim // 8
    # oracle on the SAME graph (export -> import)
    n_par = min(512, args.queries)
    import oracle as O
    g = ix.export()
    rows_h = rows.cpu().numpy()
    if cfg == "C":
        rows_h = rows_h.view(np.uint16)
    og = O.Hnsw.from_export(elem, metric, rows_h, g, dim=args.dim)
    q_h = queries.cpu().numpy()
    if cfg == "C":
        q_h = q_h.view(np.uint16)
    cores = host_threads()
    if ref:
        if env.rank != 0:
            return 0
        s = max(cores, min(args.queries, 2048))
        for i in range(args.warmup):
            og.search_batch(q_h[:s], ef, k, ties=O.TIES_PG, threads=cores)
        t0 = time.perf_counter()
        for i in range(args.steps):
            lo = (i * s) % max(1, args.queries - s + 1)
            og.search_batch(q_h[lo:lo + s], ef, k, ties=O.TIES_PG, threads=cores)
        dt = time.perf_counter() - t0
        v = args.steps * s / dt
        cb = {"value": v, "unit": "queries/s", "cores": cores, "kind": "port",
              "sample": f"{args.steps} steps of {s} queries, one query per thread (oracle port of src/hnswscan.c:25-56 + hnswutils.c:824-987, pairing-heap tie order)"}
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f16" if cfg == "C" else "u8", "data": "synthetic", "config": dict(workload, batch=s), "cpu_baseline": cb,
                          "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return 0
    nb = max(1, args.queries // B)
    qb = [queries[i * B:(i + 1) * B].contiguous() for i in range(nb)]
    ids = torch.empty((B, k), dtype=torch.int64, device=env.dev)
    dist = torch.empty((B, k), dtype=torch.float32, device=env.dev)
    nd = torch.empty((B,), dtype=torch.int64, device=env.dev)
    sampler = ClockSampler(env.local)
    if env.rank == 0:
        sampler.start()
    pv.prof_enable(True)
    pv.prof_read(pv.PROF_HNSW)
    l0 = pv.launch_count()
    ms = timed_steps(env, lambda i: ix.search_into(qb[(i + env.rank) % nb], k, ef, ids, dist, nd), args.steps, args.warmup, extra_load=30)
    launches = pv.launch_count() - l0
    k_ms, k_n = pv.prof_read(pv.PROF_HNSW)
    pv.prof_enable(False)
    nd_mean = float(nd.float().mean().item())
    with near_gpu(env.local):
        qh = [torch.empty(tuple(qb[0].shape), dtype=qb[0].dtype).pin_memory().copy_(x.cpu()).numpy() for x in qb[:2]]
    if cfg == "C":
        qh = [x.view(np.uint16) for x in qh]
    ms_h = timed_steps(env, lambda i: ix.search(qh[i % len(qh)], k=k, ef_search=ef), args.steps, args.warmup)
    # one query per scan (what one backend does: hnswgettuple's first call -> one vb_hnsw_search with host buffers, synchronous)
    lat = []
    for i in range(120):
        t0 = time.perf_counter()
        ix.search(qh[0][i:i + 1], k=k, ef_search=ef)
        lat.append(time.perf_counter() - t0)
    lat = np.sort(np.array(lat[20:])) * 1e6
    single = {"calls": "vb_hnsw_search, one query, host buffers, synchronous (timed around the Python wrapper); one warp walks the graph",
              "latency_us_p50": float(lat[len(lat) // 2]), "latency_us_p90": float(lat[int(len(lat) * 0.9)])}
    clocks = sampler.stop() if env.rank == 0 else None
    if env.rank != 0:
        env.close()
        return 0
    # recall@10 vs the exact scan; parity vs the oracle walking the same graph
    nr = min(256, args.queries)
    t = pv.Table(elem, args.dim).append(rows)
    ex, exd = t.exact_topk(metric, queries[:nr].contiguous(), k)
    got_i, got_d, got_nd = ix.search(q_h[:n_par], k=k, ef_search=ef)
    if cfg == "C":
        hit = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(got_i[:nr], ex.cpu().numpy()))
        recall = hit / (nr * k)
    else:   # tie-aware (test/t/020_hnsw_bit_build_recall.pl:85-91)
        recall = float((got_d[:nr] <= exd.cpu().numpy()[:, -1:].astype(np.float64)).mean())
    wi, wd, wnd = og.search_batch(q_h[:n_par], ef, k, ties=O.TIES_TOTAL, threads=cores)
    same_q = np.all(got_i == wi, axis=1)
    cpu_base = None
    if not args.no_cpu:
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < args.cpu_seconds / 2 or reps == 0:
            lo = (reps * 2048) % max(1, args.queries - 2048 + 1)
            og.search_batch(q_h[lo:lo + 2048], ef, k, ties=O.TIES_PG, threads=cores)
            reps += 1
        cpu_base = {"value": reps * min(2048, args.queries) / (time.perf_counter() - t0), "unit": "queries/s", "cores": cores, "kind": "port",
                    "sample": f"{reps} batches of 2048 queries on the same graph, one query per thread (oracle port of src/hnswutils.c:824-987)"}
    peak, _, peak_src = measured_peaks()
    qps = env.world * args.steps * B / (ms / 1000)
    kern = k_ms / max(k_n, 1)
    moved = nd_mean * B * row_bytes + (nd_mean / (2 * args.m) * 2) * B * 2 * args.m * 4
    line = {"metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": env.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16" if cfg == "C" else "u8",
            "data": "synthetic", "config": dict(workload, l2_policy="inputs larger than L2: random row gathers over a %d MB element table" % (args.rows * row_bytes // 2**20)),
            "recall_at_10": recall,
            "parity": {"queries": int(n_par), "same_graph": "exported GPU-built graph imported into the oracle", "queries_with_identical_ids": float(same_q.mean()),
                       "id_agreement": float((got_i == wi).mean()), "max_rel_dist_err": float(np.max(np.abs(got_d - wd) / np.maximum(np.abs(wd), 1e-30))),
                       "n_dist_equal_on_identical_walks": bool(np.array_equal(got_nd[same_q], wnd[same_q]))},
            "roofline": {"bound": "hbm", "kernel": "hnsw_search_kernel", "achieved": moved / (kern / 1000) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": moved / (kern / 1000) / 1e9 / peak, "traffic": moved,
                         "traffic_source": "n_dist (returned per query) x row bytes + one neighbour list per ~m distance evaluations (SURVEY 8d); gathers are 128-byte sectors",
                         "n_dist_per_query": nd_mean, "avg_launch_ms": kern, "share_of_step": kern * args.steps / ms},
            "cpu_baseline": cpu_base,
            "e2e": {"value": env.world * args.steps * B / (ms_h / 1000), "unit": "queries/s", "h2d_bytes_per_step": B * row_bytes, "d2h_bytes_per_step": B * (k * 16 + 8),
                    "ms_per_step": ms_h / args.steps, "call": "vb_hnsw_search"},
            "single_query": single,
            "gpu_launches": int(launches), "clocks": clocks,
            "build": {"seconds": build_s, "rows_per_s": args.rows / build_s, "mean_degree_layer0": float((g["nbr0"] >= 0).sum(axis=1).mean()),
                      "duplicates_folded": int((g["dup_of"] >= 0).sum()), "max_level": int(g["levels"].max())}}
    print(json.dumps(line))
    env.close()
    return 0


# ----------------------------------------------------------------------------- config D: sharded k-means build

def run_d(args):
    ref = args.impl == "reference"
    env = Env(args, need_gpu=not ref)
    torch = env.torch
    if ref:
        if env.rank != 0:
            return 0
        # the reference's k-means is serial (SURVEY 2.2): Elkan on one thread, on a bounded sample of the same law
        import oracle as O
        n_s, lists = 20480, 410                       # 1/10 of config D's samples and lists: the same samples-per-centre ratio
        n_rows = n_s * 10
        a2 = argparse.Namespace(**vars(args))
        a2.components, a2.queries = args.lists, 16
        rows, _ = make_dataset(a2, "mixture", env.dev, n_rows=n_rows)
        x = rows.cpu().numpy()
        cores = host_threads()
        t0 = time.perf_counter()
        init = O.kmeans_pp_init(O.VECTOR, O.L2, x[:n_s], lists, seed=42)
        centers, _, iters = O.kmeans(O.VECTOR, O.L2, x[:n_s], init, algo="elkan")
        t1 = time.perf_counter()
        O.ivf_assign(O.VECTOR, O.L2_SQUARED, x, centers, threads=cores)
        dt = time.perf_counter() - t0
        v = n_rows / dt
        print(json.dumps({"impl": "reference", "metric": D_METRIC, "value": v, "unit": "rows/s", "n_gpus": args.gpus,
                          "steps": 1, "warmup": 0, "ms_per_step": 1000 * dt, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": f"bounded sample of BASELINE.json configs[3]: k-means++ + Elkan k-means ({iters} iterations, 1 thread: the "
                                                                      f"reference's k-means is serial) on {n_s}x{args.dim} samples -> {lists} centres in {t1 - t0:.1f} s, then assign of "
                                                                      f"{n_rows} rows on {cores} threads"},
                          "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": f"{n_s} samples, {lists} centres, {n_rows} rows assigned"},
                          "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return 0
    pv = env.pv
    world, rank = env.world, env.rank
    n_local = args.rows // world
    a2 = argparse.Namespace(**vars(args))
    a2.components, a2.queries = args.lists, 256
    # every rank draws its own slice of the mixture (same component centres: generator seed 3 draws them first)
    g = torch.Generator(device=env.dev).manual_seed(3)
    comp = torch.randn((args.lists, args.dim), generator=g, device=env.dev, dtype=torch.float32)
    g = torch.Generator(device=env.dev).manual_seed(1000 + rank)
    rows = torch.empty((n_local, args.dim), device=env.dev, dtype=torch.float32)
    for lo in range(0, n_local, 65536):
        hi = min(n_local, lo + 65536)
        which = torch.randint(0, args.lists, (hi - lo,), generator=g, device=env.dev)
        rows[lo:hi] = comp[which] + 0.3 * torch.randn((hi - lo, args.dim), generator=g, device=env.dev)
    ns_local = min(n_local, max(args.lists * 50, 10000) // world)      # src/ivfbuild.c:448-452, split over the ranks
    samp = rows[torch.randperm(n_local, generator=g, device=env.dev)[:ns_local]].contiguous()
    torch.cuda.synchronize()
    t_rows = pv.Table(pv.VECTOR, args.dim).append(rows)
    del rows
    torch.cuda.empty_cache()
    t_samp = pv.Table(pv.VECTOR, args.dim).append(samp)
    pv.synchronize()
    res = {}

    def build(_):
        t0 = time.perf_counter()
        init = pv.kmeans_pp_init(t_samp, pv.L2, args.lists, seed=42)
        pv.synchronize()
        t1 = time.perf_counter()
        centers, iters = pv.kmeans(t_samp, pv.L2, init, max_iter=500)
        pv.synchronize()
        t2 = time.perf_counter()
        c_dev = torch.from_numpy(centers).to(env.dev)
        assign = pv.assign(t_rows, pv.L2_SQUARED, c_dev)
        pv.synchronize()
        t3 = time.perf_counter()
        res.update(seed_s=t1 - t0, lloyd_s=t2 - t1, assign_s=t3 - t2, iters=iters, centers=c_dev, assign=assign, rechecked=pv.last_assign_rechecked(),
                   pp_stats=pv.kmeans_pp_stats())

    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    l0 = pv.launch_count()
    pv.prof_enable(True)
    pv.prof_read(pv.PROF_ASSIGN)
    ms = timed_steps(env, build, args.steps, args.warmup)
    a_ms, a_n = pv.prof_read(pv.PROF_ASSIGN)
    pv.prof_enable(False)
    launches = pv.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    counts = torch.bincount(res["assign"].to(torch.int64), minlength=args.lists).to(torch.float64)
    if env.dist is not None:
        env.dist.all_reduce(counts)
    # recall@10 of the resulting index: every rank serves its own rows under the global list numbering
    recall = None
    free_b, _ = torch.cuda.mem_get_info()
    if not args.no_recall and free_b > n_local * args.dim * 4 * 1.15:
        try:
            recall = recall_d(env, args, comp, t_rows, res)
        except Exception as e:       # the measurement above stands; say why the check is missing
            recall = {"error": str(e)[:200]}
    if rank == 0:
        _, tf_peak, peak_src = measured_peaks()
        step_s = ms / args.steps / 1000.0
        flops_assign = 2.0 * args.rows * args.lists * args.dim
        lens = counts.cpu().numpy()
        line = {"metric": D_METRIC,
                "value": args.rows / step_s, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (assign: split-bf16 tcgen05 products, exact fp32 re-check)",
                "data": "synthetic",
                "config": {"workload": f"IVFFlat k-means build {args.rows}x{args.dim} fp32, lists={args.lists}, samples={ns_local * world} (BASELINE.json configs[3])",
                           "data_law": f"mixture of {args.lists} Gaussians (sigma 0.3), seeds 3 / 1000 + rank", "parallelism":
                               f"rows and samples sharded over {world} rank(s); ncclAllReduce of centre sums / counts / change counter per Lloyd iteration, "
                               "ncclAllGather + ncclAllReduce per k-means++ centre, all inside libvecb200; assign is collective-free",
                           "l2_policy": "inputs larger than L2 (%d MB of rows per rank)" % (n_local * args.dim * 4 // 2**20)},
                "phases_s": {"kmeans_pp_seeding": res["seed_s"], "lloyd": res["lloyd_s"], "lloyd_iterations": res["iters"], "assign": res["assign_s"],
                             "kmeans_pp_samples_skipped_by_triangle_rule / stopped_by_bf16_bound / rescored_exactly": list(res["pp_stats"])},
                "roofline": roofline_d(args, world, ns_local, a_ms, a_n, args.steps + args.warmup, tf_peak, peak_src, res),
                "list_sizes": {"min": int(lens.min()), "mean": float(lens.mean()), "max": int(lens.max()), "empty": int((lens == 0).sum())},
                "recall_at_10": recall, "cpu_baseline": None,
                "e2e": {"value": args.rows / step_s, "unit": "rows/s", "h2d_bytes_per_step": args.lists * args.dim * 4, "d2h_bytes_per_step": args.lists * args.dim * 4 * 2,
                        "note": "rows are resident (uploaded once, like the heap scan feeding the build); centres travel host <-> device every phase"},
                "gpu_launches": int(launches), "clocks": clocks}
        print(json.dumps(line))
    env.close()
    return 0


def roofline_d(args, world, ns_local, a_ms, a_n, builds, tf_peak, peak_src, res):
    """every bracketed assign launch of the timed + warm-up builds: one pass over the local samples per Lloyd iteration,
    one pass over all local rows at the end; 2 x rows x lists x dim useful flops each, x 3 bf16 products issued"""
    if not a_n:
        return None
    per_build = a_n / builds
    rows_scored = (per_build - 1) * ns_local + args.rows / world          # per build, per rank
    issued = 3.0 * 2.0 * rows_scored * args.lists * args.dim * builds
    tf = issued / (a_ms / 1000.0) / 1e12
    return {"bound": "tensor", "kernel": "assign_tc_kernel (tcgen05 split-bf16 GEMM + fused argmin) + exact re-check of flagged rows",
            "achieved": tf, "peak": tf_peak, "peak_source": peak_src, "unit": "TFLOP/s", "frac": tf / tf_peak, "traffic": None,
            "useful_tflops": tf / 3.0, "assign_launches_per_build": per_build, "ms_per_build_in_assign": a_ms / builds,
            "note": "issued bf16 MMA flops (3 products per fp32-accurate term) over the CUDA-event time of every assign call of a build "
                    "(Lloyd iterations on the samples + the final pass over all rows), exact re-checks included",
            "rows_rechecked_exactly_last_assign": res["rechecked"]}


def recall_d(env, args, comp, t_rows, res):
    """recall@10, probes = 10, of the index the build produced; exact truth by brute force over the sharded rows"""
    torch, pv = env.torch, env.pv
    import ctypes as C
    k, nq = 10, 256
    g = torch.Generator(device=env.dev).manual_seed(4)
    which = torch.randint(0, args.lists, (nq,), generator=g, device=env.dev)
    queries = (comp[which] + 0.3 * torch.randn((nq, args.dim), generator=g, device=env.dev)).contiguous()
    n_local = len(t_rows)
    # exact truth first (brute force over this rank's rows, merged over the ranks below)
    ex_ids, ex_d = t_rows.exact_topk(pv.L2_SQUARED, queries, k)
    ex_ids = ex_ids + env.rank * n_local
    # local image: this rank's rows grouped by their (global) list
    assign = res["assign"].to(torch.int64)
    order = torch.argsort(assign, stable=True)
    counts = torch.bincount(assign, minlength=args.lists)
    offsets = torch.zeros(args.lists + 1, dtype=torch.int64)
    offsets[1:] = torch.cumsum(counts.cpu(), 0)
    rows_view = table_rows_view(pv, t_rows, n_local, args.dim, env.dev)
    grouped = torch.empty((n_local, args.dim), dtype=torch.float32, device=env.dev)
    for lo in range(0, n_local, 65536):
        grouped[lo:lo + 65536] = rows_view[order[lo:lo + 65536]]
    torch.cuda.synchronize()
    del rows_view
    t_rows.free()                        # (the timed builds are over) make room for the index image
    gid = (order + env.rank * n_local).contiguous()
    pv.set_option("scan_impl", 3)        # exact list-major kernel: no second copy of the rows as packed planes
    ix = pv.IvfflatIndex("vector_l2_ops", args.dim, args.lists).load(res["centers"], offsets.numpy(), grouped, gid)
    pv.synchronize()
    del grouped
    torch.cuda.empty_cache()
    ids = torch.empty((nq, k), dtype=torch.int64, device=env.dev)
    dist = torch.empty((nq, k), dtype=torch.float32, device=env.dev)
    if env.world > 1:
        ix.search_sharded_into(queries, k, 10, ids, dist)
    else:
        ix.search_into(queries, k, 10, ids, dist)
    pv.synchronize()
    if env.dist is not None:
        gi = [torch.empty_like(ex_ids) for _ in range(env.world)]
        gd = [torch.empty_like(ex_d) for _ in range(env.world)]
        env.dist.all_gather(gi, ex_ids)
        env.dist.all_gather(gd, ex_d)
        alli, alld = torch.cat(gi, 1), torch.cat(gd, 1)
        top = torch.topk(alld, k, dim=1, largest=False)
        ex_ids = torch.gather(alli, 1, top.indices)
    hit = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(ids.cpu(), ex_ids.cpu()))
    ix.free()
    pv.set_option("scan_impl", args.scan_impl)
    return {"value": hit / (nq * k), "probes": 10, "queries": nq}


def table_rows_view(pv, table, n, dim, dev):
    """the rows appended to a vb_table as a torch view (fp32 rows whose dimension is a multiple of 4 are stored unpadded)"""
    import torch
    ptr, stride = table.device_rows()
    if stride != dim * 4:
        raise RuntimeError("padded rows: no dense view")

    class _View:
        __cuda_array_interface__ = {"shape": (n, dim), "typestr": "<f4", "data": (ptr, False), "version": 2}

    return torch.as_tensor(_View(), device=dev)


def main():
    args = parse_args()
    if args.config == "A":
        return run_a(args)
    if args.config in ("C", "E"):
        return run_hnsw(args)
    if args.config == "D":
        return run_d(args)
    if args.impl == "reference":
        return run_b_reference(args)
    return run_b_ours(args)


if __name__ == "__main__":
    sys.exit(main())
