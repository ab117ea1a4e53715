#!/usr/bin/env python
"""bench.py — headline benchmark of the MEVI index hot path on B200.

Metric (BASELINE.json): docs/sec of the RQ encode (M=4 levels x K=32 centroids, d=768, L2) on the
MSMARCO-shape corpus, 8,841,823 x 768 fp32 per GPU, resident in HBM when the timed region starts.
A "step" is one full encode pass over that corpus.  Documents shard across GPUs with no data-path
collective (weak scaling: every rank owns one MSMARCO-shape block).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # our arm
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # reference CPU path

--dump-outputs DIR writes the codes the last timed step computed as DIR/codes.npy (float32 [S, 4]) with their
row indices as DIR/codes_rows.npy (float64 [S]): every row up to 2,097,152 rows per GPU, above that a fixed seeded
sample of that many (48 MiB in all).  The corpus and codebook are seeded, so two builds run with the same arguments
can be compared output for output.  With N > 1 ranks every rank writes its own rank<r>_*.npy (a sample of
2,097,152 / N rows).  Apart from DIR, bench.py writes nothing into the source tree.

The JSON line also carries `roofline` (dominant kernel vs measured HBM peak), `e2e` (same metric
through the reference-shaped Python entry point with HOST buffers, copies inside the timed region),
`cpu_baseline` (the reference's CPU arithmetic, oracle port, bounded sample), `clocks`, `gpu_launches`
and, as its LAST key, `summary`: one compact entry per BASELINE config with ms / value / roofline fraction,
measured in the same run (verbose details go to stderr):
  enc_strong    ONE 8,841,823-row corpus split over the N ranks by the pq.py:218-225 rule (strong scaling)
  train         full train_rq_lloyd on that sharded corpus: 4 levels x 25 Lloyd iterations, one all-reduce each
  km_it         one k-means iteration on the rank's shard: assign + accumulate kernels, all-reduce timed alone (ar_ms)
  rr_stream / rr_group   cluster-restricted re-rank, 6,980 queries x 100 leaves -> top-100 over the sharded corpus
                (all-gather + merge inside the timed region at N > 1, timed alone as ag_ms); frac_img = reuse-aware
                roofline (fp16 tile image bytes / time / HBM peak), frac_nr = no-reuse byte count of SURVEY 8d
  rr_leaf       N > 1 with --rr-leaf: rr_group on a leaf-partitioned index (every leaf whole on one rank)
  rr_clust      the same on the clustered corpus of SURVEY 8d (4,096-Gaussian mixture, sigma 0.3, seed 99)
  enc_nq / flat_nq       NQ shape (21,015,324 x 768 over the N ranks): encode, exact flat IP top-100 of 3,610 queries
  flat          exact flat IP top-100, 6,980 queries x the sharded MSMARCO-shape corpus
  wid           SURVEY 8f rows (PQ encode, beam search, inverted lists)
  cpu           reference CPU legs on the host cores (BASELINE.md B1/B4/B5; bounded samples), N = 1 only
  dist_check    N > 1: sharded flat / re-rank / training results equal the single-GPU ones on a small problem
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_MARCO, D, M_LEVELS, K_CENTS = 8841823, 768, 4, 32
NQ_MARCO, TOPK, LEAVES = 6980, 100, 100
N_NQ, NQ_NQ = 21015324, 3610  # NQ-DPR corpus (dataprocess/NQ_dpr/get_inverse_answers.py:17), NQ-test queries
GOLDEN_CB = os.path.join(ROOT, "tests", "golden", "gauss768", "codebook.pt")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), float(j.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.samples = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.samples:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                clk, cmx = float(parts[0]), float(parts[1])
            except ValueError:
                continue
            mx = cmx
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                try:
                    power.append(float(parts[2]))
                except ValueError:
                    pass
                for nm, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


_ORIG_AFFINITY = set()


def bind_to_gpu_numa_node(local_rank):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (sysfs `local_cpulist` of the GPU's PCI device):
    with N ranks each pulling 27 GB of pinned host rows, buffers that all land on one node halve the H2D rate."""
    try:
        import torch

        p = torch.cuda.get_device_properties(local_rank)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        cpus = set()
        for part in open(f"{base}/local_cpulist").read().strip().split(","):
            if not part:
                continue
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        _ORIG_AFFINITY.update(allowed)  # the CPU-baseline child gets every core back
        cpus &= allowed
        if not cpus:
            return "unchanged (no local_cpulist inside the allowed set)"
        os.sched_setaffinity(0, cpus)
        node = open(f"{base}/numa_node").read().strip()
        return f"GPU {bdf} numa_node {node}, {len(cpus)} CPUs"
    except Exception as e:
        return f"unchanged ({type(e).__name__}: {e})"[:160]


def make_corpus(n, d, device, seed):
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    X = torch.empty((n, d), dtype=torch.float32, device=device)
    step = 1 << 20
    for a in range(0, n, step):
        b = min(a + step, n)
        X[a:b].normal_(generator=g)
    return X


def load_codebook():
    import torch

    return torch.load(GOLDEN_CB, map_location="cpu", weights_only=False).detach().contiguous()


# --------------------------------------------------------------------------- #
def reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path (torch CPU ops of pq.py:281-305, batch 128
    as main_models.py:3208) on the host cores — the oracle port, since the reference is Python and
    /root/reference does not exist on the GPU box.  Each step encodes a bounded sample of the workload:
    up to --ref-sample rows (default 1,048,576), shrunk so that the whole run stays within ~2.5 minutes."""
    if rank != 0:
        return
    import numpy as np
    import torch

    from oracle import oracle

    torch.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1; the reference uses every core
    torch.manual_seed(1234)
    cb = load_codebook()
    probe = torch.randn(32768, D).numpy()
    for _ in range(max(args.warmup, 1)):
        oracle.rq_encode(probe[:8192], cb, batch_size=128)
    t0 = time.perf_counter()
    oracle.rq_encode(probe, cb, batch_size=128)
    rate = len(probe) / (time.perf_counter() - t0)
    S = int(min(args.ref_sample, max(65536, rate * 150.0 / max(args.steps, 1))))
    X = torch.randn(S, D).numpy()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        codes = oracle.rq_encode(X, cb, batch_size=128)
    dt = time.perf_counter() - t0
    value = S * args.steps / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "rq_encode_docs_per_sec", "value": value, "unit": "docs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: MSMARCO-shape RQ encode, M=4 K=32 d=768 L2 (reference CPU path, pq.py:281-305, batch 128)",
                   "sample_rows_per_step": S, "host_threads": cores},
        "cpu_baseline": {"value": value, "unit": "docs/s", "cores": cores, "kind": "port",
                         "sample": f"{S} x {D} fp32 rows per step, N(0,1), reference-trained codebook"},
        "e2e": {"value": value, "unit": "docs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "codes_checksum": int(np.asarray(codes, dtype=np.int64).sum()),
    }
    print(json.dumps(line), flush=True)


def r3(x):
    """3-4 significant digits for the compact summary."""
    if x is None:
        return None
    x = float(x)
    if x == 0 or x != x:
        return x
    from math import floor, log10

    return round(x, max(0, 3 - int(floor(log10(abs(x))))))


# --------------------------------------------------------------------------- #
def our_arm(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist

    import mevi_b200
    from mevi_b200.dist_utils import all_gather_stack, shard_bounds
    from mevi_b200.pq import ProductQuantization

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)  # pinned host buffers of the e2e leg then live next to this GPU's PCIe root
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = mevi_b200.get_context(local_rank)
    hbm_peak, bf16_peak, peak_src = measured_peaks()
    n = args.docs
    log(f"[rank {rank}] host affinity: {numa}")
    log(f"[rank {rank}] generating {n} x {D} fp32 corpus on {torch.cuda.get_device_name(dev)}")
    X = make_corpus(n, D, dev, 1234 + rank)
    cb_cpu = load_codebook()
    cb = cb_cpu.to(dev)
    codes = torch.empty((n, M_LEVELS), dtype=torch.int32, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        ctx.rq_encode(X, cb, metric="l2", mode=args.mode, codes=codes)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launches
    barrier()
    t_wall0 = time.time()
    start.record()
    for _ in range(args.steps):
        step()
    stop.record()
    barrier()
    t_wall1 = time.time()
    ctx.check()
    launches = ctx.launches - l0
    if args.dump_outputs:
        dump_codes(args.dump_outputs, codes, rank, world)
    ms = torch.tensor([start.elapsed_time(stop)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    ms_step = ms_total / args.steps
    value = world * n / (ms_step / 1e3)
    _, stats = ctx.rq_encode(X[: min(n, 1 << 20)], cb, mode=args.mode, return_stats=True)
    flagged_frac = float(stats[0].item()) / max(1, int(stats[1].item()))
    refined_frac = float(stats[2].item()) / max(1, int(stats[1].item()))
    checksum = int(codes.to(torch.int64).sum().item())

    # kernel-vs-kernel agreement of the fast path with the exact path on a sample (both product kernels)
    ns_chk = min(n, 1 << 18)
    exact = ctx.rq_encode(X[:ns_chk], cb, mode="exact")
    mismatch = int((exact != codes[:ns_chk]).any(dim=1).sum().item())
    del exact

    algo_bytes = n * D * 4 + n * M_LEVELS * 4
    achieved = algo_bytes / (ms_step / 1e3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tpath):
        try:
            traffic = json.load(open(tpath)).get("rq_encode_dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": "rq_encode (all 4 levels, one pass over the corpus)", "algorithmic_bytes_per_launch": algo_bytes}

    # ---- e2e through the reference-shaped entry point with host buffers ----------------------
    e2e = None
    try:
        import psutil

        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    n_e2e = n
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))  # every rank of the node pins its own host copy
    while n_e2e * D * 4 * 1.3 > avail * 0.6 / max(1, local_world) and n_e2e > 1 << 18:
        n_e2e //= 2
    pq = ProductQuantization("rq", M_LEVELS, 5, "l2", D, "kmeans", "grad")
    pq.kernel_mode = args.mode
    pq.device_index = local_rank
    with torch.no_grad():
        pq.codebook.copy_(cb_cpu)
    Xh = torch.empty((n_e2e, D), dtype=torch.float32, pin_memory=True)
    Xh.copy_(X[:n_e2e])
    cluster = torch.empty((n_e2e, M_LEVELS), dtype=torch.int32).pin_memory()
    Xh_np = Xh.numpy()
    pq.get_rq_document_cluster(Xh_np[: 1 << 16], cluster[: 1 << 16], 0, min(n_e2e, 1 << 16), rank, 128)  # warm-up
    barrier()
    e2e_steps = max(1, min(args.steps, 3))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        pq.get_rq_document_cluster(Xh_np, cluster, 0, n_e2e, rank, 128)
    e1.record()
    barrier()
    e_ms = torch.tensor([e0.elapsed_time(e1) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    e2e_ok = bool((cluster.to(dev) == codes[:n_e2e]).all().item())
    e2e = {"value": world * n_e2e / (float(e_ms.item()) / 1e3), "unit": "docs/s",
           "h2d_bytes_per_step": n_e2e * D * 4 + int(cb_cpu.numel()) * 4, "d2h_bytes_per_step": n_e2e * M_LEVELS * 4,
           "rows_per_step": n_e2e, "ms_per_step": float(e_ms.item()), "steps": e2e_steps,
           "api": "ProductQuantization.get_rq_document_cluster(np.ndarray) -> mevi_rq_encode_host (pinned host rows, 256k-row chunks)",
           "codes_equal_device_path": e2e_ok}
    del Xh, Xh_np, cluster

    # host sample for the CPU legs (taken before the corpus is reused by the other configs)
    cpu_sample_path = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_sample_path = save_cpu_sample(X, codes)

    summary, details = {}, {}
    summary["n"] = world
    summary["enc"] = {"ms": r3(ms_step), "frac": r3(achieved / hbm_peak)}
    details["enc"] = {"flagged_fraction": flagged_frac, "refined_fraction": refined_frac}
    if not args.no_extras:
        if world > 1:
            try:
                summary["dist_check"] = dist_check(ctx, dev, rank, world)
            except Exception as e:
                summary["dist_check"] = "error: " + repr(e)[:100]
        run_configs(args, ctx, X, cb, codes, dev, rank, world, hbm_peak, bf16_peak, summary, details)
        del X, codes
        torch.cuda.empty_cache()
        if not args.no_nq:
            run_nq(args, ctx, cb, dev, rank, world, hbm_peak, bf16_peak, summary, details)

    cpu_baseline = None
    if cpu_sample_path is not None:
        legs = cpu_legs(cpu_sample_path)
        cpu_baseline = legs.pop("encode", None)
        summary["cpu"] = legs.get("summary", {"error": legs.get("error")})
        details["cpu_legs"] = legs

    if rank == 0:
        log("details: " + json.dumps(details))
        line = {
            "metric": "rq_encode_docs_per_sec", "value": value, "unit": "docs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: MSMARCO-shape RQ encode, 8,841,823 x 768 fp32 per GPU, M=4 K=32 L2, "
                                   "codebook trained by the reference (sklearn, seed 41) on N(0,1) data",
                       "docs_per_gpu": n, "parallelism": f"doc-sharded x{world}, no data-path collective",
                       "kernel_mode": args.mode, "l2_policy": "inputs (27.2 GB per GPU) are larger than L2 (126 MB)",
                       "timing": "CUDA events on the launch stream, max over ranks"},
            "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu_baseline, "clocks": clocks, "gpu_launches": launches,
            "codes_checksum": checksum, "prefilter_flagged_fraction": flagged_frac,
            "fast_vs_exact_kernel_mismatch_rows": {"rows": ns_chk, "mismatch": mismatch},
            "summary": summary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_ROWS = 1 << 21  # per run: codes as float32 (16 B a row) + row indices as float64 (8 B a row) = 48 MiB


def dump_codes(out_dir, codes, rank, world):
    """codes [n, M] int32 on the device -> out_dir/[rank<r>_]codes.npy (float32, exact below 2^24) and codes_rows.npy
    (float64 row indices, ascending): all rows, or a seeded sample of DUMP_ROWS / world of them."""
    import numpy as np
    import torch

    n = codes.shape[0]
    S = DUMP_ROWS // world
    rows = np.arange(n) if n <= S else np.sort(np.random.default_rng(rank).choice(n, size=S, replace=False))
    picked = codes[torch.from_numpy(rows).to(codes.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    np.save(os.path.join(out_dir, prefix + "codes.npy"), picked.astype(np.float32))
    np.save(os.path.join(out_dir, prefix + "codes_rows.npy"), rows.astype(np.float64))


# --------------------------------------------------------------------------- #
def save_cpu_sample(X, codes):
    """First rows of the bench corpus + their codes -> /dev/shm for the CUDA-free child process."""
    import tempfile

    import numpy as np

    S = int(min(1 << 19, X.shape[0]))
    shm = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    path = os.path.join(shm, f"mevi_bench_sample_{os.getpid()}.npz")
    np.savez(path, X=X[:S].cpu().numpy(), codes=codes[:S].cpu().numpy())
    return path


def cpu_legs(path):
    """Reference CPU arithmetic on bounded samples of the same workloads, in a CHILD process that never
    initialises CUDA: inside a CUDA process every munmap of the 12.6 MB torch temporaries goes through the
    UVM notifier and the CPU path runs ~10x slower than the reference would on its own."""
    try:
        restore = (lambda: os.sched_setaffinity(0, _ORIG_AFFINITY)) if _ORIG_AFFINITY else None
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "cpu-baseline-child", "--sample-file", path],
                             capture_output=True, text=True, timeout=900, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                             preexec_fn=restore)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)
    except Exception as e:
        return {"error": repr(e)[:300]}
    finally:
        try:
            os.remove(path)
        except OSError:
            pass


def cpu_baseline_child(args):
    """BASELINE.md section 4 on the host cores (oracle = the reference's arithmetic; the only place bench.py runs it):
    B2 encode (pq.py:281-305, batch 128), B1/B3 one level of the reference build (sklearn MiniBatchKMeans with the
    reference's hyper-parameters, pq.py:551-598) on 100k rows, B4 the re-rank loop (main_models.py:3915-4014) and
    B5 flat IP (faiss IndexFlatIP semantics in numpy), each on a bounded sample."""
    import numpy as np
    import torch

    from oracle import oracle

    torch.set_num_threads(os.cpu_count() or 1)
    z = np.load(args.sample_file)
    X, codes = z["X"], z["codes"]
    cb_cpu = load_codebook()
    cores = torch.get_num_threads()
    out = {}
    # ---- B2: encode
    sample = X[: 1 << 18]
    oracle.rq_encode(sample[:8192], cb_cpu, batch_size=128)  # warm-up (allocator, threads)
    t0 = time.perf_counter()
    oracle.rq_encode(sample[:32768], cb_cpu, batch_size=128)
    rate = 32768 / (time.perf_counter() - t0)
    reps = int(max(1, min(64, round(rate * 12.0 / len(sample)))))
    t0 = time.perf_counter()
    for _ in range(reps):
        oracle.rq_encode(sample, cb_cpu, batch_size=128)
    dt = time.perf_counter() - t0
    out["encode"] = {"value": len(sample) * reps / dt, "unit": "docs/s", "cores": cores, "kind": "port",
                     "sample": f"first {len(sample)} rows of the bench corpus x {reps} passes, torch CPU restatement of "
                               f"pq.py:281-305 (batch 128) in a CUDA-free child process, {dt:.1f} s",
                     "host_cpus": os.cpu_count()}
    summ = {"cores": cores, "enc_docs_s": r3(out["encode"]["value"])}
    # ---- B1/B3: one level of the reference build on 100k x 768
    try:
        t0 = time.perf_counter()
        oracle.rq_build_reference(X[:100000], M_LEVELS, K_CENTS, 41, levels=1)
        dt = time.perf_counter() - t0
        out["build"] = {"seconds_per_level": dt, "rows": 100000, "levels_timed": 1, "kind": "port",
                        "note": "sklearn MiniBatchKMeans(n_init=100, batch 1000, max_iter 300), pq.py:557-563; the reference "
                                "runs 4 such levels on rank 0, cost almost independent of N"}
        summ["build_s_lvl"] = r3(dt)
    except Exception as e:
        out["build"] = {"error": repr(e)[:200]}
    # ---- B4: re-rank loop on the sample corpus (queries x 100 leaves)
    try:
        clus, _ = oracle.document_cluster(codes)
        rs = np.random.RandomState(4321)
        nq = 24
        Q = rs.standard_normal((nq, D)).astype(np.float32)
        dec, _ = oracle.beam_search(torch.as_tensor(cb_cpu), torch.from_numpy(Q), LEAVES)
        oracle.cluster_rerank(Q[:2], X, clus, dec[:2].numpy(), topk=TOPK)
        t0 = time.perf_counter()
        res = oracle.cluster_rerank(Q, X, clus, dec.numpy(), topk=TOPK)
        dt = time.perf_counter() - t0
        ncand = float(np.mean([r[2] for r in res]))
        out["rerank"] = {"queries_per_sec": nq / dt, "candidates_per_sec": nq * ncand / dt, "corpus_rows": int(len(X)),
                         "candidates_mean": ncand, "queries": nq, "kind": "port",
                         "note": "main_models.py:3915-4014 restated (dict lookup, row gather, q.P^T in 1024-row chunks, "
                                 "descending sort); candidate counts scale with the corpus, compare candidates/s"}
        summ["rr_cand_s"] = r3(nq * ncand / dt)
    except Exception as e:
        out["rerank"] = {"error": repr(e)[:200]}
    # ---- B5: flat IP
    try:
        rs = np.random.RandomState(4321)
        nq = 256
        Q = rs.standard_normal((nq, D)).astype(np.float32)
        oracle.flat_ip_topk_partition(Q[:8], X[:65536], TOPK)
        t0 = time.perf_counter()
        oracle.flat_ip_topk_partition(Q, X, TOPK)
        dt = time.perf_counter() - t0
        out["flat_ip"] = {"pairs_per_sec": nq * len(X) / dt, "tflops": 2.0 * nq * len(X) * D / dt / 1e12, "queries": nq,
                          "corpus_rows": int(len(X)), "kind": "port",
                          "note": "numpy sgemm blocks + argpartition top-k (faiss IndexFlatIP semantics, BASELINE.md B5; faiss is not installable here)"}
        summ["flat_pairs_s"] = r3(nq * len(X) / dt)
    except Exception as e:
        out["flat_ip"] = {"error": repr(e)[:200]}
    out["summary"] = summ
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------- #
def run_configs(args, ctx, X, cb, codes, dev, rank, world, hbm_peak, bf16_peak, summary, details):
    """The other BASELINE.json configs on the stated shapes (see the module docstring).  Every leg is wrapped: a
    failure becomes an `error` entry, never a lost headline line."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from mevi_b200.dist_utils import all_gather_stack, shard_bounds
    from mevi_b200.pq import ProductQuantization
    from mevi_b200.rerank import ClusterIndex, ClusterReranker
    from mevi_b200.trainer import train_rq_lloyd

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(fn, reps, warm=1):
        for _ in range(warm):
            fn()
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def leg(name):
        def deco(fn):
            try:
                t0 = time.time()
                fn()
                log(f"[rank {rank}] leg {name}: {time.time() - t0:.1f} s")
            except Exception as e:  # a leg must never kill the headline line
                import traceback

                summary[name] = {"error": repr(e)[:160]}
                details[name] = {"error": traceback.format_exc()[-1500:]}
                torch.cuda.synchronize()
            return fn
        return deco

    # ---- the strong-scaling shard: ONE 8,841,823-row corpus over the N ranks (pq.py:218-225) -----------------
    s0, s1 = shard_bounds(N_MARCO if args.docs == N_MARCO else args.docs, rank, world)
    ns = s1 - s0
    n_total = N_MARCO if args.docs == N_MARCO else args.docs
    Xs, codes_s = X[:ns], codes[:ns]
    shard_bytes = ns * D * 4
    g = torch.Generator(device=dev)
    g.manual_seed(4321)
    Q = torch.empty((NQ_MARCO, D), device=dev).normal_(generator=g)
    state = {}

    @leg("enc_strong")
    def _():
        ms = timed(lambda: ctx.rq_encode(Xs, cb, metric="l2", mode=args.mode, codes=codes_s), max(3, min(args.steps, 10)))
        summary["enc_strong"] = {"ms": r3(ms), "docs_s": r3(n_total / (ms / 1e3)), "frac": r3((shard_bytes + ns * 16) / (ms / 1e3) / 1e9 / hbm_peak)}
        details["enc_strong"] = {"rows_total": n_total, "rows_this_rank": ns}

    # collectives, timed alone (SURVEY 8d "Collectives")
    ar_ms = ag_ms = None
    if world > 1:
        buf = torch.zeros(K_CENTS * D + K_CENTS, device=dev)
        ar_ms = timed(lambda: dist.all_reduce(buf), 50, warm=5)
        sc0 = torch.zeros((NQ_MARCO, TOPK), device=dev)
        id0 = torch.zeros((NQ_MARCO, TOPK), dtype=torch.int64, device=dev)
        ag_ms = timed(lambda: (all_gather_stack(sc0), all_gather_stack(id0)), 20, warm=3)
        mg_ms = timed(lambda: ctx.topk_merge(all_gather_stack(sc0).contiguous(), all_gather_stack(id0).contiguous()), 10, warm=2)
        details["collectives"] = {"allreduce_98KB_ms": ar_ms, "allgather_topk_ms": ag_ms, "allgather_plus_merge_ms": mg_ms}

    @leg("km_it")
    def _():
        # centroids as the trainer has them: K data rows (k-means++ draws data points), moved by the updates of the
        # warm-up iteration - balanced clusters, unlike the reference-trained level-0 codebook (80 % of rows in two cells)
        gk = torch.Generator(device=dev)
        gk.manual_seed(41)
        C = Xs[torch.randint(0, ns, (K_CENTS,), device=dev, generator=gk)].clone()
        buf = torch.empty(K_CENTS * D + K_CENTS, device=dev)
        assign = torch.empty(ns, dtype=torch.int32, device=dev)

        def km():
            ctx.kmeans_step(Xs, C, buf, assign=assign, mode=args.mode)
            if world > 1:
                dist.all_reduce(buf)
            ctx.kmeans_update(buf, C)

        ms = timed(km, 5)
        a2 = assign.view(ns, 1)
        ms_assign = timed(lambda: ctx.rq_encode(Xs, C[None], metric="l2", mode=args.mode, codes=a2), 5)
        ms_accum = timed(lambda: ctx.accumulate_by_code(Xs, assign, K_CENTS, buf), 5)
        fr = lambda m: (shard_bytes + ns * 4) / (m / 1e3) / 1e9 / hbm_peak
        # one-pass iteration (mevi_kmeans_step_fused): assignment + sums under the previous assignment in one read of the
        # shard, then the rows whose assignment changed are moved between centroids; steady state = after 3 iterations
        ms_fused = ms_fpass = changed = None
        try:
            a_prev, a_cur = assign, torch.empty_like(assign)
            moved = torch.empty((ns // 4 + 1, D), device=dev)

            def km_fused():
                nonlocal a_prev, a_cur, changed
                ctx.kmeans_step_fused(Xs, C, a_prev, a_cur, buf)
                ch = torch.nonzero(a_cur != a_prev).squeeze(1)
                changed = int(ch.numel())
                if changed > ns // 4:
                    ctx.accumulate_by_code(Xs, a_cur, K_CENTS, buf)
                elif changed:
                    mv = ctx.gather_rows(Xs, ch.to(torch.int32), out=moved)
                    buf.add_(ctx.accumulate_by_code(mv, a_cur[ch].contiguous(), K_CENTS)).sub_(ctx.accumulate_by_code(mv, a_prev[ch].contiguous(), K_CENTS))
                if world > 1:
                    dist.all_reduce(buf)
                ctx.kmeans_update(buf, C)
                a_prev, a_cur = a_cur, a_prev

            ms_fused = timed(km_fused, 5, warm=3)
            ms_fpass = timed(lambda: ctx.kmeans_step_fused(Xs, C, a_prev, a_cur, buf), 5)
            del moved
        except Exception as e:
            details["km_it_fused_error"] = repr(e)[:200]
        # incremental iteration (mevi_kmeans_step_delta, the trainer's default): the assignment pass is the only read of the
        # shard; float64 running sums are corrected by the rows that moved (no host synchronisation in the iteration)
        ms_delta = moved_frac = None
        try:
            a_prev, a_cur = assign, torch.empty_like(assign)
            master = torch.empty(K_CENTS * D + K_CENTS, dtype=torch.float64, device=dev)
            nchg = torch.zeros(1, dtype=torch.int32, device=dev)
            ctx.kmeans_step(Xs, C, buf, assign=a_prev, mode=args.mode)
            master.copy_(buf)

            def km_delta():
                nonlocal a_prev, a_cur
                ctx.kmeans_step_delta(Xs, C, a_prev, a_cur, master, buf, n_changed=nchg, mode=args.mode)
                if world > 1:
                    dist.all_reduce(buf)
                ctx.kmeans_update(buf, C)
                a_prev, a_cur = a_cur, a_prev

            ms_delta = timed(km_delta, 5, warm=3)
            moved_frac = float(nchg.item()) / ns
            del master
        except Exception as e:
            details["km_it_delta_error"] = repr(e)[:200]
        best = ms_delta or ms_fused or ms
        summary["km_it"] = {"ms": r3(best), "frac": r3(shard_bytes / (best / 1e3) / 1e9 / hbm_peak), "moved": r3(moved_frac),
                            "fused_ms": r3(ms_fused), "pass_ms": r3(ms_fpass), "two_pass_ms": r3(ms), "assign_ms": r3(ms_assign),
                            "accum_ms": r3(ms_accum), "ar_ms": r3(ar_ms)}
        details["km_it_changed_rows_last"] = changed
        details["km_it"] = {"assign_frac": fr(ms_assign), "accum_frac": fr(ms_accum), "rows_total": n_total,
                            "note": "frac = ONE pass over the shard / iteration time; the iteration makes two passes"}

    @leg("train")
    def _():
        sync_all()
        t0 = time.perf_counter()
        cbt, _ = train_rq_lloyd(Xs, M=M_LEVELS, K=K_CENTS, seed=41, iters=25, tol=None, mode=args.mode, device_index=dev.index,
                                presharded=True)
        sync_all()
        dt = time.perf_counter() - t0
        info = train_rq_lloyd.last_info
        iters = sum(l["iters"] for l in info["levels"])
        loop = sum(l["loop_ms_per_iter"] * l["iters"] for l in info["levels"]) / iters
        summary["train"] = {"s": r3(dt), "iters": iters, "loop_ms_per_it": r3(loop), "mse": r3(info["levels"][-1]["mse"])}
        details["train"] = info
        del cbt

    @leg("rr")
    def _():
        pq = ProductQuantization("rq", M_LEVELS, 5, "l2", D, "kmeans", "grad")
        with torch.no_grad():
            pq.codebook.copy_(cb.cpu())
        ctx.rq_encode(Xs, cb, metric="l2", mode=args.mode, codes=codes_s)
        dec = torch.cat([pq.beam_search(Q[a : a + 1024], LEAVES) for a in range(0, NQ_MARCO, 1024)])
        index = ClusterIndex.from_codes(codes_s, K_CENTS, id_base=s0, device_index=dev.index)
        ql = index.lookup(dec)
        D_leaf = ctx.gather_rows(Xs, index.leaf_docids)
        res = {}

        def rr():
            sc, ids, nc = ctx.cluster_rerank(Q, D_leaf, index.leaf_offsets, index.leaf_docids, ql, TOPK, id_base=s0, leaf_ordered=True)
            if world > 1:
                sc, ids = ctx.topk_merge(all_gather_stack(sc).contiguous(), all_gather_stack(ids).contiguous())
            res["out"] = (sc, ids, nc)

        ms = timed(rr, 2)
        ncand = res["out"][2].to(torch.float64)
        if world > 1:
            dist.all_reduce(ncand)
        cand_total = float(ncand.sum().item())
        gathered_local = float(res["out"][2].to(torch.float64).sum().item()) * D * 4
        summary["rr_stream"] = {"ms": r3(ms), "qps": r3(NQ_MARCO / (ms / 1e3)), "frac": r3(gathered_local / (ms / 1e3) / 1e9 / hbm_peak),
                                "cand_mean": r3(cand_total / NQ_MARCO), "ag_ms": r3(ag_ms)}
        details["rr_stream"] = {"cand_max": float(ncand.max().item()), "empty_leaf_fraction": float((ql < 0).float().mean().item()),
                                "n_leaves_this_rank": index.n_leaves, "rows_total": n_total}
        # independent check of the streaming kernel: fp32 matmul (TF32 off) + topk over the candidate rows of 4 queries
        prev_tf32 = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            sc_k, id_k, _ = ctx.cluster_rerank(Q, D_leaf, index.leaf_offsets, index.leaf_docids, ql, TOPK, id_base=s0, leaf_ordered=True)
            worst = 0.0
            for qi in (0, 1, NQ_MARCO // 2, NQ_MARCO - 1):
                lv = ql[qi][ql[qi] >= 0].long()
                rows = torch.cat([torch.arange(int(index.leaf_offsets[l]), int(index.leaf_offsets[l + 1]), device=dev) for l in lv.tolist()])
                sref = torch.topk(D_leaf[rows] @ Q[qi], min(TOPK, rows.numel())).values
                worst = max(worst, float(((sc_k[qi, : sref.numel()] - sref).abs() / sref.abs().clamp_min(1e-6)).max().item()))
            summary["rr_stream"]["chk_rel"] = r3(worst)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev_tf32
        # ---- leaf-grouped GEMM formulation (K3g): every leaf read once for all the queries that chose it
        t0 = time.perf_counter()
        rrg = ClusterReranker(None, index, mode="grouped", D_leaf=D_leaf)
        torch.cuda.synchronize()
        t_img = time.perf_counter() - t0
        gres = {}

        def rg():
            gres["out"] = rrg.rerank(Q, dec, topk=TOPK)  # includes the all-gather + merge when torch.distributed is up

        ms_g = timed(rg, 3)
        sg, ig, _ = gres["out"]
        ss, is_, _ = res["out"]
        fin = torch.isfinite(sg) & torch.isfinite(ss)
        img_bytes = float(rrg._grouped["img"].numel()) if rrg._grouped is not None else 0.0
        summary["rr_group"] = {"ms": r3(ms_g), "qps": r3(NQ_MARCO / (ms_g / 1e3)), "path": rrg.last_path,
                               "frac_img": r3(img_bytes / (ms_g / 1e3) / 1e9 / hbm_peak),
                               "frac_nr": r3(gathered_local / (ms_g / 1e3) / 1e9 / hbm_peak),
                               "ids_eq": r3(float((ig == is_).float().mean().item()))}
        details["rr_group"] = {"failed_queries_rerun_by_stream": getattr(rrg, "last_failed_queries", None),
                               "weak_bootstrap_queries": getattr(rrg, "last_weak_queries", None),
                               "max_abs_score_diff_vs_stream": float((sg - ss)[fin].abs().max().item()) if bool(fin.any()) else 0.0,
                               "tile_image_build_s": t_img, "tile_image_bytes": img_bytes}
        del rrg, D_leaf, index, ql
        # ---- the same call on a LEAF-partitioned index (N > 1): every leaf moved whole to one rank by one all-to-all of
        # the rows at index build; the row blocks above give every rank a slice of every leaf
        if world > 1 and args.rr_leaf:
            t0 = time.perf_counter()
            index_l, X_own = ClusterIndex.from_sharded_codes(Xs, codes_s, K_CENTS, s0, device_index=dev.index)
            D_leaf_l = ctx.gather_rows(X_own, index_l.leaf_docids)
            del X_own
            rrl = ClusterReranker(None, index_l, mode="grouped", D_leaf=D_leaf_l)
            torch.cuda.synchronize()
            t_build = time.perf_counter() - t0
            lres = {}

            def rl():
                lres["out"] = rrl.rerank(Q, dec, topk=TOPK)

            ms_l = timed(rl, 3)
            summary["rr_leaf"] = {"ms": r3(ms_l), "qps": r3(NQ_MARCO / (ms_l / 1e3)), "path": rrl.last_path,
                                  "ids_eq": r3(float((lres["out"][1] == is_).float().mean().item()))}
            details["rr_leaf"] = {"rows_this_rank": int(D_leaf_l.shape[0]), "leaves_this_rank": index_l.n_leaves,
                                  "partition_and_index_build_s": t_build}
            del rrl, D_leaf_l, index_l
        del dec

    @leg("flat")
    def _():
        from mevi_b200.faiss_search import FlatIndex

        rows = min(ns, args.flat_docs)
        t0 = time.perf_counter()
        index = FlatIndex(D, device_index=dev.index, piece_rows=rows, mode=args.mode)  # faiss: index.add(doc) once ...
        index.pieces.append((s0, Xs[:rows], ctx.flat_index_create(Xs[:rows])))         # (the shard is already on the device)
        index.ntotal = rows
        torch.cuda.synchronize()
        t_add = time.perf_counter() - t0
        ms = timed(lambda: index.search_device(Q, TOPK), 3)                             # ... index.search(query, k) many
        ms_1000 = timed(lambda: index.search_device(Q[:1024], 1000), 2)
        tf = 2.0 * NQ_MARCO * rows * D / (ms / 1e3) / 1e12
        nchk = 128
        s_t, i_t = index.search_device(Q[:nchk], TOPK)
        s_e, i_e = ctx.flat_ip_topk(Q[:nchk], Xs[:rows], TOPK, id_base=s0, mode="exact")
        if world > 1:
            s_e, i_e = ctx.topk_merge(all_gather_stack(s_e).contiguous(), all_gather_stack(i_e).contiguous())
        ms_oneshot = timed(lambda: ctx.flat_ip_topk(Q, Xs[:rows], TOPK, id_base=s0, mode=args.mode), 2)
        summary["flat"] = {"ms": r3(ms), "tf": r3(tf), "frac": r3(tf / bf16_peak), "add_ms": r3(t_add * 1e3),
                           "k1000_tf": r3(2.0 * 1024 * rows * D / (ms_1000 / 1e3) / 1e12)}
        details["flat"] = {"rows_this_rank": rows, "pairs_per_sec": world * NQ_MARCO * rows / (ms / 1e3),
                           "ids_identical_vs_fp32_kernel": float((i_t == i_e).float().mean().item()),
                           "one_shot_call_ms_incl_image_pass": ms_oneshot, "k1000_1024_queries_ms": ms_1000,
                           "note": "persistent index: the fp16 image is built once by add(); search = query image + GEMM chunks + "
                                   "compactions + exact fp32 re-score (+ all-gather and merge at N > 1)"}
        index.close()

    @leg("wid")
    def _():
        wid = {}
        gq = torch.Generator(device=dev)
        gq.manual_seed(77)
        for Mp, Kp in ((4, 32), (24, 256), (32, 256)):  # K1 route | wide-codebook tensor kernel, widths 32 and 24
            cbp = torch.empty((Mp, Kp, D // Mp), device=dev).normal_(generator=gq)
            cp = torch.empty((ns, Mp), dtype=torch.int32, device=dev)
            ms_pq = timed(lambda: ctx.pq_encode(Xs, cbp, metric="l2", codes=cp), 2)
            wid[f"pq{Mp}x{Kp}"] = r3((shard_bytes + ns * Mp * 4) / (ms_pq / 1e3) / 1e9 / hbm_peak)
            details.setdefault("wid", {})[f"pq_encode_M{Mp}_K{Kp}_ms"] = ms_pq
            del cbp, cp
        ms_beam = timed(lambda: ctx.rq_beam_search(Q, cb, LEAVES, metric="l2", prod=True), 3)
        wid["beam_ms"] = r3(ms_beam)
        ms_inv = timed(lambda: ctx.build_inverted_lists(codes_s, K_CENTS), 3)
        wid["inv_ms"] = r3(ms_inv)
        summary["wid"] = wid

    # ---- clustered corpus of SURVEY 8d: mixture of 4,096 Gaussians, sigma 0.3, seed 99 (the shard is regenerated in place)
    @leg("rr_clust")
    def _():
        gc = torch.Generator(device=dev)
        gc.manual_seed(99)
        centers = torch.empty((4096, D), device=dev).normal_(generator=gc)  # same centres on every rank
        gl = torch.Generator(device=dev)
        gl.manual_seed(99 + 1000 * (rank + 1))
        stepr = 1 << 20
        for a in range(0, ns, stepr):
            b = min(a + stepr, ns)
            lab = torch.randint(0, 4096, (b - a,), device=dev, generator=gl)
            Xs[a:b].normal_(generator=gl).mul_(0.3).add_(centers[lab])
        cbc, codes_c = train_rq_lloyd(Xs, M=M_LEVELS, K=K_CENTS, seed=41, iters=10, tol=None, mode=args.mode,
                                      device_index=dev.index, presharded=True)
        pq = ProductQuantization("rq", M_LEVELS, 5, "l2", D, "kmeans", "grad")
        with torch.no_grad():
            pq.codebook.copy_(cbc.cpu())
        ctx.rq_encode(Xs, cbc, metric="l2", mode=args.mode, codes=codes_s)
        dec = torch.cat([pq.beam_search(Q[a : a + 1024], LEAVES) for a in range(0, NQ_MARCO, 1024)])
        index = ClusterIndex.from_codes(codes_s, K_CENTS, id_base=s0, device_index=dev.index)
        sizes = (index.leaf_offsets[1:] - index.leaf_offsets[:-1]).to(torch.float64)
        ql = index.lookup(dec)
        nc = torch.where(ql >= 0, sizes[ql.clamp(min=0).long()], torch.zeros((), dtype=torch.float64, device=dev)).sum(1)
        if world > 1:
            dist.all_reduce(nc)
        D_leaf = ctx.gather_rows(Xs, index.leaf_docids)
        rrg = ClusterReranker(None, index, mode="grouped", D_leaf=D_leaf)
        out = {"cand_mean": r3(float(nc.mean().item())), "cand_max": r3(float(nc.max().item())),
               "empty": r3(float((ql < 0).float().mean().item()))}
        details["rr_clust"] = {"n_leaves_this_rank": index.n_leaves, "rows_total": n_total, "train": train_rq_lloyd.last_info}
        # a small call first: if the grouped path cannot establish its guarantee here (near-duplicate documents inside a
        # mixture component overflow the margin window) it falls back to the streaming kernel; all 6,980 queries then run
        # only if that stays within a few seconds
        nq_c = 256
        rrg.rerank(Q[:nq_c], dec[:nq_c], topk=TOPK)
        stream_s = float(nc.sum().item()) / world * D * 4 / 5e12
        if rrg.last_path == "grouped" or stream_s < 3.0:
            nq_c = NQ_MARCO
        ms_c = timed(lambda: rrg.rerank(Q[:nq_c], dec[:nq_c], topk=TOPK), 2)
        out.update({"ms": r3(ms_c), "queries": nq_c, "qps": r3(nq_c / (ms_c / 1e3)), "path": rrg.last_path,
                    "tf": r3(2.0 * float(nc[:nq_c].sum().item()) * D / world / (ms_c / 1e3) / 1e12)})
        summary["rr_clust"] = out
        del rrg, D_leaf, index, ql, dec

    return


def run_nq(args, ctx, cb, dev, rank, world, hbm_peak, bf16_peak, summary, details):
    import torch
    import torch.distributed as dist

    from mevi_b200.dist_utils import all_gather_stack, shard_bounds

    def timed(fn, reps, warm=1):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    try:
        s0, s1 = shard_bounds(N_NQ, rank, world)
        nn = s1 - s0
        free = torch.cuda.mem_get_info(dev)[0]
        need = nn * D * 4 * 1.55 + (8 << 30)  # rows + persistent fp16 image of the flat index + slack
        if free < need:
            summary["enc_nq"] = {"error": f"needs {need / 2**30:.0f} GiB, {free / 2**30:.0f} free"}
            return
        Xn = make_corpus(nn, D, dev, 777 + rank)
        cn = torch.empty((nn, M_LEVELS), dtype=torch.int32, device=dev)
        ms = timed(lambda: ctx.rq_encode(Xn, cb, metric="l2", mode=args.mode, codes=cn), 5)
        summary["enc_nq"] = {"ms": r3(ms), "frac": r3((nn * D * 4 + nn * 16) / (ms / 1e3) / 1e9 / hbm_peak)}
        details["enc_nq"] = {"rows_total": N_NQ, "rows_this_rank": nn, "docs_per_sec": N_NQ / (ms / 1e3)}
        del cn
        g = torch.Generator(device=dev)
        g.manual_seed(4322)
        Qn = torch.empty((NQ_NQ, D), device=dev).normal_(generator=g)
        piece = 1 << 22
        from mevi_b200.faiss_search import FlatIndex

        t0 = time.perf_counter()
        index = FlatIndex(D, device_index=dev.index, piece_rows=piece, mode=args.mode)
        for a in range(0, nn, piece):
            b = min(a + piece, nn)
            index.pieces.append((s0 + a, Xn[a:b], ctx.flat_index_create(Xn[a:b])))
        index.ntotal = nn
        torch.cuda.synchronize()
        t_add = time.perf_counter() - t0
        ms = timed(lambda: index.search_device(Qn, TOPK), 2)
        tf = 2.0 * NQ_NQ * nn * D / (ms / 1e3) / 1e12
        summary["flat_nq"] = {"ms": r3(ms), "qps": r3(NQ_NQ / (ms / 1e3)), "tf": r3(tf), "frac": r3(tf / bf16_peak), "add_ms": r3(t_add * 1e3)}
        details["flat_nq"] = {"rows_total": N_NQ, "queries": NQ_NQ, "piece_rows": piece}
        index.close()
    except Exception as e:
        import traceback

        summary.setdefault("flat_nq", {"error": repr(e)[:160]})
        details["nq_error"] = traceback.format_exc()[-1500:]


def dist_check(ctx, dev, rank, world):
    """N > 1: the sharded paths give the single-GPU answers on a small problem (product kernels on both sides)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from mevi_b200.dist_utils import all_gather_stack, shard_bounds
    from mevi_b200.pq import ProductQuantization
    from mevi_b200.rerank import ClusterIndex, ClusterReranker
    from mevi_b200.trainer import train_rq_lloyd

    g = torch.Generator(device=dev)
    g.manual_seed(5)
    n, d = 60001, 768
    Xall = torch.empty((n, d), device=dev).normal_(generator=g)  # same seed on every rank -> same corpus
    Qs = torch.empty((64, d), device=dev).normal_(generator=g)
    s, e = shard_bounds(n, rank, world)
    # training: every rank ends with the same codebook
    cbk, codes_l = train_rq_lloyd(Xall[s:e], M=4, K=32, seed=41, iters=5, tol=None, device_index=dev.index, presharded=True)
    allcb = all_gather_stack(cbk)
    ok_train = all(bool(torch.equal(allcb[0], allcb[r])) for r in range(world))
    # flat: sharded + merged == single GPU
    sc, ids = ctx.flat_ip_topk(Qs, Xall[s:e].contiguous(), 100, id_base=s)
    sc, ids = ctx.topk_merge(all_gather_stack(sc).contiguous(), all_gather_stack(ids).contiguous())
    s1, i1 = ctx.flat_ip_topk(Qs, Xall, 100)
    ok_flat = float((i1 == ids).float().mean().item()) > 0.995 and bool(torch.allclose(s1, sc, rtol=1e-5, atol=2e-4))
    # re-rank: sharded + merged == single GPU
    codes_all = ctx.rq_encode(Xall, cbk)
    pq = ProductQuantization("rq", 4, 5, "l2", d, "kmeans", "grad")
    with torch.no_grad():
        pq.codebook.copy_(cbk.cpu())
    dec = pq.beam_search(Qs, 20)
    rr = ClusterReranker(Xall[s:e].contiguous(), ClusterIndex.from_codes(codes_all[s:e].contiguous(), 32, id_base=s, device_index=dev.index))
    sc, ids, nc = rr.rerank(Qs, dec, topk=100)
    full = ClusterIndex.from_codes(codes_all, 32, device_index=dev.index)
    s0_, i0_, n0_ = ctx.cluster_rerank(Qs, Xall, full.leaf_offsets, full.leaf_docids, full.lookup(dec), 100)
    ok_rr = float((i0_ == ids).float().mean().item()) > 0.995 and bool((n0_ == nc).all()) and bool(torch.allclose(s0_, sc, rtol=1e-5, atol=2e-4))
    flags = torch.tensor([int(ok_train), int(ok_flat), int(ok_rr)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    names = ["train", "flat", "rerank"]
    bad = [nm for nm, f in zip(names, flags.tolist()) if not f]
    return "ok" if not bad else "FAILED:" + ",".join(bad)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "cpu-baseline-child"])
    ap.add_argument("--sample-file", type=str, default=None)
    ap.add_argument("--mode", type=str, default="auto", choices=["auto", "exact", "tensor"])
    ap.add_argument("--docs", type=int, default=N_MARCO, help="rows per GPU (default: MSMARCO 8,841,823)")
    ap.add_argument("--flat-docs", type=int, default=N_MARCO, help="rows per GPU of the MSMARCO-shape flat search")
    ap.add_argument("--ref-sample", type=int, default=1 << 20)
    ap.add_argument("--rr-leaf", action="store_true", help="N > 1: also time the grouped re-rank on a leaf-partitioned index "
                    "(measured slower than row blocks at N = 2, profiles/r02_rerank_leaf_partition_n2.txt)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-nq", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the codes of the last timed step (or a seeded sample of them) to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to the default implementation (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.impl == "cpu-baseline-child":
        cpu_baseline_child(args)
        return
    if world != args.gpus:
        log(f"note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE")
    our_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
