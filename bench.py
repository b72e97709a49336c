#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json metric: queries/sec at recall@k).

Headline workload (BASELINE.json configs[1]): GpuIndexFlatL2, N=10M, d=128, nq=10k, k=100, synthetic fp32.
A "step" = one search() of all nq queries over the whole database.

  python bench.py --gpus 1 --steps K --warmup W            # this framework (tcgen05 Flat path)
  python bench.py --impl reference --gpus 1 --steps K ...   # reference CPU IndexFlatL2 (oracle/_ref)
  torchrun --nproc-per-node N bench.py --gpus N ...         # database sharded over N GPUs
                                                            # (IndexShards semantics, NCCL all-gather merge)
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's results to DIR

--steps sets the number of timed steps of every timed loop.  The inputs are seeded: with the same arguments
(and BENCH_* environment) every run searches the same data, so the files of --dump-outputs from two builds can
be compared array for array: DIR/flat_D.npy (float32 [nq, k] distances) and DIR/flat_I.npy (float64 [nq, k]
ids), and at one GPU ivfpq_{D,I}.npy and ivfpq_synthetic_{D,I}.npy of the IVFPQ workloads (36 MB in all at
the default sizes; larger results are cut to a fixed set of query rows, see dump_outputs).

One JSON line on stdout (rank 0).  `value` = QPS with inputs resident in HBM; `e2e` = QPS through
the public API with host (pinned) buffers, H2D/D2H inside the timed region; `roofline` = algorithmic
FLOPs of the step / device time inside the tcgen05 kernel, vs the measured bf16 GEMM peak;
`parity_check` = the step's result compared (outside the timed region) with an unsharded exact answer
and with the reference CPU library; `workloads.ivfpq` (N=1 only) = BASELINE configs[3] (IVFPQ N=100M)
with its own roofline (scan kernel, HBM), e2e, CPU IndexIVFPQ baseline on the CLONED index and
recall@1/10/100 for CPU and GPU; `workloads.ivfpq_synthetic` = the same on contrib/datasets.py's
SyntheticDataset distribution, where IVF/PQ recall is meaningful.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TOTAL = int(os.environ.get("BENCH_N", 10_000_000))
DIM = int(os.environ.get("BENCH_D", 128))
NQ = int(os.environ.get("BENCH_NQ", 10_000))
K = int(os.environ.get("BENCH_K", 100))
CHUNK = 1_000_000  # database is generated in seeded chunks so shards do not depend on world size

# one metric string for BOTH arms (the driver pairs the arms on metric, unit and direction)
METRIC = "queries/sec (GpuIndexFlatL2 exact k-NN, recall@k = 1)"
UNIT = "queries/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_BYTES_PER_WORKLOAD = 20 << 20  # three workloads stay under 64 MB


def dump_outputs(dirname, name, D, I):
    """one timed step's search result as DIR/<name>_D.npy (float32) and DIR/<name>_I.npy (float64: ids < 2^53 are
    exact).  A result larger than DUMP_BYTES_PER_WORKLOAD is cut to evenly spaced query rows, whose indices go to
    DIR/<name>_rows.npy."""
    if not dirname:
        return
    os.makedirs(dirname, exist_ok=True)
    D, I = D.cpu().numpy(), I.cpu().numpy()
    row_bytes = D.shape[1] * 12
    if D.shape[0] * row_bytes > DUMP_BYTES_PER_WORKLOAD:
        rows = np.linspace(0, D.shape[0] - 1, DUMP_BYTES_PER_WORKLOAD // row_bytes).astype(np.int64)
        D, I = D[rows], I[rows]
        np.save(os.path.join(dirname, name + "_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(dirname, name + "_D.npy"), np.asarray(D, dtype=np.float32))
    np.save(os.path.join(dirname, name + "_I.npy"), np.asarray(I, dtype=np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return j, "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe).  nvidia-smi
    needs ~0.5 s to produce its first line, so it is started before the warm-up; samples are time-stamped
    on arrival and only those inside [mark_begin, mark_end] (the timed region) are used -- widened to the
    warm-up steps of the same workload if the timed region is shorter than one sampling period."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []  # (arrival time, text)
        self.t_load = self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark_load(self):
        self.t_load = time.time()

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()

        def parse(t0, t1):
            sm, smax, reasons, power = [], [], set(), []
            for ts, ln in self.lines:
                if t0 is not None and not (t0 <= ts <= t1 + 0.06):
                    continue
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                    power.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return sm, smax, reasons, power

        window = "timed region"
        sm, smax, reasons, power = parse(self.t_begin, self.t_end or time.time())
        if len(sm) < 2 and self.t_load is not None:
            window = "warm-up + timed region (same workload; the timed region is shorter than two sampling periods)"
            sm, smax, reasons, power = parse(self.t_load, self.t_end or time.time())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "lines_seen": len(self.lines)}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power)), "window": window}


def gen_rows(torch, device, r0, r1, d, n_total=None, seed0=1234):
    """rows [r0, r1) of the synthetic database: uniform [0,1) fp32, chunk c seeded with seed0 + c"""
    n_total = N_TOTAL if n_total is None else n_total
    out = torch.empty((r1 - r0, d), dtype=torch.float32, device=device)
    c = r0 // CHUNK
    while c * CHUNK < r1:
        g = torch.Generator(device=device)
        g.manual_seed(seed0 + c)
        c0, c1 = c * CHUNK, min((c + 1) * CHUNK, n_total)
        chunk = torch.rand((c1 - c0, d), dtype=torch.float32, device=device, generator=g)
        a, b = max(r0, c0), min(r1, c1)
        out[a - r0 : b - r0] = chunk[a - c0 : b - c0]
        del chunk
        c += 1
    return out


def gen_queries(torch, device, nq, d, seed=1235):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return torch.rand((nq, d), dtype=torch.float32, device=device, generator=g)


def host_threads():
    """CPUs this process may actually use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------------
# reference CPU IndexFlatL2 (oracle/_ref): thread sweep + bounded sample
# ------------------------------------------------------------------------------------------------
def _blas_sample_queries(nq, d):
    # the reference switches from its per-query SIMD loop to the BLAS-blocked path at nq*d >= 128000
    # (faiss/utils/distances.cpp:567,600), i.e. nq >= 1000 at d=128 -- anything smaller would time a
    # different (much slower) code path than the nq=10k workload takes
    return int(min(nq, max(1000, 128000 // d + 1)))


def ref_thread_sweep(ref, xb, xq, k, cores):
    """Best thread count for the reference's BLAS + OpenMP path on this host.  This image's OpenBLAS is
    a pthreads build whose pool oversubscribes badly next to OpenMP when handed every CPU of a large
    host (round 1: 96 threads were 12x slower than 16), so the count is measured, not assumed."""
    cand = sorted({t for t in (2, 4, 8, 12, 16, 24, 32, 48, 64, cores) if 1 <= t <= cores})
    rows = min(xb.shape[0], 100_000)
    idx = ref.IndexFlat(xb.shape[1], 1)
    idx.add(xb[:rows])
    ns = _blas_sample_queries(xq.shape[0], xb.shape[1])
    res = {}
    for t in cand:
        ref.set_omp_threads(t)
        ref.set_blas_threads(t)
        idx.search(xq[:ns], k)  # warm the pool at this size
        t0 = time.time()
        idx.search(xq[:ns], k)
        res[t] = time.time() - t0
    best = min(res, key=res.get)
    ref.set_omp_threads(best)
    ref.set_blas_threads(best)
    return best, {str(t): round(v, 4) for t, v in res.items()}


def cpu_flat_reference(xb_host, xq_host, k, step_budget_s, steps, warmup, total_budget_s):
    """Times faiss::IndexFlatL2 (oracle/_ref) on a bounded sample: the first ns queries (BLAS path) against a
    leading slice of the rows sized so one step fits `step_budget_s`.  Returns (qps_full, info): qps_full is
    the sample's rate scaled to the full N (exhaustive search is linear in the rows scanned);
    info['ms_per_step'] is the MEASURED step time of the sample."""
    from oracle import ref

    cores = host_threads()
    nfull, d = xb_host.shape
    best_t, sweep = ref_thread_sweep(ref, xb_host, xq_host, k, cores)
    ns = _blas_sample_queries(xq_host.shape[0], d)
    # probe the rate at the chosen thread count, then size the row slice
    probe_rows = min(nfull, 250_000)
    pidx = ref.IndexFlat(d, 1)
    pidx.add(xb_host[:probe_rows])
    pidx.search(xq_host[:ns], k)
    t0 = time.time()
    pidx.search(xq_host[:ns], k)
    t_probe = time.time() - t0
    del pidx
    nrows = int(min(nfull, max(probe_rows, probe_rows * step_budget_s / max(t_probe, 1e-6))))
    nrows = max(100_000, nrows // 100_000 * 100_000)
    nrows = min(nrows, nfull)
    idx = ref.IndexFlat(d, 1)
    idx.add(xb_host[:nrows])
    ts = []
    t_begin = time.time()
    D = I = None
    for i in range(warmup + steps):
        t0 = time.time()
        D, I = idx.search(xq_host[:ns], k)
        dt = time.time() - t0
        if i >= warmup:
            ts.append(dt)
        if time.time() - t_begin > total_budget_s and ts:
            break
    t_meas = float(np.mean(ts))
    scale = nfull / float(nrows)
    qps = ns / (t_meas * scale)
    info = {"kind": "reference", "cores": best_t, "ms_per_step": t_meas * 1e3, "nq_sample": ns, "rows_sample": nrows,
            "sample_scale": scale, "thread_sweep_s": sweep, "host_cpus": cores, "cpu_model": cpu_model(),
            "timed_steps": len(ts),
            "sample": "faiss::IndexFlatL2 (oracle/_ref = unmodified reference, %s, OpenBLAS 0.3.15 pthreads), %d threads (best of sweep %s over "
                      "%d usable CPUs, %s): first %d of %d queries (smallest batch on the reference's BLAS path), k=%d, against the first %d of "
                      "N=%d rows: %.3f s measured per step (%d timed); value = sample rate / %.2f (exhaustive search is linear in the rows scanned)" % (
                          ref.compile_options().strip(), best_t, json.dumps(sweep), cores, cpu_model(), ns, xq_host.shape[0], k, nrows, nfull,
                          t_meas, len(ts), scale)}
    return qps, info, (D, I, ns, nrows)


def cpu_flat_port(xb_host, xq_host, k):
    from oracle import oracle_np as o

    nb = min(xb_host.shape[0], 200_000)
    ns = min(xq_host.shape[0], 64)
    t0 = time.time()
    o.knn_flat(xq_host[:ns], xb_host[:nb], k, 1)
    t = time.time() - t0
    qps = ns / (t * xb_host.shape[0] / nb)
    return qps, {"kind": "port", "cores": 1, "ms_per_step": t * 1e3, "nq_sample": ns, "rows_sample": nb,
                 "sample_scale": xb_host.shape[0] / nb,
                 "sample": "numpy oracle port, %d queries x %d rows, scaled linearly to N=%d" % (ns, nb, xb_host.shape[0])}


def flat_config(world):
    return {"workload": "GpuIndexFlatL2 N=%d d=%d nq=%d k=%d (BASELINE configs[1])" % (N_TOTAL, DIM, NQ, K),
            "N": N_TOTAL, "d": DIM, "nq": NQ, "k": K,
            "parallelism": "IndexShards x%d (contiguous row shards, all-gather top-k merge)" % world if world > 1 else "single GPU",
            "l2_note": "inputs larger than L2 (database %.1f GB fp32 + %.1f GB fp16 copy per step vs 126 MB L2)" % (
                N_TOTAL * DIM * 4 / 1e9 / world, N_TOTAL * DIM * 2 / 1e9 / world)}


def reference_arm(args, torch):
    """--impl reference: the reference's own CPU implementation of the path on the host cores."""
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    xb = gen_rows(torch, dev, 0, N_TOTAL, DIM).cpu().numpy()
    xq = gen_queries(torch, dev, NQ, DIM).cpu().numpy()
    if dev != "cpu":
        torch.cuda.empty_cache()
    from oracle import ref

    # the whole --steps/--warmup run must end within a few minutes: ~150 s of search split over the steps
    total = float(os.environ.get("BENCH_REF_BUDGET_S", 150.0))
    step_budget = max(1.0, total / (steps + warmup))
    if ref.available():
        qps, info, _ = cpu_flat_reference(xb, xq, K, step_budget, steps, warmup, total * 1.5)
    else:
        qps, info = cpu_flat_port(xb, xq, K)
    out = {"impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT,
           "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": info["ms_per_step"],
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": flat_config(1),
           "sample_scale": info.get("sample_scale"),
           "note": "ms_per_step is the measured time of one step = the bounded sample described in cpu_baseline.sample; value is that sample's "
                   "query rate scaled to the full N rows (factor sample_scale)",
           "cpu_baseline": {"value": qps, "unit": UNIT, "cores": info["cores"], "kind": info["kind"], "sample": info["sample"],
                            "thread_sweep_s": info.get("thread_sweep_s"), "host_cpus": info.get("host_cpus"), "cpu_model": info.get("cpu_model")},
           "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------
# parity check of the Flat step (outside the timed region)
# ------------------------------------------------------------------------------------------------
def flat_parity_check(torch, fb, res, device, local_rank, world, index, D, I, xq, nchk=256):
    """rank 0: (a) at world > 1 the merged sharded result of the first nchk queries must equal, bit for
    bit, an UNSHARDED exact index over the same rows (model: faiss/gpu/test/test_multi_gpu.py:23-43);
    (b) the same queries vs the reference CPU IndexFlatL2 over all N rows, with the reference's own
    comparison semantics (compareLists, faiss/gpu/test/TestUtils.cpp:158-226; distances <= 1e-4 rel)."""
    from oracle import oracle_np as o

    out = {"queries": nchk, "ok": True}
    Dc, Ic = D[:nchk].cpu().numpy(), I[:nchk].cpu().numpy()
    xqc = xq[:nchk].contiguous()
    xb_full = None
    if world > 1:
        xb_full = gen_rows(torch, device, 0, N_TOTAL, DIM)
        full = fb.GpuIndexFlatL2(res, DIM, device=local_rank, use_tensor_cores=False)
        full.add(xb_full)
        uD, uI = full.search(xqc, K)
        uD, uI = uD.cpu().numpy(), uI.cpu().numpy()
        del full
        same_i = bool(np.array_equal(uI, Ic))
        same_d = bool(np.array_equal(uD, Dc))
        out["vs_unsharded_exact"] = {"ids_equal": same_i, "distances_equal": same_d,
                                     "mismatching_ids": int((uI != Ic).sum())}
        out["ok"] = out["ok"] and same_i and same_d
    try:
        from oracle import ref

        if ref.available():
            if xb_full is None:
                xb_host = index.copyTo() if world == 1 else None
            else:
                xb_host = xb_full.cpu().numpy()
            del xb_full
            ref.set_omp_threads(min(host_threads(), 32))
            t0 = time.time()
            rD, rI = ref.knn(xqc.cpu().numpy(), xb_host, K, 1)
            dt = time.time() - t0
            try:
                o.compare_lists(rD, rI, Dc, Ic, eps=1e-4, pct_max_diff1=0.01, pct_max_diffN=0.005)
                cl = True
                msg = ""
            except AssertionError as e:
                cl, msg = False, str(e)[:200]
            rel = float(np.max(np.abs(rD - Dc) / np.maximum(np.abs(rD), 1e-20)))
            out["vs_reference_cpu"] = {"compare_lists_ok": cl, "ids_equal_frac": float((rI == Ic).mean()),
                                       "max_rel_distance_err": rel, "tolerance": 1e-4, "cpu_s": round(dt, 2), "msg": msg}
            out["ok"] = out["ok"] and cl and rel <= 1e-4
        else:
            out["vs_reference_cpu"] = "oracle/_ref not built"
    except Exception as e:  # the checker failing to run is reported, not hidden
        out["vs_reference_cpu"] = "failed: %s" % str(e)[:200]
        out["ok"] = False
    return out


# ------------------------------------------------------------------------------------------------
# IVFPQ workloads (N = 1 GPU)
# ------------------------------------------------------------------------------------------------
def synthetic_dataset(d, nt, nb, nq, seed=1338):
    """contrib/datasets.py:84-105 SyntheticDataset restated (numpy RandomState(seed), 10-d latent, random
    projection, per-dimension frequency, sin warp).  Returns (xt, xb, xq) float32."""
    d1 = 10
    n = nb + nt + nq
    rs = np.random.RandomState(seed)
    x = rs.normal(size=(n, d1))
    x = np.dot(x, rs.rand(d1, d))
    x = x * (rs.rand(d) * 4 + 0.1)
    x = np.sin(x).astype("float32")
    return x[:nt], x[nt : nt + nb], x[nt + nb :]


def _recalls(I, gt):
    """recall@r = fraction of queries whose true nearest neighbour is among the first r results (the
    benchs/ convention, 1-recall@r), plus the intersection measure |I_k & gt_k| / k"""
    I = np.asarray(I)
    gt = np.asarray(gt)
    k = I.shape[1]
    out = {}
    for r in (1, 10, 100):
        if r <= k:
            out["1-recall@%d" % r] = float((I[:, :r] == gt[:, :1]).any(axis=1).mean())
    out["intersection@%d" % k] = float(np.mean([len(set(a.tolist()) & set(b.tolist())) for a, b in zip(I, gt)]) / k)
    return out


def ivfpq_workload(torch, fb, res, device, name, N, d, nlist, M, nprobe, nq, k, steps, warmup, data, n_gt, cpu_queries, dump_dir=None):
    """Build a GpuIndexIVFPQ, time search (device-resident and e2e), clone it to the reference CPU
    IndexIVFPQ (same centroids / PQ / list bytes), time that on the host cores, report recall for both.
    data = ("uniform", None) -> seeded uniform chunks generated on the device;
           ("arrays", (xt, xb, xq)) -> host arrays (SyntheticDataset)."""
    dev = device
    kind, arrays = data
    index = fb.GpuIndexIVFPQ(res, d, nlist, M, 8, fb.METRIC_L2, device=dev.index or 0)
    t0 = time.time()
    if kind == "uniform":
        g = torch.Generator(device=dev)
        g.manual_seed(4321)
        xt = torch.rand((min(1 << 20, N), d), dtype=torch.float32, device=dev, generator=g)
        xq = gen_queries(torch, dev, nq, d)
    else:
        xt = torch.from_numpy(arrays[0]).to(dev)
        xq = torch.from_numpy(arrays[2]).to(dev)
    index.train(xt)
    del xt
    torch.cuda.synchronize()
    t_train = time.time() - t0
    # add in chunks; exact ground truth of the first n_gt queries is folded in chunk by chunk with the
    # exact fp32 Flat kernel (tier-2 seam) -- the database never has to exist in one piece
    t0 = time.time()
    index.reserveMemory(N + N // 8)
    n_gt = min(n_gt, nq)
    xq_gt = xq[:n_gt].contiguous()
    bestD = torch.full((n_gt, k), float("inf"), device=dev)
    bestI = torch.full((n_gt, k), -1, dtype=torch.int64, device=dev)
    t_gt = 0.0
    for c0 in range(0, N, CHUNK):
        c1 = min(N, c0 + CHUNK)
        if kind == "uniform":
            xb = gen_rows(torch, dev, c0, c1, d, n_total=N, seed0=7000)
        else:
            xb = torch.from_numpy(arrays[1][c0:c1]).to(dev)
        index.add(xb)
        torch.cuda.synchronize()
        tg = time.time()
        cD, cI = fb.flat_search_exact(res, xb, xq_gt, k, device=dev.index or 0)
        allD = torch.cat([bestD, cD], dim=1)
        allI = torch.cat([bestI, cI + c0], dim=1)
        o_ = torch.argsort(allD, dim=1, stable=True)[:, :k]
        bestD, bestI = torch.gather(allD, 1, o_), torch.gather(allI, 1, o_)
        torch.cuda.synchronize()
        t_gt += time.time() - tg
        del xb
    t_add = time.time() - t0 - t_gt
    gt = bestI.cpu().numpy()
    log("[%s] trained %.1f s, added %d vectors in %.1f s (%.1f M/s), ground truth %.1f s" % (name, t_train, N, t_add, N / t_add / 1e6, t_gt))
    index.nprobe = nprobe
    lens = np.array([index.getListLength(l) for l in range(nlist)], dtype=np.int64)
    xq_pin = torch.empty((nq, d), dtype=torch.float32, pin_memory=True)
    xq_pin.copy_(xq)
    D_pin = torch.empty((nq, k), dtype=torch.float32, pin_memory=True)
    I_pin = torch.empty((nq, k), dtype=torch.int64, pin_memory=True)

    for _ in range(max(3, warmup)):
        D, I = index.search(xq, k)
    torch.cuda.synchronize()
    # algorithmic bytes of one step = sum over (query, probe) of the probed list's length x M
    cent = torch.from_numpy(index.getCoarseCentroids()).to(dev)
    _, probes = fb.flat_search_exact(res, cent, xq, nprobe, device=dev.index or 0)
    scanned = int(lens[probes.cpu().numpy()].sum())
    alg_bytes = scanned * M

    stream = torch.cuda.current_stream(dev)
    fb.lib.faiss_b200_kernel_timing(1)
    l0 = fb.lib.faiss_b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        D, I = index.search(xq, k)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    launches = fb.lib.faiss_b200_launch_count() - l0
    kms, kn = ctypes.c_double(), ctypes.c_int()
    fb.lib.faiss_b200_kernel_timing_collect(b"ivfpq_scan", ctypes.byref(kms), ctypes.byref(kn))
    fb.lib.faiss_b200_kernel_timing(0)

    for _ in range(2):
        index.search(xq_pin.numpy(), k, D=D_pin.numpy(), I=I_pin.numpy())
    t0 = time.time()
    for _ in range(steps):
        index.search(xq_pin.numpy(), k, D=D_pin.numpy(), I=I_pin.numpy())
    e2e_ms = (time.time() - t0) * 1e3 / steps
    dump_outputs(dump_dir, name, D, I)

    gpu_I = I[:n_gt].cpu().numpy()
    gpu_D = D[:n_gt].cpu().numpy()
    pk, src = peaks()
    roof = {"bound": "hbm", "unit": "GB/s", "peak": float(pk["hbm_gbs"]), "peak_source": src + " copy bandwidth (MEASURED_PEAKS.json)",
            "traffic": None, "kernel": "ivfpq_scan_interleaved_kernel", "algorithmic_bytes_per_step": alg_bytes, "vectors_scanned_per_step": scanned}
    tpath = os.path.join(ROOT, "profiles", "ivfpq_scan_traffic.json")
    if name == "ivfpq" and N == 100_000_000 and os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            roof["traffic"] = tj["dram_bytes_per_launch"]
            roof["traffic_source"] = tj["source"]
        except Exception:
            pass
    if kn.value:
        kms_step = kms.value / steps
        roof.update({"achieved": alg_bytes / (kms_step * 1e-3) / 1e9, "kernel_ms_per_step": kms_step, "kernel_share_of_step": kms_step / ms,
                     "launches_per_step": kn.value // steps})
        roof["frac"] = roof["achieved"] / roof["peak"]
    out = {"metric": "queries/sec (GpuIndexIVFPQ)", "value": nq / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
           "dtype": "u8 codes, f32 LUT + f32 accumulate",
           "config": {"workload": "GpuIndexIVFPQ N=%d d=%d nlist=%d M=%d nbits=8 nprobe=%d nq=%d k=%d" % (N, d, nlist, M, nprobe, nq, k),
                      "data": "uniform [0,1) fp32 (seeded chunks)" if kind == "uniform" else "SyntheticDataset (contrib/datasets.py:84-105, seed 1338)",
                      "list_len_mean": float(lens.mean()), "list_len_max": int(lens.max()), "train_s": round(t_train, 2), "add_s": round(t_add, 2),
                      "add_vec_per_s": N / t_add, "l2_note": "codes scanned per step %.1f GB vs 126 MB L2" % (alg_bytes / 1e9)},
           "e2e": {"value": nq / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * 12},
           "gpu_launches": int(launches), "roofline": roof,
           "recall": {"queries": n_gt, "ground_truth": "exact fp32 k-NN (exact SIMT Flat kernel, chunked over the database)", "gpu": _recalls(gpu_I, gt)}}

    # ---- CPU arm on the CLONED index (BASELINE.md section 3.4): same centroids, PQ codebooks and list bytes
    try:
        from oracle import ref

        if not ref.available():
            raise RuntimeError("oracle/_ref not built")
        t0 = time.time()
        cpu = ref.IndexIVFPQ(d, nlist, M, 8, 1)
        cpu.set_centroids(index.getCoarseCentroids())
        cpu.set_pq_centroids(index.getPQCentroids())
        cpu.set_is_trained(True)
        for l in range(nlist):
            if lens[l]:
                cpu.add_entries(l, index.getListIndices(l), index.getListVectorData(l))
        cpu.set_precomputed_table(0)  # 0 = the reference's auto rule (IndexIVFPQ::precompute_table)
        cpu.set_nprobe(nprobe)
        t_clone = time.time() - t0
        assert cpu.ntotal == index.ntotal, (cpu.ntotal, index.ntotal)
        cores = host_threads()
        ns = min(nq, cpu_queries)
        xq_host = xq_pin.numpy()
        best = None
        sweep = {}
        for t in sorted({t for t in (8, 16, 32, 64, cores) if t <= cores}):
            ref.set_omp_threads(t)
            ref.set_blas_threads(min(t, 16))
            nprobe_q = min(ns, 200)
            cpu.search(xq_host[:nprobe_q], k)
            t1 = time.time()
            cpu.search(xq_host[:nprobe_q], k)
            sweep[str(t)] = round(time.time() - t1, 4)
            if best is None or sweep[str(t)] < sweep[str(best)]:
                best = t
        ref.set_omp_threads(best)
        ref.set_blas_threads(min(best, 16))
        ts = []
        for _ in range(3):
            t1 = time.time()
            cD, cI = cpu.search(xq_host[:ns], k)
            ts.append(time.time() - t1)
        t_cpu = float(np.median(ts))
        out["cpu_baseline"] = {"value": ns / t_cpu, "unit": UNIT, "cores": best, "kind": "reference",
                               "sample": "faiss::IndexIVFPQ (oracle/_ref) cloned from the GPU index (identical centroids, PQ, list bytes; "
                                         "use_precomputed_table=%d by the reference's auto rule), nprobe=%d, first %d of %d queries, median of 3 searches "
                                         "= %.3f s, %d OpenMP threads (sweep %s, %d usable CPUs, %s); clone %.1f s" % (
                                             cpu.use_precomputed_table, nprobe, ns, nq, t_cpu, best, json.dumps(sweep), cores, cpu_model(), t_clone)}
        ng = min(n_gt, ns)
        out["recall"]["cpu"] = _recalls(cI[:ng], gt[:ng])
        out["recall"]["gpu_on_cpu_queries"] = _recalls(gpu_I[:ng], gt[:ng])
        # parity on the sample the CPU just answered: reference comparison semantics + distance tolerance
        from oracle import oracle_np as o

        par = {"queries": ng}
        try:
            o.compare_lists(cD[:ng], cI[:ng], gpu_D[:ng], gpu_I[:ng], eps=2e-4, pct_max_diff1=0.02, pct_max_diffN=0.01)
            par["compare_lists_ok"] = True
        except AssertionError as e:
            par["compare_lists_ok"] = False
            par["msg"] = str(e)[:200]
        par["ids_equal_frac"] = float((cI[:ng] == gpu_I[:ng]).mean())
        out["parity_check"] = par
        del cpu
    except Exception as e:
        out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": host_threads(), "kind": "reference", "sample": "failed: %s" % str(e)[:300]}
    del index
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ivfpq", action="store_true", help="skip the IVFPQ workloads (configs[3] + SyntheticDataset)")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last timed step's results to DIR as .npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    steps, warmup = args.steps, max(0, args.warmup)

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    import torch

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, torch)
        return

    # ------------------------------------------------------------------ this framework
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback exists in faiss_b200)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        # keep stdout to the one JSON line: NCCL prints its version banner to stdout when the first
        # communicator is created (any NCCL_DEBUG level >= VERSION), so that happens with fd 1 -> fd 2
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.all_reduce(torch.zeros(1, device=device))
            torch.cuda.synchronize()
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    import faiss_b200 as fb
    from faiss_b200.distributed import shard_bounds

    res = fb.StandardGpuResources()
    if world > 1:
        # the NCCL communicator of the search path is owned by the library's resources object; torch.distributed
        # only hands the 128-byte id to the other ranks (plumbing) and provides the barrier around the timed region
        ids = [fb.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0, device=device)
        res.ncclInitRank(local_rank, world, rank, ids[0])
    # order the library's work on torch's current stream so torch CUDA events bracket it
    stream = torch.cuda.current_stream(device)
    res.setDefaultStream(local_rank, stream.cuda_stream)

    r0, r1 = shard_bounds(N_TOTAL, rank, world)
    t0 = time.time()
    xb = gen_rows(torch, device, r0, r1, DIM)
    index = fb.GpuIndexFlatL2(res, DIM, device=local_rank)
    index.add(xb)
    del xb
    xq = gen_queries(torch, device, NQ, DIM)
    xq_pin = torch.empty((NQ, DIM), dtype=torch.float32, pin_memory=True)
    xq_pin.copy_(xq)
    D_pin = torch.empty((NQ, K), dtype=torch.float32, pin_memory=True)
    I_pin = torch.empty((NQ, K), dtype=torch.int64, pin_memory=True)
    torch.cuda.synchronize()
    log("[rank %d] shard rows [%d,%d) built in %.1f s" % (rank, r0, r1, time.time() - t0))

    # world > 1: IndexShards with one shard per rank behind the C ABI (faiss_DistributedIndexShards): pooled
    # thresholds per round, ONE grouped ncclAllGather of the per-shard [nq,k] blocks, device merge
    searcher = fb.DistributedIndexShards(res, index, successive_ids=True) if world > 1 else index
    assert searcher.ntotal == N_TOTAL

    def step_device():
        return searcher.search(xq, K)

    def step_e2e():
        searcher.search(xq_pin.numpy(), K, D=D_pin.numpy(), I=I_pin.numpy())  # H2D + search + D2H inside

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.7)  # nvidia-smi start-up; outside every timed region
    sampler.mark_load()
    for _ in range(max(warmup, 3)):
        step_device()
    barrier()

    # ---- timed region: device-resident inputs
    fb.lib.faiss_b200_kernel_timing(1)
    l0 = fb.lib.faiss_b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    e0.record(stream)
    for _ in range(steps):
        D, I = step_device()
    e1.record(stream)
    barrier()
    sampler.mark_end()
    ms = e0.elapsed_time(e1) / steps
    launches = fb.lib.faiss_b200_launch_count() - l0
    tc_ms = ctypes.c_double()
    tc_n = ctypes.c_int()
    fb.lib.faiss_b200_kernel_timing_collect(b"flat_tc", ctypes.byref(tc_ms), ctypes.byref(tc_n))
    ex_ms, mg_ms, ex_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
    fb.lib.faiss_b200_kernel_timing_collect(b"shards_exchange", ctypes.byref(ex_ms), ctypes.byref(ex_n))
    fb.lib.faiss_b200_kernel_timing_collect(b"shards_merge", ctypes.byref(mg_ms), ctypes.byref(ex_n))
    breakdown = {}
    for nm in (b"tc_select", b"tc_pool", b"tc_rerank"):
        v, c = ctypes.c_double(), ctypes.c_int()
        fb.lib.faiss_b200_kernel_timing_collect(nm, ctypes.byref(v), ctypes.byref(c))
        breakdown[nm.decode() + "_ms"] = v.value / steps
        breakdown[nm.decode() + "_launches"] = c.value // steps
    fb.lib.faiss_b200_kernel_timing(0)
    clocks = sampler.stop() if rank == 0 else None
    info = index.lastSearchInfo()

    # ---- e2e: host buffers through the public API
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.time()
    for _ in range(steps):
        step_e2e()
    barrier()
    e2e_ms = (time.time() - t0) * 1e3 / steps
    if rank == 0:
        dump_outputs(args.dump_outputs, "flat", D, I)

    if dist is not None:
        t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])

    rc = 0
    if rank == 0:
        pk, pk_src = peaks()
        flops_step = 2.0 * NQ * (r1 - r0) * DIM  # this rank's shard
        tc_ms_step = tc_ms.value / steps if tc_n.value else None
        peak_tf = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops")))
        roof = {"bound": "tensor", "unit": "TFLOP/s", "peak": peak_tf, "traffic": None,
                "peak_source": "%s bf16 GEMM peak (sustained; kernel timed inside a multi-step loop), MEASURED_PEAKS.json" % pk_src,
                "kernel": "flat_tc_kernel (tcgen05 fp16 scoring + fused top-k filter), %d launches/step" % (tc_n.value // steps if tc_n.value else 0),
                "algorithmic_flops_per_step": flops_step}
        # DRAM bytes per launch of this kernel, from the committed `ncu --set full` capture of this same
        # workload (profiles/flat_tc_traffic.json, written by scripts/ncu_traffic.py); single GPU only
        tpath = os.path.join(ROOT, "profiles", "flat_tc_traffic.json")
        if world == 1 and N_TOTAL == 10_000_000 and os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                roof["traffic"] = tj["dram_bytes_per_launch"]
                roof["traffic_source"] = tj["source"]
            except Exception:
                pass
        if tc_ms_step:
            roof["achieved"] = flops_step / (tc_ms_step * 1e-3) / 1e12
            roof["frac"] = roof["achieved"] / peak_tf
            roof["kernel_ms_per_step"] = tc_ms_step
            roof["kernel_share_of_step"] = tc_ms_step / ms
        else:
            roof["achieved"] = None
            roof["frac"] = None
        out = {"metric": METRIC, "value": NQ / (ms * 1e-3), "unit": UNIT,
               "n_gpus": world, "steps": steps, "warmup": max(warmup, 3), "ms_per_step": ms, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f16 mma (fp32 accumulate) + f32 exact re-rank", "data": "synthetic",
               "config": flat_config(world), "clocks": clocks,
               "e2e": {"value": NQ / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                       "h2d_bytes_per_step": NQ * DIM * 4, "d2h_bytes_per_step": NQ * K * 12},
               "gpu_launches": int(launches), "roofline": roof,
               "search_info": info,
               "step_breakdown_ms": dict(breakdown, flat_tc_ms=(tc_ms.value / steps if tc_n.value else None),
                                         note="rank 0, CUDA events around each launch (threshold select, cross-rank pooling, exact re-rank)")}
        if world > 1:
            out["collective_ms"] = ex_ms.value / steps  # rank 0's all-gather (includes waiting for the slowest rank)
            out["merge_ms"] = mg_ms.value / steps
        # ---- parity of the timed step's result (outside the timed region)
        if not args.no_parity:
            try:
                out["parity_check"] = flat_parity_check(torch, fb, res, device, local_rank, world, index, D, I, xq)
            except Exception as e:
                out["parity_check"] = {"ok": False, "error": str(e)[:300]}
            if not out["parity_check"].get("ok", False):
                rc = 3
        # ---- CPU baseline (reference CPU path on this box's host cores), N=1 only
        if world == 1 and not args.no_cpu_baseline:
            try:
                from oracle import ref

                xb_host = index.copyTo()
                if ref.available():
                    qps, cinfo, _ = cpu_flat_reference(xb_host, xq_pin.numpy(), K, step_budget_s=6.0, steps=2, warmup=1, total_budget_s=30.0)
                else:
                    qps, cinfo = cpu_flat_port(xb_host, xq_pin.numpy(), K)
                del xb_host
                out["cpu_baseline"] = {"value": qps, "unit": UNIT, "cores": cinfo["cores"], "kind": cinfo["kind"], "sample": cinfo["sample"],
                                       "sample_ms_per_step": cinfo["ms_per_step"], "sample_scale": cinfo.get("sample_scale"),
                                       "thread_sweep_s": cinfo.get("thread_sweep_s")}
            except Exception as e:
                out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": host_threads(), "kind": "reference", "sample": "failed: %s" % str(e)[:200]}
        # ---- IVFPQ workloads (BASELINE configs[3] + SyntheticDataset), single GPU
        if world == 1 and not args.no_ivfpq:
            del index
            torch.cuda.empty_cache()
            wl = {}
            try:
                n_pq = int(os.environ.get("BENCH_IVFPQ_N", 100_000_000))
                wl["ivfpq"] = ivfpq_workload(torch, fb, res, device, "ivfpq", n_pq, 128, 4096, 32, 32, NQ, K, steps, warmup,
                                             ("uniform", None), n_gt=1000, cpu_queries=1000, dump_dir=args.dump_outputs)
            except Exception as e:
                wl["ivfpq"] = {"error": str(e)[:300]}
            try:
                n_syn = int(os.environ.get("BENCH_SYNTH_N", 2_000_000))
                xt, xbs, xqs = synthetic_dataset(128, 200_000, n_syn, NQ)
                wl["ivfpq_synthetic"] = ivfpq_workload(torch, fb, res, device, "ivfpq_synthetic", n_syn, 128, 1024, 32, 32, NQ, K, steps, warmup,
                                                       ("arrays", (xt, xbs, xqs)), n_gt=1000, cpu_queries=1000,
                                                       dump_dir=args.dump_outputs)
            except Exception as e:
                wl["ivfpq_synthetic"] = {"error": str(e)[:300]}
            out["workloads"] = wl
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


if __name__ == "__main__":
    main()
