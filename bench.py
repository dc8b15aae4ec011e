#!/usr/bin/env python
"""bench.py -- one AM() forward step of the Eagle genome-scan hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic data set of the BASELINE.json shape:
    decode (ASCII -> int8)  ->  transpose (Mt)  ->  M.Mt (int8 tcgen05)  [-> all-reduce(int32) when N>1]
    -> finalize  ->  scan pre-products (int8 digit slices)  ->  a / var(a) scan (int8 digit slices)  ->  tsq argmax
`value` = markers/s of the whole job with the ASCII image, S, V and a_hat already resident in HBM;
`e2e`   = the same through the C ABI with HOST (pinned) buffers, H2D/D2H inside the timed region.
Markers are sharded over the N ranks (strong scaling: the data set is fixed, L/N markers per GPU).
`forward_search` (N=1, after the timed region): BASELINE config 3 as it is worded -- the full multi-locus AM() forward
search (<= 10 QTL, 5 planted) through eagleeverything_b200/am.py; --no-search skips it, --search-host adds the route with
every n x n matrix crossing the host-level ABI.
--dump-outputs DIR writes what the last timed step computed (a, var(a), the pick, rows of K) as float64 .npy files: the
inputs are seeded, so two builds run with the same arguments can be compared output for output.

--impl reference times the CPU restatement of the reference path (numpy/OpenBLAS, all host threads)
on a bounded sample of the same workload; it is the only leg that imports oracle/.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "c2": dict(n=2000, L=500000, name="config 2: synthetic n=2,000 x L=500,000, single trait, one forward step"),
    "c3": dict(n=10000, L=1000000, name="config 3 shape: synthetic n=10,000 x L=1,000,000, one forward step"),
    # multi-GPU shapes (marker-sharded; they do not fit one GPU next to their n x n workspaces)
    "c5": dict(n=20000, L=2000000, name="config 5 shape: synthetic n=20,000 x L=2,000,000, one forward step"),
    "c4": dict(n=50000, L=600000, name="config 4 shape: synthetic n=50,000 x L=600,000, one forward step"),
}
METRIC = "markers/s"
GENO_SEED = 20261018


def jprint(obj):
    print(json.dumps(obj), flush=True)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), bf16_tflops=d.get("bf16_tflops", 1590.0),
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", 1400.0), source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


# ====================================================================== CPU arm (reference restatement)
REF_SAMPLE_MARKERS = 4096     # fixed: independent of --steps, so every run of either arm times the same sample


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def bench_config(w, n, L, world):
    """The `config` object, identical in both arms (the driver compares them key by key)."""
    return {"workload": w["name"], "n": n, "L": L, "n_gpus": world}


class CpuReference:
    """The reference's CPU path for one forward step, timed on a bounded marker sample at full n.

    What runs is the C restatement's control flow (oracle/eagle_oracle.c: the in-memory branches of
    calculateMMt_rcpp.cpp:84-95 and calculate_a_and_vara_rcpp.cpp:76-112 -- ReadBlock's getline decode of M.ascii and
    Mt.ascii from real files, the products, the OpenMP row-dot loop) with its dense products routed to the OpenBLAS
    that numpy bundles (the reference runs them in Eigen's GEBP kernel; the restatement's plain loops are 10x slower
    than either).  Threads are set explicitly to every host core (torchrun exports OMP_NUM_THREADS=1).
    Stages linear in the marker count (decode of both files, M.Mt, Mt*v, Mt*W, row dots) are scaled by L / sample;
    the two n^3 pre-products and S*a are counted once per step, as measured (calculate_a_and_vara_rcpp.cpp:90,97-98)."""

    def __init__(self, n, L, Ls=REF_SAMPLE_MARKERS):
        import tempfile

        import numpy as np

        from eagleeverything_b200 import synth
        from oracle import eagle_oracle as eo  # the CPU checker doubles as the CPU baseline
        from oracle import np_oracle as npo
        self.eo, self.n, self.L, self.Ls = eo, n, L, int(min(L, Ls))
        self.cores = host_cores()
        self.blas = eo.use_openblas_dgemm(self.cores)
        self.dir = tempfile.TemporaryDirectory(prefix="eagle_ref_")
        G = synth.genotypes(n, self.Ls, seed=GENO_SEED, n_total=n)
        self.m, self.mt = os.path.join(self.dir.name, "M.ascii"), os.path.join(self.dir.name, "Mt.ascii")
        npo.write_ascii(self.m, G)
        npo.write_ascii(self.mt, np.ascontiguousarray(G.T))
        del G
        rng = np.random.default_rng(1)
        S = rng.standard_normal((n, n)); S = (S + S.T) * (0.5 / np.sqrt(n)) + 2 * np.eye(n)
        V = rng.standard_normal((n, n)); V = (V + V.T) * (0.5 / np.sqrt(n)) + 1.5 * np.eye(n)
        self.S, self.V, self.a = np.asfortranarray(S), np.asfortranarray(V), rng.standard_normal(n)

    def step(self):
        """One timed pass over the sample -> (markers/s extrapolated to the whole workload, stage seconds)."""
        eo, n, L, Ls = self.eo, self.n, self.L, self.Ls
        t0 = time.perf_counter()
        K = eo.calculateMMt_rcpp(self.m, 1e9, self.cores, [eo.NA_REAL], (n, Ls))
        st = eo.last_stages()
        t = {"decode_M": st["readblock"], "mmt": st["mmt_gemm"]}
        r = eo.calculate_a_and_vara_rcpp(self.mt, [eo.NA_REAL], self.S, self.V, 1e9, (Ls, n), self.a)
        st = eo.last_stages()
        t.update(decode_Mt=st["readblock"], S_a=st["S_a"], pre_products=st["pre_products"], Mt_W=st["Mt_W"],
                 rowdots=st["rowdots"], Mt_v=st["Mt_v"])
        wall = time.perf_counter() - t0
        _ = (K[0, 0], r["a"][0], r["vara"][0])
        linear = t["decode_M"] + t["mmt"] + t["decode_Mt"] + t["Mt_v"] + t["Mt_W"] + t["rowdots"]
        const = t["S_a"] + t["pre_products"]
        total = linear * (L / Ls) + const
        t["gemm_gflops"] = 2.0 * Ls * n * n / max(t["Mt_W"], 1e-9) / 1e9
        return L / total, t, wall

    def baseline(self, value, t, wall):
        return dict(value=value, unit=METRIC, cores=self.cores, kind="port",
                    sample=f"oracle/eagle_oracle.c control flow (ReadBlock getline decode from files, in-memory branches) "
                           f"with {self.blas} for the products, {self.cores} threads, on {self.Ls} of {self.L} markers at "
                           f"n={self.n}: decode M {t['decode_M']:.2f}s + Mt {t['decode_Mt']:.2f}s, M.Mt {t['mmt']:.2f}s, "
                           f"Mt*W {t['Mt_W']:.2f}s ({t['gemm_gflops']:.0f} GFLOP/s), row dots {t['rowdots']:.2f}s, Mt*v "
                           f"{t['Mt_v']:.2f}s scaled by L/sample; W=S(VS) {t['pre_products']:.2f}s and S*a {t['S_a']:.3f}s "
                           f"counted once",
                    seconds=wall, stage_seconds={k: round(v, 4) for k, v in t.items()})


def cpu_reference_sample(n, L, steps=1, warmup=0):
    ref = CpuReference(n, L)
    for _ in range(warmup):
        ref.step()
    vals, last = [], None
    for _ in range(max(1, steps)):
        last = ref.step()
        vals.append(last[0])
    v = sorted(vals)[len(vals) // 2]          # median pass
    out = ref.baseline(v, last[1], last[2])
    out["per_step_values"] = [round(x, 1) for x in vals]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    n, L = w["n"], w["L"]
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    t0 = time.perf_counter()
    last = cpu_reference_sample(n, L, steps=args.steps, warmup=min(args.warmup, 1))
    wall = time.perf_counter() - t0
    v = last["value"]
    jprint({"impl": "reference", "metric": METRIC, "value": v, "unit": METRIC, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * L / v, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": bench_config(w, n, L, world),
            "note": "CPU restatement of the reference path (the reference itself runs inside R with RcppEigen); "
                    f"{args.steps} timed passes over the same fixed {REF_SAMPLE_MARKERS}-marker sample",
            "cpu_baseline": last,
            "e2e": {"value": v, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": wall})


# ====================================================================== GPU arm
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measure_library_ceilings(torch):
    """cuBLAS ceilings measured in this run: FP64 DGEMM (denominator of the scan roofline; there is no
    FP64 entry in MEASURED_PEAKS.json) and the int8 GEMM reachable through torch._int_mm."""
    out = {}
    N = 8192
    a = torch.randn(N, N, dtype=torch.float64, device="cuda")
    b = torch.randn(N, N, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(); a @ b; e1.record(); e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    out["dgemm_tflops"] = 2.0 * N ** 3 / (best * 1e-3) / 1e12
    del a, b
    try:
        ai = torch.randint(-1, 2, (N, N), dtype=torch.int8, device="cuda")
        bi = torch.randint(-1, 2, (N, N), dtype=torch.int8, device="cuda")
        for _ in range(2):
            torch._int_mm(ai, bi)
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
            e0.record(); torch._int_mm(ai, bi); e1.record(); e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        out["int8_gemm_tops"] = 2.0 * N ** 3 / (best * 1e-3) / 1e12
        # the same GEMM back to back for ~1.5 s: what the library sustains under the 1 kW power cap
        reps = max(50, int(1.5 / (best * 1e-3)))
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(reps):
            torch._int_mm(ai, bi)
        e1.record(); e1.synchronize()
        out["int8_gemm_tops_sustained"] = 2.0 * N ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12
        torch.cuda.synchronize()
        time.sleep(1.0)  # let the clocks recover before the timed region
    except Exception as ex:  # noqa: BLE001
        out["int8_gemm_tops"] = None
        out["int8_gemm_note"] = f"torch._int_mm unavailable: {type(ex).__name__}"
    return out


class TailGuard:
    """Watchdog over the legs that follow the timed region.  Rank 0 holds the output line; when the deadline passes with
    a leg still running (a rank that failed inside a collective leaves the others waiting), rank 0 prints the line with
    the legs that did finish and a note naming the one that did not, and every rank leaves with status 0."""

    def __init__(self, rank, out, seconds):
        import threading
        self.rank, self.out, self.leg, self.lock, self.done = rank, out, None, threading.Lock(), False
        self.timer = threading.Timer(seconds + (0.0 if rank == 0 else 10.0), self._expired)
        self.timer.daemon = True
        self.timer.start()

    def _expired(self):
        with self.lock:
            if self.done:
                return
            self.done = True
            try:
                if self.out is not None:
                    self.out["tail_note"] = f"leg '{self.leg}' did not finish before the deadline; the line is printed without it"
                    for _ in range(3):          # the main thread may be filling in a leg's dictionary right now
                        try:
                            line = json.dumps(self.out)
                            break
                        except RuntimeError:
                            time.sleep(0.05)
                    else:
                        line = json.dumps({k: v for k, v in self.out.items() if k != "extra_workloads"})
                    print(line, flush=True)
            finally:
                os._exit(0)

    def finish(self):
        with self.lock:
            if self.done:       # the watchdog is printing
                time.sleep(3600)
            self.done = True
            self.timer.cancel()
        if self.out is not None:
            jprint(self.out)


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from eagleeverything_b200 import _lib, device
    from eagleeverything_b200 import dist as egd

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = device.init(local)
    w = WORKLOADS[args.workload]
    n, L = w["n"], w["L"]
    c0, c1 = egd.shard_range(L, world, rank)
    Lg = c1 - c0
    peaks = load_peaks()
    ceil = measure_library_ceilings(torch) if rank == 0 else {}

    # ---------------- inputs resident in HBM
    img = device.synth_ascii(n, Lg, GENO_SEED, col_offset=c0, n_total=n)
    g = torch.Generator(device="cuda"); g.manual_seed(1234)
    S = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    S = (S + S.T) * (0.5 / n ** 0.5); S.diagonal().add_(2.0)
    V = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    V = (V + V.T) * (0.5 / n ** 0.5); V.diagonal().add_(1.5)
    ah = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    pitch_t = device.store_pitch(n)
    store = torch.empty(((Lg + 127) // 128, n, 128), dtype=torch.int8, device="cuda")  # K-blocked M store
    storeT = torch.empty((Lg, pitch_t), dtype=torch.int8, device="cuda")
    err = torch.zeros(4, dtype=torch.int32, device="cuda")
    C32 = torch.empty((n, n), dtype=torch.int32, device="cuda")
    K = torch.empty((n, n), dtype=torch.float64, device="cuda")
    Wp = torch.empty(lib.eg_scan_wp_elems(n), dtype=torch.float64, device="cuda")
    tmp = torch.empty(n * n, dtype=torch.float64, device="cuda")
    oa = torch.empty(Lg, dtype=torch.float64, device="cuda")
    ov = torch.empty(Lg, dtype=torch.float64, device="cuda")

    STAGES = ["decode", "transpose", "syrk", "allreduce", "finalize", "prepare", "scan", "argmax"]

    def step(evs=None):
        def mark(i):
            if evs is not None:
                evs[i].record()
        mark(0)
        device.decode_kb(img, Lg + 1, n, Lg, out=store, err=err)
        mark(1)
        device.transpose_kb(store, n, Lg, out=storeT)
        mark(2)
        device.syrk_kb(store, n, Lg, C32=C32, zero=True)
        mark(3)
        egd.allreduce_partial_mmt(C32)
        mark(4)
        device.mmt_finalize(C32, n, out=K)
        mark(5)
        if world > 1:
            device.scan_prepare_sharded(S, V, ah, n, rank, world, Wp=Wp, tmp=tmp)
        else:
            device.scan_prepare(S, V, ah, n, Wp=Wp, tmp=tmp)
        mark(6)
        device.scan(storeT, Lg, n, Wp, out_a=oa, out_vara=ov)
        mark(7)
        best, idx = device.argmax_tsq(oa, ov)
        res = egd.global_argmax(best, idx, c0) if world > 1 else (best, idx)
        mark(8)
        return res

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sync_all()
    assert int(err[0].item()) == 0, "synthetic image failed decode validation"

    # the decode kernel timed alone (burst clocks), beside its in-step figure: at the head of a step it inherits the
    # power-capped clocks of the previous step's scan
    time.sleep(0.5)
    de0, de1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    device.decode_kb(img, Lg + 1, n, Lg, out=store, err=err)
    de0.record()
    for _ in range(5):
        device.decode_kb(img, Lg + 1, n, Lg, out=store, err=err)
    de1.record()
    sync_all()
    decode_alone_ms = de0.elapsed_time(de1) / 5.0
    time.sleep(0.5)

    sampler = ClockSampler(local) if rank == 0 else None
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(9)] for _ in range(args.steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    launches0 = int(lib.eg_launch_count())
    t0.record()
    for k in range(args.steps):
        res = step(evs[k])
    t1.record()
    sync_all()
    launches = int(lib.eg_launch_count()) - launches0
    clocks = sampler.stop() if sampler else None
    ms_total = t0.elapsed_time(t1)
    stage_ms = [sum(evs[k][i].elapsed_time(evs[k][i + 1]) for k in range(args.steps)) / args.steps for i in range(8)]
    if os.environ.get("EAGLE_BENCH_DEBUG"):
        print(f"[rank {rank}] stage_ms " + " ".join(f"{a}={b:.2f}" for a, b in zip(STAGES, stage_ms)), file=sys.stderr, flush=True)
    if world > 1:
        tt = torch.tensor([ms_total] + stage_ms, dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, stage_ms = tt[0].item(), tt[1:].tolist()
    ms_step = ms_total / args.steps
    value = L / (ms_step * 1e-3)

    mode = int(lib.eg_get_scan_mode())
    k_ms, k_ops, p_ms, p_ops = C.c_double(), C.c_double(), C.c_double(), C.c_double()
    _lib.check(lib.eg_last_scan_kernel(C.byref(k_ms), C.byref(k_ops)))   # CUDA events around the scan kernel of the last timed step
    _lib.check(lib.eg_last_prep_kernels(C.byref(p_ms), C.byref(p_ops)))
    # ---------------- results of the last step, hashed (the same hashes must come out at every N) and, at N > 1, compared
    # bit for bit with a single-GPU run of the same data set computed here (rank 0) -- a mismatch fails the run
    a_all, v_all = egd.gather_sharded(oa, L, world), egd.gather_sharded(ov, L, world)   # a, var(a) over ALL markers
    checks = result_checks(args, torch, dist, device, egd, lib, n, L, Lg, c0, world, rank, K, a_all, v_all, S, V, ah, res)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, K, a_all, v_all, res)
    del a_all, v_all
    if checks.get("failed"):
        if rank == 0:
            jprint({"metric": METRIC, "value": None, "n_gpus": world, "error": "multi-rank parity failed", "checks": checks})
        if world > 1:
            dist.destroy_process_group()
        sys.exit(3)

    # ---------------- the line as far as the timed region decides it; the legs below fill in their parts.  They use
    # collectives and one process driving every GPU: should one of them stall, the guard prints the line with what is
    # there instead of losing the measurement to NCCL's ten-minute timeout
    out = None
    if rank == 0:
        stages = dict(zip(STAGES, stage_ms))
        k_ms, k_ops = k_ms.value, k_ops.value
        # reference-equivalent FP64 work of the scan (full T = Mt*W, row-dot): 2n(n+1)+2n flops per marker
        scan_ref_flops = (2.0 * n * (n + 1) + 2.0 * n) * Lg
        syrk_ops = float(Lg) * n * (n + 1)                      # symmetric half, 2 ops per MAC
        dec_bytes = float(n) * (Lg + 1) + float(n) * Lg
        syrk_tops = syrk_ops / (stages["syrk"] * 1e-3) / 1e12
        dec_gbs = dec_bytes / (stages["decode"] * 1e-3) / 1e9
        dgemm = ceil.get("dgemm_tflops") or 37.0
        int8_meas = ceil.get("int8_gemm_tops")
        # int8 denominators.  MEASURED_PEAKS.json has no int8 entry: the peak of the line is the cuBLASLt int8 GEMM measured
        # in THIS run -- its sustained figure (~1.5 s back to back), since these kernels are timed inside a long power-capped
        # step -- with the burst figure, the 2 x bf16 proxies from MEASURED_PEAKS.json and the nominal 4500 beside it
        proxy_sust, proxy_burst = 2.0 * peaks["bf16_tflops_sustained"], 2.0 * peaks["bf16_tflops"]
        int8_peak = ceil.get("int8_gemm_tops_sustained") or proxy_sust
        int8_burst = int8_meas or proxy_burst
        int8_src = ("cuBLASLt int8 GEMM 8192^3 measured in this run, sustained over ~1.5 s (burst: %.0f); proxies 2 x measured bf16 "
                    "from MEASURED_PEAKS.json: %.0f sustained / %.0f burst; nominal 4500" % (int8_burst, proxy_sust, proxy_burst)
                    if ceil.get("int8_gemm_tops_sustained") else
                    "2 x measured sustained bf16 (no int8 entry in MEASURED_PEAKS.json, in-run int8 GEMM unavailable); 2 x burst bf16 = %.0f, "
                    "nominal 4500" % proxy_burst)

        def int8_fracs(rate):
            return {"frac": rate / int8_peak, "frac_of_burst_peak": rate / int8_burst,
                    "frac_of_2x_bf16_sustained": rate / proxy_sust, "frac_of_2x_bf16_burst": rate / proxy_burst, "frac_of_nominal_4500": rate / 4500.0}
        k_rate = k_ops / (k_ms * 1e-3) / 1e12
        if mode == 1:
            roofline = {"kernel": "scan_i8_kernel", "bound": "tensor", "achieved": k_rate, "peak": int8_peak,
                        "unit": "TOP/s (int8)", **int8_fracs(k_rate), "executed_ops": k_ops,
                        "digits": int(lib.eg_get_scan_digits()), "algorithmic_ops": float(lib.eg_get_scan_digits()) * Lg * n * (n + 1),
                        "traffic": None, "kernel_ms": k_ms,
                        "ops_convention": "executed int8 ops: `digits` balanced-byte slices x symmetric-half contraction, 2 ops per MAC "
                                          "(DESIGN.md section 4)",
                        "reference_equiv_fp64_tflops": scan_ref_flops / (k_ms * 1e-3) / 1e12,
                        "peak_source": int8_src, "cublaslt_int8_gemm_tops_this_run": int8_meas,
                        "cublaslt_int8_gemm_tops_sustained_this_run": ceil.get("int8_gemm_tops_sustained")}
        else:
            roofline = {"kernel": "scan_f64_kernel", "bound": "tensor", "achieved": k_rate, "peak": dgemm,
                        "unit": "TFLOP/s (fp64)", "frac": k_rate / dgemm, "traffic": None, "kernel_ms": k_ms,
                        "ops_convention": "executed FP64 flops of the symmetric-half contraction (DESIGN.md section 4)",
                        "reference_equiv_fp64_tflops": scan_ref_flops / (k_ms * 1e-3) / 1e12,
                        "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (MEASURED_PEAKS.json has no FP64 "
                                       "entry); B200 FP64 nominal 37-40 TFLOP/s"}
        rooflines = {
            "decode_kb_kernel": {"bound": "hbm", "achieved": dec_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "frac": dec_gbs / peaks["hbm_gbs"], "peak_source": peaks["source"],
                                 "timed_alone_gbs": dec_bytes / (decode_alone_ms * 1e-3) / 1e9,
                                 "timed_alone_frac": dec_bytes / (decode_alone_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                 "note": "achieved/frac = inside the step (power-capped clocks inherited from the previous "
                                         "step's scan); timed_alone = 5 back-to-back launches after an idle gap"},
            "transpose_kb128_kernel": {"bound": "hbm", "achieved": 2.0 * n * Lg / (stages["transpose"] * 1e-3) / 1e9,
                                       "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                       "frac": 2.0 * n * Lg / (stages["transpose"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                       "peak_source": peaks["source"]},
            "syrk_i8_kernel": {"bound": "tensor", "achieved": syrk_tops, "unit": "TOP/s (int8, symmetric-half ops)",
                               "full_product_equiv_tops": 2.0 * n * n * Lg / (stages["syrk"] * 1e-3) / 1e12,
                               "peak": int8_peak, **int8_fracs(syrk_tops), "algorithmic_ops": syrk_ops,
                               "peak_source": int8_src, "cublaslt_int8_gemm_tops_this_run": int8_meas},
            roofline["kernel"]: roofline,
        }
        if p_ms.value > 0:
            p_rate = p_ops.value / (p_ms.value * 1e-3) / 1e12
            rooflines["prep_i8_kernel"] = {"bound": "tensor", "achieved": p_rate, "unit": "TOP/s (int8)", "peak": int8_peak,
                                           **int8_fracs(p_rate), "executed_ops": p_ops.value,
                                           "kernel_ms": p_ms.value, "peak_source": int8_src,
                                           "ops_convention": "executed int8 ops of the 28 + 28 digit-slice products of "
                                                             "X = V S and upper(W = S X); reference-equivalent FP64: 3 n^3 flops",
                                           "reference_equiv_fp64_tflops": 3.0 * n ** 3 / (stages["prepare"] * 1e-3) / 1e12}
        scan_tf = scan_ref_flops / (stages["scan"] * 1e-3) / 1e12
        # DRAM traffic per launch from the committed `ncu --set full` capture of the same kernel at the same shape
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:  # noqa: BLE001
            tr = {}
        for kname, rf in rooflines.items():
            rec = tr.get(kname)
            if rec and rec.get("workload") == args.workload and rec.get("n_gpus") == world:
                rf["traffic"] = rec["dram_bytes_per_launch"]
                rf["traffic_source"] = rec.get("source")
                if "tensor_pipe_active_pct" in rec:
                    rf["tensor_pipe_active_pct_ncu"] = rec["tensor_pipe_active_pct"]
            else:
                rf.setdefault("traffic", None)
        out = {
            "metric": METRIC, "value": value, "unit": METRIC, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": bench_config(w, n, L, world),
            "config_detail": {"markers_per_gpu": Lg, "parallelism": f"markers/{world}",
                              "l2": f"inputs larger than L2 ({(dec_bytes + 16.0 * n * n) / 1e9:.1f} GB streamed per step)",
                              "note": "dtype f64 = the scan's results (a, var(a)); decode is u8, M.Mt is s8 x s8 -> s32 "
                                      "(bit-exact); var(a) is contracted on int8 slices of the FP64 matrix (exact) or on FP64 DMMA"},
            "stage_ms": stages, "mmt_int8_tops": syrk_tops, "decode_gbs": dec_gbs,
            "scan_mode": f"int8 slices (tcgen05), {int(lib.eg_get_scan_digits())} digits per column" if mode == 1 else "fp64 (DMMA)", "scan_reference_equiv_fp64_tflops": scan_tf,
            "roofline": roofline, "rooflines": rooflines, "cpu_baseline": None, "e2e": None, "clocks": clocks,
            "allreduce": (None if world == 1 else {
                "bytes": 4 * n * n, "ms": stages["allreduce"],
                "algbw_gbs": 4.0 * n * n / (stages["allreduce"] * 1e-3) / 1e9,
                "busbw_gbs": 2.0 * (world - 1) / world * 4.0 * n * n / (stages["allreduce"] * 1e-3) / 1e9,
                "note": "NCCL int32 sum of the n x n partial M.Mt; measured reference on this pool: 725 GB/s bus bandwidth "
                        "for an 8-rank all-reduce at 1 GiB (B200_PROFILING.md)"}),
            "gpu_launches": launches, "library_ceilings": ceil, "forward_search": None, "checks": checks,
            "extra_workloads": None,
            "picked_marker": int(res[1]) if not hasattr(res[1], "item") else int(res[1].item()),
        }
    guard = TailGuard(rank, out, float(os.environ.get("EAGLE_BENCH_TAIL_S", "900")))

    # ---------------- end to end with host buffers (H2D of the image / S / V / a, D2H of K, a, vara)
    if args.no_e2e:
        e2e = {"value": None, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": "skipped (--no-e2e)"}
    else:
        del store, storeT, C32, K, Wp, tmp, oa, ov
        torch.cuda.empty_cache()
        if world > 1 and rank != 0:   # the ranks' GPUs are driven by rank 0 alone in this leg; inputs are rebuilt after it
            img = S = V = ah = None
            torch.cuda.empty_cache()
        guard.leg = "e2e"
        e2e = run_e2e(args, torch, dist, lib, device, egd, n, L, Lg, c0, world, rank, img, S, V, ah)
        if world > 1 and rank != 0:
            img = device.synth_ascii(n, Lg, GENO_SEED, col_offset=c0, n_total=n)

    if out is not None:
        out["e2e"] = e2e

    # BASELINE config 3 as it is worded: the full forward search, marker-sharded at N > 1 (collective calls: every rank)
    search = None
    if not args.no_search and args.workload in ("c2", "c3"):
        guard.leg = "forward_search"
        try:
            search = run_forward_search(args, torch, dist, egd, n, L, Lg, c0, world, rank, img)
        except Exception as ex:  # noqa: BLE001
            search = {"note": f"failed: {type(ex).__name__}: {ex}"}
    if out is not None:
        out["forward_search"] = search
    extras = None
    if (world >= 8 or os.environ.get("EAGLE_BENCH_EXTRAS_SHRINK")) and world > 1 and args.workload == "c3" and not args.no_extras:
        del img, S, V, ah
        torch.cuda.empty_cache()
        extras = {}
        if out is not None:
            out["extra_workloads"] = extras
        for wl in ("c5", "c4"):
            guard.leg = "extra_workloads." + wl
            try:
                extras[wl] = run_extra_workload(args, wl, torch, dist, device, egd, lib, world, rank)
            except Exception as ex:  # noqa: BLE001
                extras[wl] = {"note": f"failed: {type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()

    if rank != 0:
        guard.finish()
        if world > 1:
            dist.destroy_process_group()
        return

    guard.leg = "cpu_baseline"
    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            cpu = cpu_reference_sample(n, L, steps=3, warmup=1)   # the same passes as --impl reference: warm-up, then the median
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": METRIC, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    out["cpu_baseline"] = cpu
    guard.finish()
    if world > 1:
        dist.destroy_process_group()


def _wait_rank0(dist, rank, world, key):
    """CPU-side rendezvous (the TCP store): the other ranks' GPUs must stay idle while rank 0 drives them itself."""
    if world == 1:
        return
    from datetime import timedelta
    store = dist.distributed_c10d._get_default_store()
    if rank == 0:
        store.set(key, "1")
    else:
        store.wait([key], timedelta(seconds=3600))


def run_e2e(args, torch, dist, lib, device, egd, n, L, Lg, c0, world, rank, img, S, V, ah):
    """The same step end to end through the C ABI a single R session would call, with HOST buffers in and out, on the
    N GPUs of the run: ONE process (rank 0 of the launch; the other ranks release their GPUs and wait), eg_init_multi(N)
    -- one host thread per GPU, NCCL inside the library -- then per step
        eg_store_from_host_ascii (the whole M.ascii image: every GPU pulls and decodes its own marker columns, M.Mt of each
        chunk accumulated under the copy)  ->  eg_store_mmt (all-reduce, K back to the host in parallel row blocks)
        ->  eg_store_transpose  ->  eg_store_a_and_vara (S, V uploaded once in 1/N slices and exchanged over NVLink; a,
        var(a) written by every GPU into the host vectors)  ->  the pick on the host vectors (find_qtl.R:71-80).
    Extra legs: the drop-in route of the Rcpp exports on FILES with pageable S / V (first call and steady state), and at
    N = 1 the packed 2-bit container."""
    from eagleeverything_b200 import _lib
    import numpy as np
    vp = C.c_void_p
    dp = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_double))  # noqa: E731
    if rank != 0:
        del img, S, V, ah
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        store = dist.distributed_c10d._get_default_store()
        store.set("e2e_free_%d" % rank, "1")
        _wait_rank0(dist, rank, world, "e2e_done")
        return None
    img_bytes = n * (L + 1)
    try:
        if world > 1:
            full = device.synth_ascii(n, L, GENO_SEED, col_offset=0, n_total=n)
        else:
            full = img
        img_h = torch.empty(img_bytes + 64, dtype=torch.uint8, pin_memory=True)
        img_h[:img_bytes].copy_(full[:img_bytes]); img_h[img_bytes:].zero_()
        del full
        S_h = torch.empty((n, n), dtype=torch.float64, pin_memory=True); S_h.copy_(S)
        V_h = torch.empty((n, n), dtype=torch.float64, pin_memory=True); V_h.copy_(V)
        a_h = torch.empty(n, dtype=torch.float64, pin_memory=True); a_h.copy_(ah)
        K_h = torch.empty((n, n), dtype=torch.float64, pin_memory=True)
        oa_h = torch.empty(L, dtype=torch.float64, pin_memory=True)
        ov_h = torch.empty(L, dtype=torch.float64, pin_memory=True)
    except RuntimeError as ex:
        _wait_rank0(dist, rank, world, "e2e_done")
        return {"value": None, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": f"could not pin host buffers: {ex}"}
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    try:
        return _run_e2e_rank0(args, torch, dist, lib, device, n, L, world, rank, img, img_h, S_h, V_h, a_h, K_h, oa_h, ov_h)
    finally:
        if world > 1:
            try:   # back to this rank's own GPU whatever happened, and release the ranks that wait on the TCP store
                lib.eg_shutdown()
                lib.eg_init(int(os.environ.get("LOCAL_RANK", "0")))
            finally:
                _wait_rank0(dist, rank, world, "e2e_done")


def _run_e2e_rank0(args, torch, dist, lib, device, n, L, world, rank, img, img_h, S_h, V_h, a_h, K_h, oa_h, ov_h):
    from eagleeverything_b200 import _lib
    vp = C.c_void_p
    dp = lambda t: C.cast(t.data_ptr(), C.POINTER(C.c_double))  # noqa: E731
    img_bytes = n * (L + 1)
    if world > 1:   # the other ranks have released their memory
        from datetime import timedelta
        store = dist.distributed_c10d._get_default_store()
        store.wait(["e2e_free_%d" % r for r in range(1, world)], timedelta(seconds=600))
        _lib.check(lib.eg_init_multi(world, None))
    ngpu = int(lib.eg_gpu_count())

    def pick_host():
        tsq = oa_h * oa_h / ov_h                     # the R side's pick (find_qtl.R:71-80) on the host result
        return int(torch.argmax(torch.nan_to_num(tsq, nan=-1.0)))

    def step_host_abi():
        h, ht = vp(), vp()
        _lib.check(lib.eg_store_from_host_ascii(vp(img_h.data_ptr()), n, L, 0, L, C.byref(h)))
        _lib.check(lib.eg_store_mmt(h, None, 0, dp(K_h)))
        _lib.check(lib.eg_store_transpose(h, C.byref(ht)))
        _lib.check(lib.eg_store_a_and_vara(ht, None, 0, dp(S_h), dp(V_h), dp(a_h), dp(oa_h), dp(ov_h)))
        lib.eg_store_free(h); lib.eg_store_free(ht)
        return pick_host()

    ksteps = max(1, min(args.steps, args.e2e_steps))

    def time_host(f, reps=ksteps, warm=1):
        for _ in range(warm):
            f()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = f()
        wall_ms = (time.perf_counter() - t0) * 1e3   # every call of the host-level ABI synchronises before it returns
        return wall_ms / reps, r

    out = {}
    try:
        ms, picked = time_host(step_host_abi)
        t8 = (C.c_double * 8)()
        lib.eg_last_timing(t8, 8)
        abi_timing = dict(zip(["h2d_decode_ms", "syrk_ms", "allreduce_or_finalize_ms", "mmt_d2h_ms", "scan_h2d_ms", "prepare_ms",
                               "scan_ms", "scan_d2h_ms"], [round(x, 3) for x in t8]))
        out = {"value": L / (ms * 1e-3), "unit": METRIC, "ms_per_step": ms, "steps": ksteps, "n_gpus": ngpu,
               "h2d_bytes_per_step": int(img_bytes + 2 * n * n * 8 + n * 8), "d2h_bytes_per_step": int(n * n * 8 + 2 * L * 8),
               "picked_marker": picked, "abi_stage_ms_gpu0_last_step": abi_timing,
               "path": "host-level C ABI (eg_store_from_host_ascii / eg_store_mmt / eg_store_transpose / eg_store_a_and_vara) on pinned "
                       "host buffers, ONE process" + (f", eg_init_multi({ngpu}): one host thread per GPU, NCCL inside the library" if ngpu > 1 else ""),
               "timing": "host clock around the calls (each returns after its results are in host memory)"}
    except Exception as ex:  # noqa: BLE001
        out = {"value": None, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "note": f"failed: {type(ex).__name__}: {ex}"}
    # ---- the drop-in route: the Rcpp exports on files, S / V / outputs in pageable memory as R owns them
    if not args.no_dropin:
        try:
            out["dropin_files"] = run_dropin(args, torch, lib, device, n, L, img_h, S_h, V_h, a_h, time_host)
        except Exception as ex:  # noqa: BLE001
            out["dropin_files"] = {"note": f"failed: {type(ex).__name__}: {ex}"}
    if ngpu == 1:
        # the same step from the packed 2-bit container (SURVEY.md 8(f) rank 2): 4x fewer bytes over PCIe
        try:
            wpr = int(lib.eg_packed_words_per_row(L))
            kb = torch.empty(((L + 127) // 128, n, 128), dtype=torch.int8, device="cuda")
            device.decode_kb(img, L + 1, n, L, out=kb)
            wd = torch.empty((n, wpr), dtype=torch.int64, device="cuda")
            _lib.check(lib.eg_dev_pack_2bit(vp(kb.data_ptr()), n, L, 0, vp(wd.data_ptr()), None))
            words_h = torch.empty((n, wpr), dtype=torch.int64, pin_memory=True); words_h.copy_(wd)
            del kb, wd
            torch.cuda.synchronize()
            torch.cuda.empty_cache()

            def step_host_packed():
                h, ht = vp(), vp()
                _lib.check(lib.eg_store_from_host_packed(vp(words_h.data_ptr()), n, L, 1, C.byref(h)))
                _lib.check(lib.eg_store_mmt(h, None, 0, dp(K_h)))
                _lib.check(lib.eg_store_transpose(h, C.byref(ht)))
                _lib.check(lib.eg_store_a_and_vara(ht, None, 0, dp(S_h), dp(V_h), dp(a_h), dp(oa_h), dp(ov_h)))
                lib.eg_store_free(h); lib.eg_store_free(ht)
                return pick_host()
            pms, ppick = time_host(step_host_packed)
            out["from_packed_container"] = {
                "value": L / (pms * 1e-3), "unit": METRIC, "ms_per_step": pms,
                "h2d_bytes_per_step": int(n * wpr * 8 + 2 * n * n * 8 + n * 8), "picked_marker": ppick,
                "container": "2-bit packed genotypes (RcppFunctions.cpp.gpu:224-345 layout) instead of the ASCII image"}
        except Exception as ex:  # noqa: BLE001
            out["from_packed_container"] = {"value": None, "note": f"{type(ex).__name__}: {ex}"}
    return out


def run_dropin(args, torch, lib, device, n, L, img_h, S_h, V_h, a_h, time_host):
    """What the untouched R package does per forward step, through the entry points its Rcpp glue binds
    (src/RcppExports.cpp:37-71): calculateMMt_rcpp(M.ascii) and calculate_a_and_vara_rcpp(Mt.ascii, S, V, a) on FILES (in
    the page cache), every matrix and vector in PAGEABLE host memory as R owns them.  `first_call`: nothing resident (a
    fresh R session); `steady_state`: the genotype stores are resident under their path (every later iteration of AM(), or
    an AM() that follows ReadMarker() in the same session) -- the contraction still runs (EAGLE_KEEP_PRODUCT=0)."""
    import shutil
    import tempfile

    import numpy as np

    from eagleeverything_b200 import _lib
    need = 2 * n * (L + 1) + (1 << 26)
    base = None
    for cand in ("/dev/shm", tempfile.gettempdir()):
        try:
            if shutil.disk_usage(cand).free > need * 1.2:
                base = cand
                break
        except OSError:
            pass
    if base is None:
        return {"note": "no room for the two ASCII files"}
    d = tempfile.mkdtemp(prefix="eagle_bench_", dir=base)
    vp = C.c_void_p
    try:
        m, mt = os.path.join(d, "M.ascii"), os.path.join(d, "Mt.ascii")
        t0 = time.perf_counter()
        img_np = img_h[: n * (L + 1)].numpy()
        with open(m, "wb") as f:
            f.write(memoryview(img_np))
        # Mt.ascii through the library's own writer (createMt_ASCII_rcpp: decode, transpose, encode on the device)
        dims = (C.c_int64 * 2)(n, L)
        _lib.check(lib.eg_createMt_ASCII_rcpp(os.fsencode(m), os.fsencode(mt), b"text", 8.0, dims, 1, _lib.MESSAGE_FN(0), None))
        lib.eg_cache_clear()
        t_files = time.perf_counter() - t0
        S_p, V_p, a_p = S_h.numpy().copy(), V_h.numpy().copy(), a_h.numpy().copy()      # pageable copies
        K_p, oa_p, ov_p = np.empty((n, n)), np.empty(L), np.empty(L)
        NA = np.array([float("nan")])
        dpp = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))  # noqa: E731
        dimsM, dimsMt = (C.c_int64 * 2)(n, L), (C.c_int64 * 2)(L, n)
        os.environ["EAGLE_KEEP_PRODUCT"] = "0"
        stage = {}

        def step():
            t1 = time.perf_counter()
            _lib.check(lib.eg_calculateMMt_rcpp(os.fsencode(m), 8.0, 1, dpp(NA), 1, dimsM, 1, _lib.MESSAGE_FN(0), None, dpp(K_p)))
            t2 = time.perf_counter()
            _lib.check(lib.eg_calculate_a_and_vara_rcpp(os.fsencode(mt), dpp(NA), 1, dpp(S_p), dpp(V_p), 8.0, dimsMt, dpp(a_p), 1,
                                                        _lib.MESSAGE_FN(0), None, dpp(oa_p), dpp(ov_p)))
            t3 = time.perf_counter()
            stage["calculateMMt_rcpp_ms"], stage["calculate_a_and_vara_rcpp_ms"] = (t2 - t1) * 1e3, (t3 - t2) * 1e3
            with np.errstate(divide="ignore", invalid="ignore"):
                tsq = oa_p * oa_p / ov_p
            return int(np.nanargmax(tsq))

        def cold():
            lib.eg_cache_clear()
            return step()
        first_ms, pick1 = time_host(cold, reps=1, warm=0)
        first_stage = {k: round(v, 2) for k, v in stage.items()}
        steady_ms, pick2 = time_host(step, reps=3, warm=1)
        steady_stage = {k: round(v, 2) for k, v in stage.items()}
        t8 = (C.c_double * 8)()
        lib.eg_last_timing(t8, 8)
        return {"first_call": {"ms_per_step": first_ms, "value": L / (first_ms * 1e-3), "unit": METRIC, "stages": first_stage,
                               "h2d_bytes": int(2 * n * (L + 1) + 2 * n * n * 8 + n * 8),
                               "what": "cache cleared: both files read from the page cache, uploaded and decoded inside the calls"},
                "steady_state": {"ms_per_step": steady_ms, "value": L / (steady_ms * 1e-3), "unit": METRIC, "stages": steady_stage,
                                 "h2d_bytes": int(2 * n * n * 8 + n * 8), "d2h_bytes": int(n * n * 8 + 2 * L * 8),
                                 "gpu0_stage_ms": dict(zip(["-", "syrk_ms", "allreduce_or_finalize_ms", "mmt_d2h_ms", "scan_h2d_ms",
                                                            "prepare_ms", "scan_ms", "scan_d2h_ms"], [round(x, 3) for x in t8])),
                                 "what": "genotype stores resident under their path; M.Mt contracted again on every call; S, V, a "
                                         "uploaded from and K, a, var(a) returned to pageable memory"},
                "picked_marker": [pick1, pick2], "files_in": base, "file_setup_s": round(t_files, 2),
                "path": "eg_calculateMMt_rcpp(path) + eg_calculate_a_and_vara_rcpp(path, S, V, a): the entry points the Rcpp glue binds"}
    finally:
        os.environ.pop("EAGLE_KEEP_PRODUCT", None)
        lib.eg_cache_clear()
        shutil.rmtree(d, ignore_errors=True)


DUMP_K_BYTES = 24 << 20   # rows of K kept by --dump-outputs; with a and var(a) of the largest workload under 64 MB
DUMP_SEED = 7


def dump_outputs(d, torch, K, a, vara, res):
    """--dump-outputs: what the timed step hands its caller, as one float64 .npy per array under `d`: a and var(a) of
    every marker, the picked marker and its t^2 statistic, and the rows of K -- every row when K fits DUMP_K_BYTES,
    otherwise a fixed seeded sample of rows, listed in K_rows_index.npy.  The inputs are seeded as well, so two builds
    run with the same arguments can be compared file by file."""
    import numpy as np
    n = K.shape[0]
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, min(n, DUMP_K_BYTES // (8 * n)), replace=False))
    arrays = {"a": a, "vara": vara, "K_rows": K[torch.from_numpy(rows).to(K.device)], "K_rows_index": rows,
              "picked_marker": [int(res[1])], "picked_tsq": [float(res[0])]}
    os.makedirs(d, exist_ok=True)
    for name, v in arrays.items():
        v = v.cpu().numpy() if torch.is_tensor(v) else v
        np.save(os.path.join(d, name + ".npy"), np.asarray(v, dtype=np.float64))


def _sha(t):
    import hashlib
    return hashlib.sha256(t.contiguous().cpu().numpy().tobytes()).hexdigest()


def result_checks(args, torch, dist, device, egd, lib, n, L, Lg, c0, world, rank, K, a_all, v_all, S, V, ah, res):
    """sha256 of the results of the last timed step -- K (after the all-reduce), a, var(a) over ALL markers, the pick -- so
    that the lines of a scaling run can be compared with each other; and at N > 1 (when the whole data set fits one GPU)
    the same step recomputed on rank 0 alone and compared bit for bit: the all-reduced K, every shard of a / var(a), the
    pick.  `failed` is set on any mismatch (the run then exits non-zero)."""
    out = {}
    picked = int(res[1]) if not hasattr(res[1], "item") else int(res[1].item())
    if world > 1:   # every rank holds the same K after the all-reduce: compare 128-bit fingerprints across ranks
        kv = K.view(torch.int64).reshape(-1)
        fp = torch.stack([kv.sum(), (kv * (torch.arange(kv.numel(), device=kv.device, dtype=torch.int64) | 1)).sum()])
        fps = torch.empty(2 * world, dtype=torch.int64, device=kv.device)
        dist.all_gather_into_tensor(fps, fp)
        out["K_identical_on_all_ranks"] = bool((fps.view(world, 2) == fp).all().item())
    if rank == 0:
        out.update(K_sha256=_sha(K), a_sha256=_sha(a_all), vara_sha256=_sha(v_all), picked_marker=picked)
    fits = 3.0 * n * (L + 1) + 60.0 * n * n < 120e9
    if world > 1 and not args.no_parity:
        if fits:
            if rank == 0:
                img_f = device.synth_ascii(n, L, GENO_SEED, col_offset=0, n_total=n)
                kb, err = device.decode_kb(img_f, L + 1, n, L)
                del img_f
                tT = device.transpose_kb(kb, n, L)
                C32 = device.syrk_kb(kb, n, L)
                del kb
                K1 = device.mmt_finalize(C32, n)
                del C32
                Wp1 = device.scan_prepare(S, V, ah, n)
                a1, v1 = device.scan(tT, L, n, Wp1)
                b1, i1 = device.argmax_tsq(a1, v1)
                out["vs_single_gpu"] = {
                    "K_bit_identical": bool(torch.equal(K1, K)), "a_bit_identical": bool(torch.equal(a1, a_all)),
                    "vara_bit_identical": bool(torch.equal(v1, v_all)), "pick_identical": int(i1.item()) == picked,
                    "how": "the same data set decoded, contracted and scanned on rank 0 alone in this run; compared with the "
                           "all-reduced K and the gathered shards of a / var(a)"}
                del K1, Wp1, a1, v1, tT
                torch.cuda.empty_cache()
                ok = all(v for k, v in out["vs_single_gpu"].items() if k != "how")
            flag = torch.tensor([1 if (rank != 0 or ok) else 0], device="cuda")
            dist.broadcast(flag, src=0)
            if not out.get("K_identical_on_all_ranks", True) or int(flag.item()) == 0:
                out["failed"] = True
        else:
            out["vs_single_gpu"] = {"note": "data set does not fit one GPU: spot checks instead (extra_workloads)"}
            if not out.get("K_identical_on_all_ranks", True):
                out["failed"] = True
    return out


def spot_check(torch, dist, device, egd, n, Lg, world, kb, tT, K, S, V, ah, oa, ov, rows=64, markers=1024):
    """Parity at sizes where nothing can be recomputed whole: `rows` rows of K and a / var(a) of `markers` of this rank's
    markers recomputed with plain FP64 torch products from the decoded genotypes (an independent evaluation of
    calculateMMt_rcpp.cpp:95 and calculate_a_and_vara_rcpp.cpp:90-112) -- K rows exactly, a / var(a) to 1e-9."""
    g = torch.Generator(device="cpu"); g.manual_seed(99)
    ridx = torch.randperm(n, generator=g)[:rows].cuda()
    # M of this shard as doubles (reference sign: stores hold the negated value, products do not see it)
    part = torch.zeros((rows, n), dtype=torch.float64, device="cuda")
    step = max(1024, int(2e9 / (8 * n)))
    for b0 in range(0, Lg, step):
        b1 = min(Lg, b0 + step)
        Mt_blk = tT[b0:b1, :n].to(torch.float64)              # (markers, n)
        part += Mt_blk[:, ridx].T @ Mt_blk
    if world > 1:
        dist.all_reduce(part)
    k_ok = bool(torch.equal(part, K[ridx, :]))
    midx = torch.randperm(Lg, generator=g)[:markers].cuda()
    Mj = tT[midx, :n].to(torch.float64).T.contiguous()          # n x markers, stored value = -(reference value)
    T1 = S @ Mj
    vara_ref = (T1 * (V @ T1)).sum(0)
    a_ref = -(Mj.T @ (S @ ah))
    av, vv = oa[midx], ov[midx]
    tol_v = 1e-9 * vara_ref.abs() + 4 * (n + 10) * 2.2e-16 * (T1.abs() * (V @ T1).abs()).sum(0)
    tol_a = 1e-9 * a_ref.abs() + 4 * (n + 10) * 2.2e-16 * (Mj.abs().T @ (S @ ah).abs())
    a_ok = bool(((av - a_ref).abs() <= tol_a).all().item())
    v_ok = bool(((vv - vara_ref).abs() <= tol_v).all().item())
    flags = torch.tensor([int(k_ok), int(a_ok), int(v_ok)], device="cuda")
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    return {"K_rows_checked": rows, "K_rows_exact": bool(flags[0].item()), "markers_checked_per_rank": markers,
            "a_within_1e-9": bool(flags[1].item()), "vara_within_1e-9": bool(flags[2].item()),
            "max_rel_err_vara": float(((vv - vara_ref).abs() / vara_ref.abs().clamp_min(1e-300)).max().item()),
            "how": "FP64 torch products from the decoded genotypes on every rank (K rows all-reduced)"}


def run_extra_workload(args, wl, torch, dist, device, egd, lib, world, rank):
    """One forward step of a shape that needs the 8 GPUs (BASELINE configs 4 and 5), recorded beside the headline run.
    c5 (n = 20,000 x L = 2,000,000, Z incidence matrix for repeated measures and fixed-effect covariates): a REAL first
    iteration of AM() with 30,000 records, X = [1, x1, x2] -- M.Mt, eigen(C^1/2 K C^1/2), EMMA's REML / ML with Z through the
    secular solve, the Z-aware right-hand side, the sharded scan and pick (am.AM_resident, maxit = 1, Z = ...) -- plus a
    kernel-level step with spot-check parity.
    c4 (n = 50,000 x L = 600,000): decode, M.Mt with the 10 GB int32 all-reduce, pre-products and scan on synthetic S, V
    (an eigendecomposition of order 50,000 is not part of this path), with spot-check parity."""
    import numpy as np
    from eagleeverything_b200 import am
    w = WORKLOADS[wl]
    n, L = w["n"], w["L"]
    shrink = float(os.environ.get("EAGLE_BENCH_EXTRAS_SHRINK", "1"))   # smoke tests of this leg on fewer GPUs
    if shrink > 1:
        n, L = int(n / shrink) // 32 * 32, int(L / shrink) // 128 * 128
    c0, c1 = egd.shard_range(L, world, rank)
    Lg = c1 - c0
    out = {"workload": w["name"] + (f" (shrunk by {shrink:g} for a smoke test)" if shrink > 1 else ""), "n": n, "L": L, "n_gpus": world}
    img = device.synth_ascii(n, Lg, GENO_SEED, col_offset=c0, n_total=n)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]

    def sync():
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    sync()
    ev[0].record()
    kb, err = device.decode_kb(img, Lg + 1, n, Lg)
    del img
    tT = device.transpose_kb(kb, n, Lg)
    ev[1].record()
    C32 = device.syrk_kb(kb, n, Lg)
    ev[2].record()
    egd.allreduce_partial_mmt(C32)
    ev[3].record()
    K = device.mmt_finalize(C32, n)
    del C32
    ev[4].record()
    g = torch.Generator(device="cuda"); g.manual_seed(1234)
    S = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    S = (S + S.T) * (0.5 / n ** 0.5); S.diagonal().add_(2.0)
    V = torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g)
    V = (V + V.T) * (0.5 / n ** 0.5); V.diagonal().add_(1.5)
    ah = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    # one untimed pass of the two stages whose workspaces depend on n (digit slices of S, V, X: 8 - 52 GB here; partial
    # sums of the scan): their first allocation is not part of a step.  torch's cache is emptied first: the library sizes
    # its digit-slice workspace by the FREE device memory, and at n = 50,000 the 14 GB of released image / int32 product
    # blocks that torch still held made it fall back to two library DGEMMs (1.4 s instead of 0.64 s).
    torch.cuda.empty_cache()
    Wp = device.scan_prepare_sharded(S, V, ah, n, rank, world)
    device.scan(tT, min(Lg, 4096), n, Wp)
    del Wp
    sync()
    ev[5].record()
    Wp = device.scan_prepare_sharded(S, V, ah, n, rank, world)
    ev[6].record()
    oa, ov = device.scan(tT, Lg, n, Wp)
    best, idx = device.argmax_tsq(oa, ov)
    pick = egd.global_argmax(best, idx, c0)
    ev[7].record()
    sync()
    ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(7)]
    tt = torch.tensor(ms, dtype=torch.float64, device="cuda")
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = tt.tolist()
    step_ms = ms[0] + ms[1] + ms[2] + ms[3] + ms[5] + ms[6]
    out["kernel_step"] = {"stage_ms": dict(zip(["decode_transpose", "syrk", "allreduce", "finalize", "(inputs)", "prepare", "scan_argmax"],
                                               [round(x, 3) for x in ms])),
                          "ms_per_step": step_ms, "markers_per_s": L / (step_ms * 1e-3),
                          "mmt_int8_tops_per_gpu": float(Lg) * n * (n + 1) / (ms[1] * 1e-3) / 1e12,
                          "allreduce_busbw_gbs": 2.0 * (world - 1) / world * 4.0 * n * n / (ms[2] * 1e-3) / 1e9,
                          "picked_marker": int(pick[1]), "inputs": "synthetic symmetric S, V, a_hat", "steps": 1}
    del Wp
    out["spot_check"] = spot_check(torch, dist, device, egd, n, Lg, world, kb, tT, K, S, V, ah, oa, ov)
    del S, V, K, oa, ov
    torch.cuda.empty_cache()
    if wl == "c5":
        rng = np.random.default_rng(11)          # the same on every rank
        nrec = n + n // 2                        # repeated measures: 1.5 records per individual (SURVEY.md 8(d))
        zidx = np.concatenate([np.arange(n), rng.integers(0, n, nrec - n)])
        rng.shuffle(zidx)
        X0 = np.column_stack([np.ones(nrec), rng.standard_normal(nrec), rng.integers(0, 2, nrec).astype(np.float64)])
        shard = egd.Shard(L, world, rank)
        qtl = np.linspace(L // 10, L - L // 10 - 1, 5).astype(np.int64)
        y = 10.0 + rng.standard_normal(nrec) + 0.5 * X0[:, 1] - 0.3 * X0[:, 2] + 0.7 * rng.standard_normal(n)[zidx]
        for b, j in zip([1.0, 0.8, 0.6, 0.5, 0.4], qtl):
            col = shard.fetch_col(lambda jj: device.extract_col(kb, n, jj, kblocked=True), n, int(j), "cuda")
            y = y + b * col.cpu().numpy().astype(np.float64)[zidx]
        sync()
        r = am.AM_resident(kb, tT, n, L, y, X0=X0, maxit=1, shard=shard, Z=zidx)
        sec = torch.tensor([r["seconds"][k] for k in sorted(r["seconds"])], dtype=torch.float64, device="cuda")
        dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        out["forward_iteration_with_Z_and_covariates"] = {
            "design": f"{nrec} records of {n} individuals (incidence matrix Z, one 1 per row), intercept + 2 fixed-effect "
                      "covariates (q = 3): EMMA's Z branches (R/emma_eigen_R_w_Z.R, R/emma_REMLE.R:78-131, R/emma_MLE.R:57-117) "
                      "through the secular solve, and the scan fed with H = ve I + vg Z K Z' (the Z-aware find_qtl of SURVEY.md "
                      "8(f) rank 4; the reference snapshot stops Z at EMMA)",
            "picked_1based": r["all_picked"], "planted_qtl_1based": [int(j) + 1 for j in qtl], "extBIC": r["extBIC"],
            "vc": {k: float(v) for k, v in r["vc"].items()}, "seconds_max_over_ranks": dict(zip(sorted(r["seconds"]), [round(x, 4) for x in sec.tolist()])),
            "secular": r["secular"]}
    del kb, tT
    return out


def run_forward_search(args, torch, dist, egd, n, L, Lg, c0, world, rank, img):
    """BASELINE config 3 as it is worded: the full multi-locus AM() forward search (<= 10 QTL) on the synthetic data set
    of SURVEY.md 8(d) (5 planted QTL), through the mirror of the R loop in eagleeverything_b200/am.py -- everything
    resident in HBM, the n x n algebra in the basis of eigen(K) (am.AM_resident).  At N > 1 the markers are sharded as in
    the timed step: partial M.Mt all-reduced, scans sharded, sharded pick, the picked column broadcast by its owner; the
    n x n algebra is replicated.  --search-host (N = 1) adds the route an R session would take today: every matrix
    crossing the host-level ABI as a host buffer (am.AM over api.*)."""
    import numpy as np
    from eagleeverything_b200 import am, api, device, synth
    qtl = np.linspace(L // 10, L - L // 10 - 1, 5).astype(np.int64)          # synth.phenotype's evenly spaced loci
    shard = egd.Shard(L, world, rank) if world > 1 else None
    t0 = time.perf_counter()
    kb = device.decode_kb(img, Lg + 1, n, Lg)[0]
    tT = device.transpose_kb(kb, n, Lg)
    torch.cuda.synchronize()
    t_stores = time.perf_counter() - t0
    rng = np.random.default_rng(synth.PHENO_SEED)
    y = 10.0 + rng.standard_normal(n)
    for b, j in zip([1.0, 0.8, 0.6, 0.5, 0.4], qtl):
        if shard is None:
            col = device.extract_col(kb, n, int(j), kblocked=True)
        else:
            col = shard.fetch_col(lambda jj: device.extract_col(kb, n, jj, kblocked=True), n, int(j), "cuda")
        y = y + b * col.cpu().numpy().astype(np.float64)
    # warm-up (untimed, like the W warm-up steps of the timed region): two iterations of the same search on the same
    # individuals and 4,096 markers -- library handles, lazily loaded kernels, and every workspace that depends on n at
    # its final size (a workspace that grows inside the timed search costs a cudaFree + cudaMalloc next to the memory
    # pools: dsyevd 1.5 - 2.0 s instead of 0.8, a secular solve 0.5 s instead of 0.01)
    Lw = 4096
    imgw = device.synth_ascii(n, Lw, GENO_SEED + 1)
    kbw = device.decode_kb(imgw, Lw + 1, n, Lw)[0]
    yw = np.random.default_rng(3).standard_normal(n) + device.extract_col(kbw, n, 17, kblocked=True).cpu().numpy()
    am.AM_resident(kbw, device.transpose_kb(kbw, n, Lw), n, Lw, yw, maxit=2)
    del kbw, imgw
    if world > 1:
        torch.cuda.synchronize(); dist.barrier()
    rr = am.AM_resident(kb, tT, n, L, y, maxit=args.search_maxit, shard=shard)
    del kb, tT
    torch.cuda.empty_cache()
    secs = rr["seconds"]
    if world > 1:   # the slowest rank defines the time; the picks must agree everywhere
        keys = sorted(secs)
        tt = torch.tensor([secs[k] for k in keys], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        secs = dict(zip(keys, [round(x, 4) for x in tt.tolist()]))
        mine = torch.tensor(rr["all_picked"] + [-1] * (args.search_maxit + 1 - len(rr["all_picked"])), dtype=torch.int64, device="cuda")
        allp = torch.empty(world * mine.numel(), dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(allp, mine)
        if not bool((allp.view(world, -1) == mine).all().item()):
            raise RuntimeError("ranks disagree on the selected loci")
    out = {"workload": f"AM() forward search, n={n}, L={L}, maxit={args.search_maxit}, 5 planted QTL", "n_gpus": world,
           "iterations": rr["iterations"], "selected_loci_1based": rr["selected"], "all_picked_1based": rr["all_picked"],
           "planted_qtl_1based": [int(j) + 1 for j in qtl],
           "planted_recovered": int(sum(1 for j in qtl if int(j) + 1 in rr["selected"])),
           "extBIC": [round(x, 6) for x in rr["extBIC"]], "seconds": secs, "secular": rr["secular"], "scan_route": rr.get("scan_route"), "scan_kernels": rr.get("scan_kernels"),
           "decode_transpose_s": round(t_stores, 4), "scans": len(rr["all_picked"]),
           "markers_per_s_whole_search": len(rr["all_picked"]) * L / secs["total_s"],
           "path": "am.AM_resident (mirror of R/AM.R:395-504): device-level C ABI; eigen(K) once, then per iteration a secular "
                   "solve for EMMA's eigenproblem, ONE n^3 product (int8 digit slices) for the scan's right-hand side, the "
                   "sharded scan and pick; EMMA's 1-D likelihood search on the host"}
    if args.search_host and world == 1:
        try:
            nbytes = n * (L + 1)
            img_h = torch.empty(nbytes + 64, dtype=torch.uint8, pin_memory=True)
            img_h[:nbytes].copy_(img[:nbytes]); img_h[nbytes:].zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            M = api.GenotypeStore.from_host_ptr(img_h.data_ptr(), n, L)
            Mt = M.transpose()
            t_load = time.perf_counter() - t0
            del img_h
            r = am.AM(am.ResidentGeno(M, Mt), y, maxit=args.search_maxit)
            M.free(); Mt.free()
            out["host_matrix_route"] = {
                "iterations": r["iterations"], "all_picked_1based": r["all_picked"], "seconds": r["seconds"],
                "upload_decode_transpose_s": round(t_load, 4), "same_sequence": r["all_picked"] == rr["all_picked"],
                "extBIC_max_rel_diff": float(max(abs(a - b) / abs(b) for a, b in zip(rr["extBIC"], r["extBIC"]))),
                "markers_per_s_whole_search": len(r["all_picked"]) * L / r["seconds"]["total_s"],
                "path": "am.AM over the host-level C ABI: every n x n matrix crosses as a (pageable) host buffer, as from R"}
        except Exception as ex:  # noqa: BLE001
            out["host_matrix_route"] = {"note": f"failed: {type(ex).__name__}: {ex}"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("EAGLE_BENCH_WORKLOAD", "c3"), choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--search", action="store_true", help="(default at N=1 for c2 / c3; kept for compatibility)")
    ap.add_argument("--no-search", action="store_true", help="skip the full multi-locus AM() forward search after the timed step")
    ap.add_argument("--search-host", action="store_true", help="also run the search with every matrix crossing the host-level ABI")
    ap.add_argument("--search-maxit", type=int, default=10)
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (shapes that leave no room for its copies)")
    ap.add_argument("--no-dropin", action="store_true", help="skip the file-based drop-in legs of the end-to-end measurement")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the in-run comparison with a single-GPU evaluation")
    ap.add_argument("--no-extras", action="store_true", help="N = 8: skip the one-step config 5 / config 4 legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results; --impl reference has none to write")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
