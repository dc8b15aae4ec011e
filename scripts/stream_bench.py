"""Streamed stores against resident ones at a given shape (default BASELINE config 3: n = 10,000, L = 1,000,000), one GPU.

The genotypes come from eg_dev_synth_ascii and are packed to a SNP-major .bed image on the device.  For the resident stores
(eg_store_from_host_bed) and the streamed ones (eg_store_stream_host_bed from page-locked memory, eg_store_stream_bed from a
file in a temporary directory, read from the page cache), with the same seeded S, V and a:
  * per-call wall times of M.Mt (eg_store_mmt) and of the scan (eg_store_a_and_vara), and scan markers/s;
  * the scan kernel's device time (eg_last_scan_kernel: the sum over the pieces for a streamed scan);
  * hashes of K, a and var(a), which must be equal across the routes;
  * the card's name and power limit, read in the same run.
EAGLE_INGEST_PIECE_BYTES sets the piece size of the streamed routes; --pieces runs several sizes in one call.  Every route
runs one untimed call first, then --reps timed calls.

--large: a set larger than HBM (default n = 20,000 x L = 10,000,000: a 50 GB .bed, 200 GB per int8 orientation).  The .bed
image is built in host memory range by range on the device and never exists there whole.  One streamed M.Mt and one
streamed scan run from it; K must equal the sum of the resident M.Mt of five equal SNP ranges, and a / var(a) of the first
and last --check-markers markers must equal resident scans of those ranges, bit for bit.  Host and device memory are
checked first; when either is short, a "not run" record with the reason is written instead.
Usage: python scripts/stream_bench.py [--n N] [--L L] [--reps R] [--pieces MB,MB,..] [--large] [--out FILE]"""
import argparse
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from eagleeverything_b200 import api, device, synth

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=None)
ap.add_argument("--L", type=int, default=None)
ap.add_argument("--large", action="store_true", help="the larger-than-HBM case (default n = 20,000, L = 10,000,000)")
ap.add_argument("--check-markers", type=int, default=1000000)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--pieces", default="256", help="piece sizes in MB of .bed bytes, comma-separated")
ap.add_argument("--out", default=None)
args = ap.parse_args()
n = args.n or (20000 if args.large else 10000)
L = args.L or (10000000 if args.large else 1000000)
bpr = (n + 3) // 4
lines = []


def emit(**rec):
    lines.append(rec)
    print(json.dumps(rec), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def write_out():
    if args.out:
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


def pack_bed(j0, j1):
    """SNPs [j0, j1) of the synthetic genotypes as .bed rows ((j1 - j0) x bpr uint8 on the device)."""
    img = device.synth_ascii(n, j1 - j0, synth.GENO_SEED, col_offset=j0, n_total=n)
    c = img[: n * (j1 - j0 + 1)].view(n, j1 - j0 + 1)[:, : j1 - j0] - ord("0")   # codes 0 / 1 / 2
    v = torch.zeros((j1 - j0, 4 * bpr), dtype=torch.uint8, device="cuda")
    v[:, :n] = (c + (c > 0).to(torch.uint8)).t()                                      # .bed values 0 / 2 / 3
    v = v.view(j1 - j0, bpr, 4)
    return v[:, :, 0] | (v[:, :, 1] << 2) | (v[:, :, 2] << 4) | (v[:, :, 3] << 6)


def mem_available():
    with open("/proc/meminfo") as f:
        for ln in f:
            if ln.startswith("MemAvailable:"):
                return int(ln.split()[1]) * 1024
    return 0


def scan_kernel():
    ms, ops = C.c_double(), C.c_double()
    lib.eg_last_scan_kernel(C.byref(ms), C.byref(ops))
    return ms.value, ops.value


lib = device.init(0)
emit(what="card", n=n, L=L, **card())


def large():
    bed_bytes = 3 + L * bpr
    host_need = bed_bytes + 12 * 8 * n * n + 64 * L + (8 << 30)   # image, S / V / K copies and scratch, outputs, slack
    free_dev, total_dev = torch.cuda.mem_get_info()
    ranges = 5
    w = -(-L // ranges)
    # the largest resident check store and its E2M1 copy for M.Mt, the n x n buffers, the pieces
    dev_need = n * w * 3 // 2 + 5 * 4 * n * n + (16 << 30)
    emit(what="large_memory", host_available=mem_available(), host_needed=host_need, device_free=free_dev,
         device_total=total_dev, device_needed=dev_need, bed_bytes=bed_bytes, int8_bytes_per_orientation=n * L)
    if mem_available() < host_need:
        emit(what="large_not_run", reason=f"host memory: {mem_available() / 1e9:.1f} GB available, {host_need / 1e9:.1f} GB "
                                          f"needed for the {bed_bytes / 1e9:.1f} GB .bed image and the n x n matrices")
        return
    if free_dev < dev_need:
        emit(what="large_not_run", reason=f"device memory: {free_dev / 1e9:.1f} GB free, {dev_need / 1e9:.1f} GB needed for the "
                                          f"resident check stores (the GPU is shared; it is not filled on purpose)")
        return
    t0 = time.perf_counter()
    h = np.empty(bed_bytes, dtype=np.uint8)
    h[:3] = (0x6C, 0x1B, 0x01)
    step = max(128, (1 << 30) // n // 128 * 128)
    for j0 in range(0, L, step):
        j1 = min(L, j0 + step)
        torch.from_numpy(h[3 + j0 * bpr: 3 + j1 * bpr]).view(j1 - j0, bpr).copy_(pack_bed(j0, j1))
    torch.cuda.empty_cache()
    emit(what="large_image_built", seconds=round(time.perf_counter() - t0, 1), host="pageable")
    S, V, a = synth.scan_inputs(n)
    Ms = api.GenotypeStore.stream_host_bed(h, n, L)
    Mts = api.GenotypeStore.stream_host_bed(h, n, L, kblocked=False)
    t0 = time.perf_counter()
    K = Ms.mmt()
    t_mmt = time.perf_counter() - t0
    t0 = time.perf_counter()
    av, vv = Mts.a_and_vara(S, V, a)
    t_scan = time.perf_counter() - t0
    k_ms, k_ops = scan_kernel()
    tm = api.last_timing()
    pieces = -(-L // max(128, int(os.environ.get("EAGLE_INGEST_PIECE_BYTES", 256 << 20)) // bpr // 128 * 128))
    emit(what="large_streamed", pieces=pieces, mmt_s=round(t_mmt, 2), mmt_syrk_ms=round(tm["syrk_ms"], 1),
         scan_s=round(t_scan, 2), scan_prepare_ms=round(tm["prepare_ms"], 1), scan_markers_ms=round(tm["scan_ms"], 1),
         scan_kernel_ms_sum=round(k_ms, 1), scan_kernel_pops=round(k_ops / k_ms / 1e12, 3) if k_ms else None,
         scan_markers_per_s=round(L / t_scan), K=sha(K), a=sha(av), vara=sha(vv))
    Ms.free()
    Mts.free()
    Ksum = np.zeros((n, n))
    for r in range(ranges):
        r0, r1 = r * w, min(L, (r + 1) * w)
        R = api.GenotypeStore.from_host_bed(h, n, L, r0, r1)
        Ksum += R.mmt()
        R.free()
    emit(what="large_check_mmt", ranges=ranges, equal=bool(np.array_equal(K, Ksum)))
    cm = min(args.check_markers, L)
    for r0, r1 in ((0, cm), (L - cm, L)):
        R = api.GenotypeStore.from_host_bed(h, n, L, r0, r1, kblocked=False)
        ra, rv = R.a_and_vara(S, V, a)
        R.free()
        emit(what="large_check_scan", markers=[r0, r1], a_equal=bool(np.array_equal(ra, av[r0:r1])),
             vara_equal=bool(np.array_equal(rv, vv[r0:r1])))


if args.large:
    try:
        large()
    finally:
        emit(what="card_after", **card())
        write_out()
    sys.exit(0)

# ---------------------------------------------------------------- the .bed image, built on the device, kept page-locked
img = device.synth_ascii(n, L, synth.GENO_SEED)
bed = torch.empty(3 + L * bpr, dtype=torch.uint8, device="cuda")
bed[:3] = torch.tensor([0x6C, 0x1B, 0x01], dtype=torch.uint8)
rows = bed[3:].view(L, bpr)
lut = torch.tensor([0, 2, 3], dtype=torch.uint8, device="cuda")
M = img[: n * (L + 1)].view(n, L + 1)
step = max(1, (256 << 20) // n)
for j0 in range(0, L, step):
    j1 = min(L, j0 + step)
    v = torch.zeros((j1 - j0, 4 * bpr), dtype=torch.uint8, device="cuda")
    v[:, :n] = lut[(M[:, j0:j1] - ord("0")).long()].t()
    v = v.view(j1 - j0, bpr, 4)
    rows[j0:j1] = v[:, :, 0] | (v[:, :, 1] << 2) | (v[:, :, 2] << 4) | (v[:, :, 3] << 6)
    del v
h_bed = torch.empty(bed.numel(), dtype=torch.uint8, pin_memory=True)
h_bed.copy_(bed)
del bed, img, M, rows
torch.cuda.empty_cache()
S, V, a = synth.scan_inputs(n)


def run(route, Ms, Mts, **extra):
    t0 = time.perf_counter()   # untimed first call (module loads, workspace allocations)
    Ms.mmt()
    Mts.a_and_vara(S, V, a)
    first = (time.perf_counter() - t0) * 1e3
    t_mmt, t_scan, k_scan = [], [], []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        K = Ms.mmt()
        t_mmt.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        av, vv = Mts.a_and_vara(S, V, a)
        t_scan.append((time.perf_counter() - t0) * 1e3)
        k_scan.append(scan_kernel()[0])
    tsq = av * av / vv
    pick = int(np.nanargmax(tsq))
    best = min(t_scan)
    timing = api.last_timing()
    timing.pop("h2d_decode_ms")   # set by uploads only: the resident stores' upload, not a streamed call
    emit(what="route", route=route, first_call_ms=round(first, 1), mmt_ms=[round(t, 1) for t in t_mmt],
         scan_ms=[round(t, 1) for t in t_scan], scan_kernel_ms=[round(t, 1) for t in k_scan],
         scan_markers_per_s=round(L / best * 1e3), timing=timing,
         K=sha(K), a=sha(av), vara=sha(vv), pick=pick, tsq=float(tsq[pick]), **extra)


tmpdir = tempfile.mkdtemp(prefix="stream_bench_")
try:
    Mr = api.GenotypeStore.from_host_bed(h_bed, n, L, kblocked=True)
    Tr = api.GenotypeStore.from_host_bed(h_bed, n, L, kblocked=False)
    os.environ["EAGLE_KEEP_PRODUCT"] = "0"   # contract on every M.Mt call, as the streamed store must
    run("resident", Mr, Tr)
    Mr.free()
    Tr.free()
    path = os.path.join(tmpdir, "g.bed")
    h_bed.numpy().tofile(path)
    for mb in [int(x) for x in args.pieces.split(",")]:
        os.environ["EAGLE_INGEST_PIECE_BYTES"] = str(mb << 20)
        pieces = -(-L // max(128, (mb << 20) // bpr // 128 * 128))
        run("streamed_pinned", api.GenotypeStore.stream_host_bed(h_bed, n, L), api.GenotypeStore.stream_host_bed(h_bed, n, L, kblocked=False),
            piece_MB=mb, pieces=pieces)
        run("streamed_file_page_cache", api.GenotypeStore.stream_bed(path, n, L), api.GenotypeStore.stream_bed(path, n, L, kblocked=False),
            piece_MB=mb, pieces=pieces)
finally:
    shutil.rmtree(tmpdir, ignore_errors=True)
emit(what="card_after", **card())
write_out()
