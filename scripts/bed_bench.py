"""PLINK .bed input at a given shape (default BASELINE config 3: n = 10,000, L = 1,000,000) on one GPU.

Genotypes from eg_dev_synth_ascii, packed to a SNP-major .bed image on the device with torch ops.  Reports, as JSON lines:
  * eg_dev_decode_bed for both layouts: CUDA events over repeated launches (the 2.5 GB input and the 10 GB store are far
    larger than L2), GB/s of algorithmic traffic (.bed bytes read + store bytes written), next to a device-to-device copy
    and the ASCII decoder measured in the same run;
  * eg_store_from_host_bed from a page-locked buffer, eg_store_from_bed from a file (written to a temporary directory that
    is deleted at the end, so read from the page cache), against eg_store_from_host_ascii from a page-locked buffer
    (which also accumulates M.Mt under its copy);
  * hashes of K, a, var(a) and the picked marker for every route;
  * the card's name and power limit, read in the same run.
Usage: python scripts/bed_bench.py [--n N] [--L L] [--reps R] [--out FILE]"""
import argparse
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
ap.add_argument("--n", type=int, default=10000)
ap.add_argument("--L", type=int, default=1000000)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--host-reps", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()
n, L = args.n, args.L
bpr = (n + 3) // 4
lines = []


def emit(**rec):
    lines.append(rec)
    print(json.dumps(rec), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


lib = device.init(0)
emit(what="card", n=n, L=L, **card())

# ---------------------------------------------------------------- inputs: ASCII image, and the same genotypes as .bed
img = device.synth_ascii(n, L, synth.GENO_SEED)                     # n x (L + 1) bytes + 64
bed = torch.empty(3 + L * bpr, dtype=torch.uint8, device="cuda")
bed[:3] = torch.tensor([0x6C, 0x1B, 0x01], dtype=torch.uint8)
rows = bed[3:].view(L, bpr)
lut = torch.tensor([0, 2, 3], dtype=torch.uint8, device="cuda")    # codes AA / AB / BB -> .bed values
M = img[: n * (L + 1)].view(n, L + 1)
step = max(1, (256 << 20) // n)
for j0 in range(0, L, step):
    j1 = min(L, j0 + step)
    v = torch.zeros((j1 - j0, 4 * bpr), dtype=torch.uint8, device="cuda")
    v[:, :n] = lut[(M[:, j0:j1] - ord("0")).long()].t()
    v = v.view(j1 - j0, bpr, 4)
    rows[j0:j1] = v[:, :, 0] | (v[:, :, 1] << 2) | (v[:, :, 2] << 4) | (v[:, :, 3] << 6)
    del v
torch.cuda.synchronize()

# ---------------------------------------------------------------- kernels
kb = torch.empty(((L + 127) // 128, n, 128), dtype=torch.int8, device="cuda")
rm = torch.empty((L, device.store_pitch(n)), dtype=torch.int8, device="cuda")
cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
bed_in = L * bpr
for name, out in (("kblocked", kb), ("rowmajor", rm)):
    ms = events(lambda: device.decode_bed(bed, n, L, kblocked=name == "kblocked", out=out, missing=cnt), args.reps)
    moved = bed_in + out.numel()
    emit(what="decode_bed", layout=name, ms=round(ms, 4), bytes_read=bed_in, bytes_written=out.numel(),
         GBps=round(moved / ms / 1e6, 1))
kb_ref = torch.empty_like(kb)
err = torch.zeros(4, dtype=torch.int32, device="cuda")
ms = events(lambda: device.decode_kb(img, L + 1, n, L, out=kb_ref, err=err), args.reps)
emit(what="decode_kb_ascii", ms=round(ms, 4), GBps=round((n * (L + 1) + kb_ref.numel()) / ms / 1e6, 1))
emit(what="kblocked_store_equals_ascii_decode", equal=bool(torch.equal(kb, kb_ref)), missing_counted=int(cnt.item()))
ms = events(lambda: kb_ref.copy_(kb), args.reps)
emit(what="d2d_copy", ms=round(ms, 4), GBps=round(2 * kb.numel() / ms / 1e6, 1))
del kb, rm, kb_ref
torch.cuda.empty_cache()

# ---------------------------------------------------------------- host routes
h_bed = torch.empty(bed.numel(), dtype=torch.uint8, pin_memory=True)
h_bed.copy_(bed)
h_img = torch.empty(img.numel(), dtype=torch.uint8, pin_memory=True)
h_img.copy_(img)
del bed, img, M, rows
torch.cuda.empty_cache()
tmpdir = tempfile.mkdtemp(prefix="bed_bench_")
S, V, a = synth.scan_inputs(n)


def timed(make):
    ts, s = [], None
    for _ in range(args.host_reps):
        if s is not None:
            s.free()
        t0 = time.perf_counter()
        s = make()
        ts.append((time.perf_counter() - t0) * 1e3)
    return s, ts


def results(route, Ms, Mts, **ms):
    K = Ms.mmt()
    av, vv = Mts.a_and_vara(S, V, a)
    tsq = av * av / vv
    pick = int(np.nanargmax(tsq))
    emit(what="route", route=route, **{k: [round(t, 1) for t in v] for k, v in ms.items()},
         K=sha(K), a=sha(av), vara=sha(vv), pick=pick, tsq=float(tsq[pick]), n_missing=getattr(Ms, "n_missing", None))
    Ms.free()
    Mts.free()


try:
    Mb, tb = timed(lambda: api.GenotypeStore.from_host_bed(h_bed, n, L, kblocked=True))
    Tb, tt = timed(lambda: api.GenotypeStore.from_host_bed(h_bed, n, L, kblocked=False))
    results("bed_pinned", Mb, Tb, M_store_ms=tb, Mt_store_ms=tt)
    path = os.path.join(tmpdir, "g.bed")
    h_bed.numpy().tofile(path)
    Mf, tf = timed(lambda: api.GenotypeStore.from_bed(path, n, L, kblocked=True))
    Tf, tft = timed(lambda: api.GenotypeStore.from_bed(path, n, L, kblocked=False))
    results("bed_file_page_cache", Mf, Tf, M_store_ms=tf, Mt_store_ms=tft)
    os.remove(path)
    Ma, ta = timed(lambda: api.GenotypeStore.from_host_ptr(h_img.data_ptr(), n, L))
    t0 = time.perf_counter()
    Ta = Ma.transpose()
    t_tr = (time.perf_counter() - t0) * 1e3
    results("ascii_pinned", Ma, Ta, M_store_ms=ta, Mt_transpose_ms=[t_tr])
finally:
    shutil.rmtree(tmpdir, ignore_errors=True)
emit(what="card_after", **card())
if args.out:
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
