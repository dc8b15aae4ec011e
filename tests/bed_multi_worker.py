"""Worker of tests/test_bed.py::test_sharded_bed_store_equals_one_gpu (a fresh interpreter: the multi-GPU set is process-wide
state): stores read from a .bed file on an eg_init_multi set against the same calls on one GPU, bit for bit."""
import faulthandler
faulthandler.dump_traceback_later(int(__import__("os").environ.get("EAGLE_TEST_WATCHDOG_S", "240")), exit=True)
import os, sys, tempfile
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from eagleeverything_b200 import _lib, api, synth
from plink_bed import write_bed
ngpu, n, L = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3])
rng = np.random.default_rng(n + L)
G = rng.integers(0, 3, (n, L), dtype=np.uint8)
miss = rng.random((n, L)) < 0.02
S, V, a = synth.scan_inputs(n)
d = tempfile.mkdtemp()
bed = os.path.join(d, "g.bed")
with open(bed, "wb") as f:
    f.write(write_bed(G, missing=miss))
def run():
    out = {}
    for snp0, snp1, tag in ((0, L, ""), (77, L - 300, "shard")):
        M = api.GenotypeStore.from_bed(bed, n, L, snp0, snp1, kblocked=True)
        Mt = api.GenotypeStore.from_bed(bed, n, L, snp0, snp1, kblocked=False)
        w = snp1 - snp0
        out["K" + tag] = M.mmt([3, w - 2])
        out["a" + tag], out["v" + tag] = Mt.a_and_vara(S, V, a, [7])
        out["cols" + tag] = np.stack([M.extract_col(j) for j in (0, 127, 128, w // 2, w - 1)])
        out["miss" + tag] = np.array([M.n_missing, Mt.n_missing])
        M.free(); Mt.free()
    return out
_lib.check(_lib.require_gpu().eg_init(0))
one = run()
assert api.init_multi(ngpu) == ngpu
many = run()
for k in one:
    assert np.array_equal(one[k], many[k]), k
assert one["miss"][0] == int(miss.sum())
api.shutdown()
print("BED_MULTI_OK", ngpu)
