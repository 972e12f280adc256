"""Times the lookup pre-work calls on one GPU: python tools/prework_time.py [workload] [instances] [permute instances].

After each permutation, the grand-product column z of the same instances (h2sha_lookup_product) at n_perm / 4 and n_perm
instances, against the integer-instruction probe (h2sha_debug_int_probe) timed in the same run."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
n_perm = int(sys.argv[3]) if len(sys.argv) > 3 else 256
pkg = ge.load_package()
if os.environ.get("TUNE_LIB"):   # A/B: time another build of the engine (tools/build_ab.sh) with the same harness
    pkg.LIB_PATH = os.path.abspath(os.environ["TUNE_LIB"])
else:
    ge.build()
S = ge.load_package_module("synthetic")
w = S.WORKLOADS[wl]
cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=0)
lay = cfg.layout
blob, offs, lens = S.generate(w, 0, n)
msgs = [[bytes(blob[int(o):int(o) + int(l)])] for o, l in zip(offs, lens)]
res = cfg.digest_batch(msgs)
usable = (1 << 17) - 6
info = cfg.lookup_info()
L = pkg.load_library()
dev = torch.device("cuda", 0)
st = torch.cuda.current_stream(dev)
mult = torch.empty((n, info["mult_words_per_instance"]), dtype=torch.int32, device=dev)
bad = torch.zeros(1, dtype=torch.int32, device=dev)
a = torch.empty((n_perm, usable, 4), dtype=torch.int64, device=dev)
s = torch.empty((n_perm, usable, 4), dtype=torch.int64, device=dev)


def timed(fn, reps=5):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); fn(); e1.record(st); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts[1:])


t_m = timed(lambda: L.h2sha_lookup_multiplicities(cfg._h, n, res.lookup.data_ptr(), res.spread.data_ptr(), usable, mult.data_ptr(), bad.data_ptr(), st.cuda_stream))
print(f"multiplicities: {n} instances {t_m:.3f} ms, reads {n * (lay.n_lookup_cells + 2 * lay.n_spread_limbs) * 32 / t_m / 1e6:.0f} GB/s, bad={int(bad.item())}")

# Thread-level instructions per row of k_product_tiles<LookupRows> + k_product_fill<LookupRows>, counted once from `cuobjdump -sass` of
# the sm_100a build: a Montgomery product (mont_mul_dev) with its loads and additions is ~516 SASS instructions (k_product_fill: 35 296
# for its 8 rows a thread, 68 products); a row costs 4 + 10/8 products in k_product_tiles and 7 + 1/8 in k_product_fill, one more in
# each pass for the theta compression of a spread lookup.
INST_PER_ROW = {"range": 6400, "spread": 7400}

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"GPU: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")
scratch = torch.zeros(torch.cuda.get_device_properties(0).multi_processor_count * 8 * 256, dtype=torch.int32, device=dev)
probe_iters = 4096
probe_inst = [0]


def _probe():
    probe_inst[0] = cfg.int_probe(scratch.data_ptr(), probe_iters, st.cuda_stream)


t_probe = timed(_probe)
probe_rate = probe_inst[0] / t_probe / 1e9
print(f"int probe: {probe_inst[0] / 1e9:.2f} G thread instructions in {t_probe:.3f} ms = {probe_rate:.1f} T inst/s")
z = torch.empty((n_perm, usable + 1, 4), dtype=torch.int64, device=dev)
zerr = torch.zeros(1, dtype=torch.int32, device=dev)
theta = np.array([3, 5, 7, 11], dtype=np.uint64)
beta = np.array([13, 17, 19, 23], dtype=np.uint64)
gamma = np.array([29, 31, 37, 41], dtype=np.uint64)
for l in range(info["n_range_lookups"] + info["n_spread_lookups"]):
    th = theta.ctypes.data if l >= info["n_range_lookups"] else None
    t_p = timed(lambda: L.h2sha_permute_lookup(cfg._h, n_perm, l, mult.data_ptr(), usable, th, a.data_ptr(), s.data_ptr(), None, st.cuda_stream))
    print(f"permute lookup {l}: {n_perm} instances {t_p:.3f} ms, writes {n_perm * usable * 64 / t_p / 1e6:.0f} GB/s")
    kind = "range" if l < info["n_range_lookups"] else "spread"
    for m in (n_perm // 4, n_perm):
        zerr.zero_()
        t_z = timed(lambda: L.h2sha_lookup_product(cfg._h, m, l, res.lookup.data_ptr(), res.spread.data_ptr(), a.data_ptr(), s.data_ptr(), usable, th,
                                                   beta.ctypes.data, gamma.ctypes.data, z.data_ptr(), zerr.data_ptr(), st.cuda_stream))
        rows = m * usable
        rate = rows * INST_PER_ROW[kind] / t_z / 1e9
        print(f"lookup product {l} ({kind}): {m} instances {t_z:.3f} ms, {rows / t_z / 1e6:.2f} G rows/s, writes z {rows * 32 / t_z / 1e6:.0f} GB/s, "
              f"~{rate:.1f} T inst/s = {rate / probe_rate:.2f} of the int probe, instances with z[U] != 1: {int(zerr.item()) // 5}")
