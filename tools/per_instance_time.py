"""Times the per-instance-challenge calls against the shared-challenge calls on one GPU: python tools/per_instance_time.py [instances].

Workload: config 2 ([64], synthetic cfg2 messages), 256 instances by default, k = 17 (usable_rows = 2^17 - 6).  For the spread
permute, the range z, a spread z and the permutation z (7 columns, 2 per chunk) it times
  (a) the shared-challenge batch call,
  (b) the per-instance batch call (every instance its own random challenges),
  (c) the loop of single-instance shared calls a caller with independent proofs makes without (b),
each with CUDA events around the whole call (the loop ends in the same stream), one warm-up and the best of 5 repeats.  Then the
per-instance spread permute with num_bits_lookup = 16 (2^16-row tables) at 64 instances, split by a torch.profiler run into the
table build + sort kernels and the scan + fill kernels; its multiplicities are a synthetic histogram (uniform limbs, the rest on
row 0), since the engine does not count 16-bit spread multiplicities."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402
from oracle import oracle as O  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
n16 = 64
pkg = ge.load_package()
ge.build()
S = ge.load_package_module("synthetic")
L = pkg.load_library()
dev = torch.device("cuda", 0)
st = torch.cuda.current_stream(dev)
usable = (1 << 17) - 6
REPS = 6   # one warm-up + 5 timed


def timed(fn):
    ts = []
    for _ in range(REPS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); fn(); e1.record(st); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts[1:])


def ok(rc):
    assert rc == 0, L.h2sha_last_error().decode()


def rows(rng, k):
    return np.ascontiguousarray(np.stack([O.int_to_mont(int.from_bytes(rng.bytes(32), "little") % O.P) for _ in range(k)]))


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"GPU: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")
print(f"workload: cfg2, {n} instances, usable_rows = {usable}; best of 5 after one warm-up; (c) = {n} single-instance shared calls in a loop")

w = S.WORKLOADS["cfg2"]
cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=0, build_shape=True)
blob, offs, lens = S.generate(w, 0, n)
res = cfg.digest_batch([[bytes(blob[int(o):int(o) + int(l)])] for o, l in zip(offs, lens)])
info = cfg.lookup_info()
n_r = info["n_range_lookups"]
mult, bad = cfg.lookup_multiplicities(res, usable)
assert bad == 0
rng = np.random.default_rng(7)
thetas, betas, gammas = rows(rng, n), rows(rng, n), rows(rng, n)
th1, be1, ga1 = thetas[0].copy(), betas[0].copy(), gammas[0].copy()
a = torch.empty((n, usable, 4), dtype=torch.int64, device=dev)
s = torch.empty((n, usable, 4), dtype=torch.int64, device=dev)
z = torch.empty((n, usable + 1, 4), dtype=torch.int64, device=dev)
err = torch.zeros(n, dtype=torch.int32, device=dev)
mw, cell, ucell = info["mult_words_per_instance"], usable * 4 * 8, (usable + 1) * 4 * 8
sp_l = n_r   # the first spread lookup


def report(name, ta, tb, tc):
    print(f"{name:<28} (a) shared {ta:9.3f} ms | (b) per-instance {tb:9.3f} ms | (c) loop {tc:9.3f} ms | (b)/(a) {tb / ta:5.2f} | (c)/(b) {tc / tb:6.1f}")


# spread permute
ta = timed(lambda: ok(L.h2sha_permute_lookup(cfg._h, n, sp_l, mult.data_ptr(), usable, th1.ctypes.data, a.data_ptr(), s.data_ptr(), None, st.cuda_stream)))
tb = timed(lambda: ok(L.h2sha_permute_lookup_per_instance(cfg._h, n, sp_l, mult.data_ptr(), usable, thetas.ctypes.data, a.data_ptr(), s.data_ptr(),
                                                          err.data_ptr(), st.cuda_stream)))


def loop_permute():
    for i in range(n):
        ok(L.h2sha_permute_lookup(cfg._h, 1, sp_l, mult.data_ptr() + i * mw * 4, usable, thetas[i].ctypes.data, a.data_ptr() + i * cell,
                                  s.data_ptr() + i * cell, None, st.cuda_stream))


tc = timed(loop_permute)
report(f"spread permute (lookup {sp_l})", ta, tb, tc)
assert not err.any()


# lookup products: the per-instance A', S' of the spread lookup are in a, s; the range lookup's are permuted first
def product_times(l, th_rows):
    thp = None if th_rows is None else th1.ctypes.data
    ta = timed(lambda: ok(L.h2sha_lookup_product(cfg._h, n, l, res.lookup.data_ptr(), res.spread.data_ptr(), a.data_ptr(), s.data_ptr(), usable, thp,
                                                 be1.ctypes.data, ga1.ctypes.data, z.data_ptr(), None, st.cuda_stream)))
    err.zero_()
    tb = timed(lambda: ok(L.h2sha_lookup_product_per_instance(cfg._h, n, l, res.lookup.data_ptr(), res.spread.data_ptr(), a.data_ptr(), s.data_ptr(), usable,
                                                              None if th_rows is None else th_rows.ctypes.data, betas.ctypes.data, gammas.ctypes.data,
                                                              z.data_ptr(), err.data_ptr(), st.cuda_stream)))
    assert not err.any(), "per-instance z[U] != 1"
    li, si = res.lookup.stride(0) * 8, res.spread.stride(0) * 8

    def loop():
        for i in range(n):
            ok(L.h2sha_lookup_product(cfg._h, 1, l, res.lookup.data_ptr() + i * li, res.spread.data_ptr() + i * si, a.data_ptr() + i * cell,
                                      s.data_ptr() + i * cell, usable, None if th_rows is None else th_rows[i].ctypes.data, betas[i].ctypes.data,
                                      gammas[i].ctypes.data, z.data_ptr() + i * ucell, None, st.cuda_stream))

    return ta, tb, timed(loop)


report(f"spread z (lookup {sp_l})", *product_times(sp_l, thetas))
ok(L.h2sha_permute_lookup(cfg._h, n, 0, mult.data_ptr(), usable, None, a.data_ptr(), s.data_ptr(), None, st.cuda_stream))
report("range z (lookup 0)", *product_times(0, None))
del a, s, z

# permutation product
lay = cfg.layout
nc = lay.n_spread_cols // 2
cols = [(pkg.COL_GATE, i) for i in range(lay.n_gate_cols)] + [(pkg.COL_LOOKUP, i) for i in range(lay.n_lookup_cols)] + [(pkg.COL_FIXED, 0)]
cols += [(pkg.COL_DENSE, i) for i in range(nc)] + [(pkg.COL_SPREAD, i) for i in range(nc)]
m = 2
n_chunks = -(-len(cols) // m)
d, keep = cfg._perm_desc(cols, 1, m, False, 0)
zp = torch.empty((n, n_chunks, usable + 1, 4), dtype=torch.int64, device=dev)
g, lk, sp = res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr()
gi, li, si = res.gate.stride(0) * 8, res.lookup.stride(0) * 8, res.spread.stride(0) * 8
ok(L.h2sha_permutation_product(cfg._h, 1, C.byref(d), usable, g, lk, sp, None, be1.ctypes.data, ga1.ctypes.data, zp.data_ptr(), None, st.cuda_stream))   # plans the moved cells
ta = timed(lambda: ok(L.h2sha_permutation_product(cfg._h, n, C.byref(d), usable, g, lk, sp, None, be1.ctypes.data, ga1.ctypes.data, zp.data_ptr(), None,
                                                  st.cuda_stream)))
err.zero_()
tb = timed(lambda: ok(L.h2sha_permutation_product_per_instance(cfg._h, n, C.byref(d), usable, g, lk, sp, None, betas.ctypes.data, gammas.ctypes.data,
                                                               zp.data_ptr(), err.data_ptr(), st.cuda_stream)))
assert not err.any(), "per-instance z[U] != 1"


def loop_perm():
    for i in range(n):
        ok(L.h2sha_permutation_product(cfg._h, 1, C.byref(d), usable, g + i * gi, lk + i * li, sp + i * si, None, betas[i].ctypes.data, gammas[i].ctypes.data,
                                       zp.data_ptr() + i * n_chunks * ucell, None, st.cuda_stream))


report(f"permutation z ({len(cols)} cols, {m}/chunk)", ta, tb, timed(loop_perm))
del zp
cfg.close()


# 16-bit limbs: per-instance spread permute, table build + sort vs scan + fill
def kernel_split(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tab = scan = 0.0
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
        if "k_permute_scan" in ev.key or "k_permute_fill" in ev.key:
            scan += us
        elif "k_spread_" in ev.key or "cub" in ev.key.lower() or "Segmented" in ev.key:
            tab += us
    return tab / 1e3, scan / 1e3


cfg16 = pkg.Sha256DynamicConfig.configure([64], device=0, num_bits_lookup=16)
info16 = cfg16.lookup_info()
n_r16 = info16["n_range_lookups"]
mult16 = np.zeros((n16, info16["mult_words_per_instance"]), dtype=np.int32)
n_limb = cfg16.layout.n_spread_limbs // info16["n_spread_lookups"]
for i in range(n16):
    h = np.bincount(rng.integers(0, 1 << 16, n_limb), minlength=1 << 16)
    h[0] += usable - n_limb
    mult16[i, n_r16 << 16:(n_r16 + 1) << 16] = h
mult16 = torch.from_numpy(mult16).to(dev)
th16 = rows(rng, n16)
a = torch.empty((n16, usable, 4), dtype=torch.int64, device=dev)
s = torch.empty((n16, usable, 4), dtype=torch.int64, device=dev)
err16 = torch.zeros(n16, dtype=torch.int32, device=dev)
call16 = lambda: ok(L.h2sha_permute_lookup_per_instance(cfg16._h, n16, n_r16, mult16.data_ptr(), usable, th16.ctypes.data, a.data_ptr(), s.data_ptr(),
                                                        err16.data_ptr(), st.cuda_stream))
t16 = timed(call16)
assert not err16.any()
ta16 = timed(lambda: ok(L.h2sha_permute_lookup(cfg16._h, n16, n_r16, mult16.data_ptr(), usable, th16[0].ctypes.data, a.data_ptr(), s.data_ptr(), None,
                                               st.cuda_stream)))
tab, scan = kernel_split(call16)
print(f"16-bit spread permute, {n16} instances: (b) per-instance {t16:.3f} ms, (a) shared {ta16:.3f} ms; "
      f"kernels (one profiled call): table build + sort {tab:.3f} ms, scan + fill {scan:.3f} ms")
cfg16.close()
