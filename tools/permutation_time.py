"""Times the permutation argument's product columns (h2sha_permutation_product) on one GPU:
python tools/permutation_time.py [cfg2 instances] [TestCircuit instances].

Workloads: config 2 ([64], 256 instances by default) and the reference's TestCircuit ([128, 128] with the output bytes bound to the
instance column, 64 instances), both at k = 17 (usable_rows = 2^17 - 6), two columns per chunk (cs.degree() = 4).  Next to each
figure: the z bytes written per second against the plain 256-bit store probe (h2sha_debug_store_probe) timed in the same run,
the rate of moved cells, and the one-off planning call (copy replay + upload)."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

n_cfg2 = int(sys.argv[1]) if len(sys.argv) > 1 else 256
n_tc = int(sys.argv[2]) if len(sys.argv) > 2 else 64
pkg = ge.load_package()
if os.environ.get("TUNE_LIB"):   # A/B: time another build of the engine (tools/build_ab.sh) with the same harness
    pkg.LIB_PATH = os.path.abspath(os.environ["TUNE_LIB"])
else:
    ge.build()
dev = torch.device("cuda", 0)
st = torch.cuda.current_stream(dev)
usable, m = (1 << 17) - 6, 2


def timed(fn, reps=5):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st); fn(); e1.record(st); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return min(ts[1:])


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"GPU: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")

probe_buf = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
probe_cfg = pkg.Sha256DynamicConfig.configure([64], device=0)
t_store = timed(lambda: probe_cfg.store_probe(probe_buf.data_ptr(), probe_buf.numel(), st.cuda_stream))
store_peak = probe_buf.numel() / t_store / 1e6
print(f"store probe: {probe_buf.numel() / 2**30:.0f} GiB in {t_store:.3f} ms = {store_peak:.0f} GB/s")
del probe_buf
probe_cfg.close()


def columns_of(lay, bind):
    nc = lay.n_spread_cols // 2
    cols = [(pkg.COL_GATE, i) for i in range(lay.n_gate_cols)] + [(pkg.COL_LOOKUP, i) for i in range(lay.n_lookup_cols)] + [(pkg.COL_FIXED, 0)]
    cols += [(pkg.COL_DENSE, i) for i in range(nc)] + [(pkg.COL_SPREAD, i) for i in range(nc)]
    return cols + ([(pkg.COL_INSTANCE, 0)] if bind else [])


def run(name, sizes, n, bind):
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0, build_shape=True)
    rng = np.random.default_rng(1)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, s - 8)), dtype=np.uint8)) for s in sizes] for _ in range(n)]
    res = cfg.digest_batch(msgs)
    cols = columns_of(cfg.layout, bind)
    mapping = cfg.permutation_mapping(cols, usable, columns_per_chunk=m, bind_output_bytes=bind)
    moved = int((mapping != np.stack(np.meshgrid(np.arange(len(cols)), np.arange(usable), indexing="ij"), -1).astype(np.uint32)).any(-1).sum())
    n_chunks = -(-len(cols) // m)
    z = torch.empty((n, n_chunks, usable + 1, 4), dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    dg = torch.from_numpy(res.digests).to(dev) if bind else None
    L = pkg.load_library()
    d, keep = cfg._perm_desc(cols, 1, m, bind, 0)
    beta = np.array([13, 17, 19, 23], dtype=np.uint64)
    gamma = np.array([29, 31, 37, 41], dtype=np.uint64)

    def call(k):
        rc = L.h2sha_permutation_product(cfg._h, k, C.byref(d), usable, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(),
                                         dg.data_ptr() if dg is not None else None, beta.ctypes.data, gamma.ctypes.data, z.data_ptr(),
                                         err.data_ptr(), st.cuda_stream)
        assert rc == 0, L.h2sha_last_error()

    t0 = time.perf_counter(); call(1); torch.cuda.synchronize(); t_plan = (time.perf_counter() - t0) * 1e3
    print(f"{name} {sizes}: {len(cols)} columns, {n_chunks} chunks of {m}, {moved} moved cells; first call (replay + upload) {t_plan:.0f} ms")
    for k in (max(1, n // 4), n):
        err.zero_()
        t = timed(lambda: call(k))
        zb = k * n_chunks * (usable + 1) * 32
        print(f"  {k} instances: {t:.3f} ms = {t / k * 1e3:.1f} us/instance, writes z {zb / t / 1e6:.0f} GB/s = {zb / t / 1e6 / store_peak:.2f} of the store probe, "
              f"{k * moved / t / 1e6:.2f} G moved cells/s, instances with z[U] != 1: {int(err.item()) // 5}")
    cfg.close()


run("cfg2", [64], n_cfg2, False)
run("TestCircuit", [128, 128], n_tc, True)
