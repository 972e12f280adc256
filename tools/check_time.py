"""Times the device constraint check on one GPU: python tools/check_time.py [workload] [instances] [repetitions].

The first h2sha_check_batch builds the check tables (shape plan + upload) and is timed on the host clock around the synchronising
call; the warm calls of h2sha_check_batch and h2sha_check_batch_per_instance are timed with CUDA events (median over the
repetitions).  Prints one JSON line.  TUNE_LIB=<library> times another build of the engine with the same harness; a build without
the per-instance call reports null for it."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
pkg = ge.load_package()
if os.environ.get("TUNE_LIB"):   # A/B: time another build of the engine (tools/build_ab.sh) with the same harness
    pkg.LIB_PATH = os.path.abspath(os.environ["TUNE_LIB"])
else:
    ge.build()
S = ge.load_package_module("synthetic")
w = S.WORKLOADS[wl]
cfg = pkg.Sha256DynamicConfig.configure(list(w.max_variable_byte_sizes), device=0)
blob, offs, lens = S.generate(w, 0, n)
res = cfg.digest_batch([[bytes(blob[int(o):int(o) + int(l)])] for o, l in zip(offs, lens)])
dig = torch.from_numpy(res.digests).cuda()
L = pkg.load_library()
dev = torch.device("cuda", 0)
st = torch.cuda.current_stream(dev)
v = np.zeros(5, dtype=np.uint64)
ptrs = (res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr())


def check_batch():
    rc = L.h2sha_check_batch(cfg._h, n, *ptrs, dig.data_ptr(), v.ctypes.data, st.cuda_stream)
    assert rc == 0, L.h2sha_last_error()


torch.cuda.synchronize()
t0 = time.perf_counter()
check_batch()   # builds the tables
first_ms = (time.perf_counter() - t0) * 1e3
assert int(v.sum()) == 0, v


def timed(fn):
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn()
        b.record(st)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(np.min(ms))


out = dict(workload=wl, instances=n, reps=reps, lib=os.path.basename(pkg.LIB_PATH), first_check_batch_ms=round(first_ms, 3))
out["check_batch_ms"] = [round(x, 4) for x in timed(check_batch)]
if hasattr(L, "h2sha_check_batch_per_instance"):
    cf = torch.empty((2, n, 5), dtype=torch.int32, device=dev)

    def per_instance():
        rc = L.h2sha_check_batch_per_instance(cfg._h, n, *ptrs, dig.data_ptr(), cf[0].data_ptr(), cf[1].data_ptr(), st.cuda_stream)
        assert rc == 0, L.h2sha_last_error()

    per_instance()
    out["per_instance_ms"] = [round(x, 4) for x in timed(per_instance)]
    assert int(cf[0].sum().item()) == 0
else:
    out["per_instance_ms"] = None
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
out["gpu"] = q
print(json.dumps(out))
cfg.close()
