import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import __graft_entry__ as ge
from oracle import oracle as O
pkg = ge.load_package()
rng = np.random.default_rng(3)
for m in (6144, 7808, 7872):
    t0 = time.perf_counter()
    try:
        cfg = pkg.Sha256DynamicConfig.configure([m], device=0)
    except pkg.EngineError as e:
        print(m, "create failed:", e); continue
    lay = cfg.layout
    msgs = [[bytes(rng.integers(0, 256, int(n), dtype=np.uint8))] for n in (0, m - 9, m // 2 + 3)]
    res = cfg.digest_batch(msgs)
    olay = O.Layout(lay.n_gate_cols, lay.gate_col_rows, lay.n_lookup_cols, lay.lookup_col_rows, lay.spread_rows)
    ref = O.batch(O.OracleConfig(max_variable_byte_sizes=(m,)), olay, msgs, None, want_cells=True, n_threads=3)
    ok = (res.digests == ref["digests"]).all() and (res.checksums == ref["checksums"]).all()
    for name in ("gate", "lookup", "spread"):
        ok = ok and bool((getattr(res, name).cpu().numpy().view(np.uint64) == ref[name]).all())
    v = cfg.check_batch(res, torch.from_numpy(res.digests).cuda().data_ptr())
    print(m, "blocks", lay.n_blocks, "gate cols", lay.n_gate_cols, "lookup cols", lay.n_lookup_cols, "cells", lay.cells_per_instance, "ok", bool(ok), v, f"{time.perf_counter()-t0:.1f}s", flush=True)
    cfg.close()
