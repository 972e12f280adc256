"""h2sha_permutation_product over a batch split into several launches of instances (H2SHA_TUNE pmchunk) gives the columns of
one launch, bit for bit: the launches share the tile workspace, and each starts at its own instance."""
import numpy as np
import pytest

from oracle import oracle as O


@pytest.mark.gpu
def test_chunked_instances_give_the_same_columns(pkg, monkeypatch):
    import torch
    cfg = pkg.Sha256DynamicConfig.configure([128, 128], device=0, build_shape=True)
    rng = np.random.default_rng(56)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, 120)), dtype=np.uint8)) for _ in range(2)] for _ in range(5)]
    res = cfg.digest_batch(msgs)
    lay = cfg.layout
    nc = lay.n_spread_cols // 2
    columns = [(pkg.COL_GATE, i) for i in range(lay.n_gate_cols)] + [(pkg.COL_LOOKUP, i) for i in range(lay.n_lookup_cols)]
    columns += [(pkg.COL_FIXED, 0)] + [(pkg.COL_DENSE, i) for i in range(nc)] + [(pkg.COL_SPREAD, i) for i in range(nc)]
    columns += [(pkg.COL_INSTANCE, 0)]
    usable = (1 << 17) - 6
    beta, gamma = (O.int_to_mont(int.from_bytes(rng.bytes(32), "little") % O.P) for _ in range(2))
    kw = dict(columns_per_chunk=2, bind_output_bytes=True, digests=res.digests)
    want, err = cfg.permutation_product(res, columns, usable, beta, gamma, **kw)
    assert err == 0
    monkeypatch.setenv("H2SHA_TUNE", "pmchunk=2")            # three launches share the workspace
    got, err = cfg.permutation_product(res, columns, usable, beta, gamma, **kw)
    monkeypatch.delenv("H2SHA_TUNE")
    assert err == 0 and torch.equal(got, want)
    cfg.close()
