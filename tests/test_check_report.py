"""Per-instance verdicts of the device constraint check (h2sha_check_batch_per_instance) and the cells behind a failing item
(h2sha_check_site), the way halo2's MockProver names a VerifyFailure by column and row.

The item numbering is restated here from the shape (h2sha_get_shape, h2sha_get_breaks, the handles) and the lookup geometry, and
compared with the resolver on plan-only engines.  On the GPU: a clean batch reports nothing, one corruption per instance stays with
its instance and resolves to the corrupted cell, and ~50 random corruptions match a host restatement of the check exactly."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from oracle.mock_prover import spread_bits

MAX_ROWS = (1 << 17) - 9
NONE = 0xFFFFFFFF
GATE, LOOKUP, DENSE, SPREAD, FIXED = 0, 1, 2, 3, 4


class Restated:
    """The item numbering of include/h2sha_b200.h, from the shape of a build_shape engine."""

    def __init__(self, shp, max_rows, spread_cols):
        self.sh, self.brk, self.lay = shp.shape(), shp.breaks(), shp.layout
        self.on = np.nonzero(self.sh.selectors)[0]
        self.out = [shp.handles(d).output_bytes for d in range(self.lay.n_digests)]
        self.max_rows, self.sc = max_rows, spread_cols
        L = self.lay
        self.sizes = [len(self.on), L.n_copies + L.n_lookup_cells + 2 * L.n_spread_limbs, L.n_lookup_cells, L.n_spread_limbs, 32 * L.n_digests]

    def pos(self, idx):
        c = int(np.searchsorted(self.brk, idx, side="right") - 1)
        return (GATE, c, int(idx - self.brk[c]))

    def lookup_cell(self, k):
        return (LOOKUP, k // self.max_rows, k % self.max_rows)

    def limb(self, n):
        return (n % self.sc, n // self.sc)

    def cells(self, cls, item):
        sh, L = self.sh, self.lay
        if cls == 0:
            s = int(self.on[item])
            return [self.pos(s + j) for j in range(4)]
        if cls == 1:
            if item < L.n_copies:
                ak, ai, bk, bi = (int(x) for x in sh.copies[item])
                return [self.pos(ai) if ak == 0 else (FIXED, 0, ai), self.pos(bi) if bk == 0 else (FIXED, 0, bi)]
            q = item - L.n_copies
            if q < L.n_lookup_cells:
                return [self.lookup_cell(q), self.pos(int(sh.lookup_src[q]))]
            n, which = divmod(q - L.n_lookup_cells, 2)
            if which == 0:
                return [(DENSE,) + self.limb(n), self.pos(int(sh.limb_dense_src[n]))]
            return [(SPREAD,) + self.limb(n), self.pos(int(sh.limb_spread_src[n]))]
        if cls == 2:
            return [self.lookup_cell(item)]
        if cls == 3:
            return [(DENSE,) + self.limb(item), (SPREAD,) + self.limb(item)]
        d, j = divmod(item, 32)
        return [self.pos(int(self.out[d][j]))]


def _site(cfg, cls, item):
    s = cfg.check_site(cls, item)
    return list(zip(s["kind"], s["index"], s["row"]))


CPU_CONFIGS = [
    dict(sizes=[64]),                                                          # cfg2
    dict(sizes=[64, 64], split=True, num_advice_columns=3, num_bits_lookup=4),   # two digests, two lookup columns, three spread pairs
    dict(sizes=[128], num_bits_lookup=16),
    dict(sizes=[64, 64], gate_col_rows=1 << 17, lookup_col_rows=1 << 17, spread_rows=1 << 17, num_lookup_advice=2),   # widened strides
]


def _kw(pkg, c):
    c = dict(c)
    sizes, split = c.pop("sizes"), c.pop("split", False)
    if split:
        probe = pkg.Sha256DynamicConfig.configure(sizes, device=-1, **c)
        c["max_rows"] = (probe.layout.n_lookup_cells + 1) // 2
        probe.close()
    c.setdefault("max_rows", MAX_ROWS)
    return sizes, c


@pytest.mark.parametrize("conf", CPU_CONFIGS, ids=["cfg2", "two_digests_two_lookup_cols_3pairs", "limb16", "widened"])
def test_sites_follow_the_documented_numbering(pkg, conf):
    sizes, kw = _kw(pkg, conf)
    shp = pkg.Sha256DynamicConfig.configure(sizes, device=-1, build_shape=True, **kw)
    plain = pkg.Sha256DynamicConfig.configure(sizes, device=-1, **kw)   # no build_shape: the resolver builds the shape itself
    R = Restated(shp, kw["max_rows"], kw.get("num_advice_columns", 2))
    if conf.get("split"):
        assert shp.layout.n_lookup_cols == 2 and shp.lookup_info()["n_range_lookups"] == 2
    rng = np.random.default_rng(5)
    L = shp.layout
    for cls, n in enumerate(R.sizes):
        assert n > 0
        items = {0, n - 1} | set(int(x) for x in rng.integers(0, n, size=12))
        if cls == 1:   # the segment boundaries: shape copies | range.finalize | dense, spread per limb
            b = [L.n_copies, L.n_copies + L.n_lookup_cells]
            items |= {b[0] - 1, b[0], b[1] - 1, b[1], b[1] + 1}
        if cls == 2:   # the first cell of the second lookup column
            items |= {min(n - 1, kw["max_rows"])}
        for it in sorted(items):
            want = R.cells(cls, it)
            assert _site(plain, cls, it) == want, (cls, it)
            assert _site(shp, cls, it) == want, (cls, it)
    # out of range
    lib = pkg.load_library()
    s = pkg._CheckSite()
    assert lib.h2sha_check_site(plain._h, 5, 0, C.byref(s)) == pkg.H2SHA_EINVAL
    for cls, n in enumerate(R.sizes):
        assert lib.h2sha_check_site(plain._h, cls, n, C.byref(s)) == pkg.H2SHA_EINVAL
    shp.close(); plain.close()


def test_plan_only_engine_refuses_the_per_instance_check(pkg):
    cfg = pkg.Sha256DynamicConfig.configure([64], device=-1)
    buf = (C.c_uint64 * 8)()
    assert pkg.load_library().h2sha_check_batch_per_instance(cfg._h, 1, buf, buf, buf, None, buf, buf, None) == pkg.H2SHA_ECUDA
    cfg.close()


# ------------------------------------------------------------------------------------------------------------- GPU

def _mont(v):
    import torch
    return torch.from_numpy(O.int_to_mont(v).view(np.int64))


def _raw_per_instance(pkg, cfg, gate, lookup, spread, dig_ptr, n, fill=None):
    """the C call on (possibly offset) buffers, into arrays pre-filled with `fill`"""
    import torch
    out = torch.full((2, n, 5), 0 if fill is None else fill, dtype=torch.int32, device="cuda")
    rc = pkg.load_library().h2sha_check_batch_per_instance(cfg._h, n, gate, lookup, spread, C.c_void_p(dig_ptr or None), out[0].data_ptr(),
                                                           out[1].data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, pkg.load_library().h2sha_last_error()
    o = out.cpu().numpy().view(np.uint32)
    return o[0].copy(), o[1].copy()


def _batch(pkg, sizes, n, seed, **kw):
    import torch
    rng = np.random.default_rng(seed)
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0, **kw)
    msgs = [[bytes(rng.integers(0, 256, size=int(rng.integers(0, s - 8)), dtype=np.uint8)) for s in sizes] for _ in range(n)]
    res = cfg.digest_batch(msgs)
    return cfg, res, torch.from_numpy(res.digests).cuda()


GPU_CONFIGS = [
    dict(sizes=[128, 128]),
    dict(sizes=[320], max_rows=9973),                                      # two lookup columns
    dict(sizes=[128], num_bits_lookup=16, num_advice_columns=3),           # 16-bit limbs, three spread pairs
    dict(sizes=[128], gate_col_rows=1 << 17, lookup_col_rows=1 << 17, spread_rows=1 << 17),   # widened strides
]
GPU_IDS = ["two_digests", "two_lookup_cols", "limb16_3pairs", "widened"]


@pytest.mark.gpu
@pytest.mark.parametrize("conf", GPU_CONFIGS, ids=GPU_IDS)
def test_clean_batch_reports_nothing_and_overwrites(pkg, conf):
    conf = dict(conf)
    sizes = conf.pop("sizes")
    cfg, res, dig = _batch(pkg, sizes, 5, 21, **conf)
    n = res.gate.shape[0]
    for dig_ptr in (dig.data_ptr(), 0):
        for fill in (0x5A5A5A5A, -1):
            counts, first = _raw_per_instance(pkg, cfg, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(), dig_ptr, n, fill)
            assert (counts == 0).all() and (first == NONE).all()
        counts, first = cfg.check_batch_per_instance(res, dig_ptr)
        assert counts.shape == (n, 5) and (counts == 0).all() and (first == NONE).all()
    cfg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("conf", GPU_CONFIGS, ids=GPU_IDS)
def test_one_corruption_per_instance_stays_with_its_instance(pkg, conf):
    conf = dict(conf)
    sizes = conf.pop("sizes")
    D = len(sizes)
    cfg, res, dig = _batch(pkg, sizes, 7, 22, **conf)
    kw = {k: v for k, v in conf.items() if k not in ("gate_col_rows", "lookup_col_rows", "spread_rows")}
    shp = pkg.Sha256DynamicConfig.configure(sizes, device=-1, build_shape=True, **kw)
    R = Restated(shp, conf.get("max_rows", MAX_ROWS), conf.get("num_advice_columns", 2))
    sh = R.sh
    sc = conf.get("num_advice_columns", 2)
    # (a) instance 1: the output cell of a gate
    g = int(R.on[len(R.on) // 2])
    _, c, r = R.pos(g + 3)
    res.gate[1, c, r] = _mont(123456789).cuda()
    cell_a = (GATE, c, r)
    # (b) instance 2: a cell copy-constrained to a fixed constant
    fixed_copies = [cp for cp in sh.copies.tolist() if cp[2] == 1 or cp[0] == 1]
    cp = fixed_copies[len(fixed_copies) // 3]
    gidx = cp[1] if cp[0] == 0 else cp[3]
    _, c, r = R.pos(gidx)
    old = O.mont_to_int(res.gate[2, c, r].cpu().numpy().view(np.uint64))
    res.gate[2, c, r] = _mont(77 if old != 77 else 78).cuda()
    cell_b = (GATE, c, r)
    # (c) instance 3: a lookup-column cell outside the range table
    lk_col = 1 if R.lay.n_lookup_cells > R.max_rows + 9 else 0   # the second lookup column where there is one
    res.lookup[3, lk_col, 9] = _mont((1 << 16) + 5).cuda()
    cell_c = (LOOKUP, lk_col, 9)
    # (d) instance 4: the spread half of a table row (spread column of pair 0, row 5)
    ncol = R.lay.n_spread_cols // 2
    res.spread[4, ncol, 5] = _mont(2).cuda()
    cell_d = (SPREAD, 0, 5)
    # (e) instance 5: byte 7 of its last digest
    dig2 = dig.clone()
    dig2[5 * D + D - 1, 7] ^= 1
    n = res.gate.shape[0]

    counts, first = cfg.check_batch_per_instance(res, dig2.data_ptr())
    total = cfg.check_batch(res, dig2.data_ptr())
    assert [int(x) for x in counts.sum(axis=0)] == [total[k] for k in ("gates", "copies", "range_lookups", "spread_lookups", "digest_bytes")]
    for i in (0, 6):
        assert (counts[i] == 0).all() and (first[i] == NONE).all(), i
    site = lambda i, cls: _site(cfg, cls, int(first[i, cls]))
    # (a)
    assert counts[1, 0] >= 1 and counts[1, 2] == 0 and counts[1, 3] == 0 and counts[1, 4] == 0, counts[1]
    assert site(1, 0)[3] == cell_a
    if counts[1, 1]:
        assert cell_a in site(1, 1)
    # (b)
    assert counts[2, 1] >= 1 and counts[2, 2] == 0 and counts[2, 3] == 0 and counts[2, 4] == 0, counts[2]
    assert cell_b in site(2, 1)
    # (c)
    assert counts[3, 2] == 1 and counts[3, 1] >= 1 and counts[3, 0] == 0 and counts[3, 3] == 0 and counts[3, 4] == 0, counts[3]
    assert site(3, 2) == [cell_c] and cell_c in site(3, 1)
    # (d)
    assert counts[4, 3] == 1 and counts[4, 1] >= 1 and counts[4, 0] == 0 and counts[4, 2] == 0 and counts[4, 4] == 0, counts[4]
    assert cell_d in site(4, 3) and cell_d in site(4, 1)
    assert int(first[4, 3]) == 5 * sc
    # (e)
    assert list(counts[5]) == [0, 0, 0, 0, 1] and int(first[5, 4]) == (D - 1) * 32 + 7
    assert site(5, 4) == [R.pos(int(R.out[D - 1][7]))]
    # every instance alone, through offset pointers
    for i in range(n):
        one_c, one_f = _raw_per_instance(pkg, cfg, res.gate[i].data_ptr(), res.lookup[i].data_ptr(), res.spread[i].data_ptr(),
                                         dig2[i * D].data_ptr(), 1, 0x3C3C3C3C)
        assert (one_c[0] == counts[i]).all() and (one_f[0] == first[i]).all(), i
        v = np.zeros(5, dtype=np.uint64)
        import torch
        assert pkg.load_library().h2sha_check_batch(cfg._h, 1, res.gate[i].data_ptr(), res.lookup[i].data_ptr(), res.spread[i].data_ptr(),
                                                    C.c_void_p(dig2[i * D].data_ptr()), v.ctypes.data_as(C.c_void_p),
                                                    torch.cuda.current_stream().cuda_stream) == 0
        assert [int(x) for x in v] == [int(x) for x in counts[i]], i
    cfg.close(); shp.close()


def _canon(a):
    """[..., 4] int64 Montgomery -> object array of canonical ints"""
    flat = np.ascontiguousarray(a).view(np.uint64).reshape(-1, 4)
    return np.array([O.mont_to_int(x) for x in flat], dtype=object).reshape(a.shape[:-1])


@pytest.mark.gpu
def test_random_corruptions_match_a_host_restatement(pkg):
    sizes = [128]
    cfg, res, dig = _batch(pkg, sizes, 3, 23)
    shp = pkg.Sha256DynamicConfig.configure(sizes, device=-1, build_shape=True)
    R = Restated(shp, MAX_ROWS, 2)
    sh, L = R.sh, R.lay
    rng = np.random.default_rng(24)
    inst = 1
    used_gate = [R.pos(int(i)) for i in rng.integers(0, L.n_gate_cells, size=30)]
    for _, c, r in used_gate:
        res.gate[inst, c, r] = _mont(int(rng.integers(0, 1 << 17))).cuda()
    for k in rng.integers(0, L.n_lookup_cells, size=10):
        _, c, r = R.lookup_cell(int(k))
        res.lookup[inst, c, r] = _mont(int(rng.integers(0, 1 << 17))).cuda()
    for n_ in rng.integers(0, L.n_spread_limbs, size=10):
        col, row = R.limb(int(n_))
        res.spread[inst, col + (L.n_spread_cols // 2) * int(rng.integers(0, 2)), row] = _mont(int(rng.integers(0, 1 << 9))).cuda()
    counts, first = cfg.check_batch_per_instance(res, dig.data_ptr())

    g = _canon(res.gate[inst].cpu().numpy())
    lk = _canon(res.lookup[inst].cpu().numpy())
    sp = _canon(res.spread[inst].cpu().numpy())
    fixed = [int(x[0]) | int(x[1]) << 64 | int(x[2]) << 128 | int(x[3]) << 192 for x in sh.fixed]
    digest = res.digests[inst * L.n_digests:(inst + 1) * L.n_digests]
    half = L.n_spread_cols // 2

    def val(cell):
        k, c, r = cell
        return {GATE: lambda: g[c, r], LOOKUP: lambda: lk[c, r], DENSE: lambda: sp[c, r], SPREAD: lambda: sp[half + c, r],
                FIXED: lambda: fixed[r]}[k]()

    def fails(cls, it):
        cells = [val(x) for x in R.cells(cls, it)]
        if cls == 0:
            a, b, c_, d = cells
            return (a + b * c_ - d) % O.P != 0
        if cls == 1:
            return cells[0] != cells[1]
        if cls == 2:
            return cells[0] >= 1 << 16
        if cls == 3:
            d, s = cells
            return not (d < 1 << 8 and spread_bits(d) == s)
        return cells[0] != int(digest[it // 32][it % 32])

    for cls, n in enumerate(R.sizes):
        bad = [it for it in range(n) if fails(cls, it)]
        assert int(counts[inst, cls]) == len(bad), (cls, counts[inst], len(bad))
        assert int(first[inst, cls]) == (bad[0] if bad else NONE), cls
    assert sum(len([1 for it in range(n) if fails(cls, it)]) for cls, n in enumerate(R.sizes)) > 10
    for i in (0, 2):
        assert (counts[i] == 0).all()
    cfg.close(); shp.close()
