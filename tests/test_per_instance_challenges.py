"""Per-instance challenges (theta_i, beta_i, gamma_i) for the lookup and permutation argument columns: h2sha_permute_lookup_per_instance,
h2sha_permute_lookup_from_raw_per_instance, h2sha_lookup_product_per_instance and h2sha_permutation_product_per_instance.

The contract: for every instance i, A', S' and z are bit-identical to the shared-challenge call on instance i alone with row i's
challenges, except that a theta_i making two compressed spread-table rows equal (which the shared call refuses) is counted in
errors[i] and leaves that instance's A', S' rows unwritten.  With all rows equal the outputs are those of the shared call on the
whole batch and the per-instance errors sum to its counter.

CPU part: the argument checks of the C-ABI.  GPU part: every lookup of several configurations, 16-bit limbs, raw value lists,
the permutation product, equal rows, failures that stay with their instance, chunked launches and guard bands."""
import ctypes as C

import numpy as np
import pytest

from oracle import mock_prover as MP
from oracle import oracle as O

P = O.P
GATE, LOOKUP, DENSE, SPREAD, FIXED, INSTANCE = 0, 1, 2, 3, 4, 6


def _rand(rng):
    return int.from_bytes(rng.bytes(32), "little") % P


def _rows(rng, n):
    """[n, 4] u64: one random challenge per instance, Montgomery form"""
    return np.stack([O.int_to_mont(_rand(rng)) for _ in range(n)])


def _columns(lay, bind):
    nc = lay.n_spread_cols // 2
    cols = [(GATE, i) for i in range(lay.n_gate_cols)] + [(LOOKUP, i) for i in range(lay.n_lookup_cols)] + [(FIXED, 0)]
    cols += [(DENSE, i) for i in range(nc)] + [(SPREAD, i) for i in range(nc)]
    return cols + ([(INSTANCE, 0)] if bind else [])


# ----------------------------------------------------------------------------------------------------------------
# CPU: argument checks
# ----------------------------------------------------------------------------------------------------------------
def test_argument_checks_without_a_device(pkg):
    cfg = pkg.Sha256DynamicConfig.configure([64], device=-1, build_shape=True)
    L = pkg.load_library()
    info = cfg.lookup_info()
    spread_l = info["n_range_lookups"]
    buf = (C.c_uint64 * 8)()
    rows = np.stack([O.int_to_mont(1), O.int_to_mont(2)])
    ch = rows.ctypes.data
    usable = 1 << 17
    d, cols = cfg._perm_desc(_columns(cfg.layout, False), 1, 2, False, 0)
    # no CPU path: a plan-only engine refuses the calls
    assert L.h2sha_permute_lookup_per_instance(cfg._h, 2, 0, buf, usable, None, buf, buf, None, None) == pkg.H2SHA_ECUDA
    assert L.h2sha_permute_lookup_per_instance(cfg._h, 2, spread_l, buf, usable, ch, buf, buf, None, None) == pkg.H2SHA_ECUDA
    assert L.h2sha_lookup_product_per_instance(cfg._h, 2, 0, buf, buf, buf, buf, usable, None, ch, ch, buf, None, None) == pkg.H2SHA_ECUDA
    assert L.h2sha_permutation_product_per_instance(cfg._h, 2, C.byref(d), usable, buf, buf, buf, None, ch, ch, buf, None, None) == pkg.H2SHA_ECUDA
    # NULL challenge arrays
    assert L.h2sha_lookup_product_per_instance(cfg._h, 2, 0, buf, buf, buf, buf, usable, None, None, ch, buf, None, None) == pkg.H2SHA_EINVAL
    assert L.h2sha_lookup_product_per_instance(cfg._h, 2, 0, buf, buf, buf, buf, usable, None, ch, None, buf, None, None) == pkg.H2SHA_EINVAL
    assert L.h2sha_permutation_product_per_instance(cfg._h, 2, C.byref(d), usable, buf, buf, buf, None, None, ch, buf, None, None) == pkg.H2SHA_EINVAL
    assert L.h2sha_permutation_product_per_instance(cfg._h, 2, C.byref(d), usable, buf, buf, buf, None, ch, None, buf, None, None) == pkg.H2SHA_EINVAL
    # a spread lookup needs thetas
    assert L.h2sha_permute_lookup_per_instance(cfg._h, 2, spread_l, buf, usable, None, buf, buf, None, None) == pkg.H2SHA_EINVAL
    assert L.h2sha_permute_lookup_from_raw_per_instance(cfg._h, 0, 2, spread_l, usable, None, buf, buf, None, None) == pkg.H2SHA_EINVAL
    assert L.h2sha_lookup_product_per_instance(cfg._h, 2, spread_l, buf, buf, buf, buf, usable, None, ch, ch, buf, None, None) == pkg.H2SHA_EINVAL
    # a row that is not reduced is named
    bad = rows.copy()
    bad[1] = [0xFFFFFFFFFFFFFFFF] * 4
    assert L.h2sha_permute_lookup_per_instance(cfg._h, 2, spread_l, buf, usable, bad.ctypes.data, buf, buf, None, None) == pkg.H2SHA_EINVAL
    assert "thetas_mont row 1" in L.h2sha_last_error().decode()
    assert L.h2sha_permutation_product_per_instance(cfg._h, 2, C.byref(d), usable, buf, buf, buf, None, ch, bad.ctypes.data, buf, None, None) == pkg.H2SHA_EINVAL
    assert "gammas_mont row 1" in L.h2sha_last_error().decode()
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------
def _batch(pkg, sizes, n, seed, **kw):
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0, **kw)
    rng = np.random.default_rng(seed)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, s - 8)), dtype=np.uint8)) for s in sizes] for _ in range(n)]
    return cfg, cfg.digest_batch(msgs), rng


def _one(pkg, res, i):
    return pkg.BatchResult(None, None, res.gate[i:i + 1], res.lookup[i:i + 1], res.spread[i:i + 1])


def _check_lookups(pkg, cfg, res, mult, usable, lookups, rng):
    """per-instance A', S', z of every lookup in `lookups` == the shared calls on each instance alone"""
    import torch
    n = mult.shape[0]
    n_r = cfg.lookup_info()["n_range_lookups"]
    thetas, betas, gammas = _rows(rng, n), _rows(rng, n), _rows(rng, n)
    for l in lookups:
        th = None if l < n_r else thetas
        a_p, s_p, err = cfg.permute_lookup_per_instance(mult, l, usable, th)
        assert not err.any(), f"lookup {l}: {err}"
        z, err = cfg.lookup_product_per_instance(res, l, a_p, s_p, usable, betas, gammas, th)
        assert not err.any(), f"lookup {l}: {err}"
        for i in range(n):
            th_i = None if l < n_r else thetas[i]
            want_a, want_s = cfg.permute_lookup(mult[i:i + 1], l, usable, th_i)
            assert torch.equal(a_p[i], want_a[0]) and torch.equal(s_p[i], want_s[0]), f"lookup {l}, instance {i}: permuted pair"
            want_z, e = cfg.lookup_product(_one(pkg, res, i), l, want_a, want_s, usable, betas[i], gammas[i], th_i)
            assert e == 0 and torch.equal(z[i], want_z[0]), f"lookup {l}, instance {i}: z"
        if l >= n_r:   # the tables really are per instance
            assert not torch.equal(s_p[0], s_p[1]) and not torch.equal(a_p[0], a_p[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [
    dict(sizes=[64], n=8),                                                         # config 2 shape
    dict(sizes=[128, 128], n=3),                                                   # the reference's TestCircuit
    dict(sizes=[320], n=4, max_rows=9973),                                         # two range lookups
    dict(sizes=[192], n=3, lookup_bits=9, num_bits_lookup=4, num_advice_columns=3),
], ids=["cfg2", "128x128", "320_wraps", "9bit-3cols"])
def test_every_lookup_matches_the_shared_call_per_instance(pkg, kw):
    kw = dict(kw)
    sizes, n = kw.pop("sizes"), kw.pop("n")
    cfg, res, rng = _batch(pkg, sizes, n, 61, **kw)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6 if kw.get("lookup_bits", 16) == 16 else info["min_usable_rows"] + 11
    if "max_rows" in kw:
        assert info["n_range_lookups"] == 2
    mult, bad = cfg.lookup_multiplicities(res, usable)
    assert bad == 0
    _check_lookups(pkg, cfg, res, mult, usable, range(info["n_range_lookups"] + info["n_spread_lookups"]), rng)
    cfg.close()


@pytest.mark.gpu
def test_sixteen_bit_limbs(pkg):
    """num_bits_lookup = 16: a 2^16-row spread table sorted per instance on the device.  The spread multiplicities are counted on the
    host (the engine refuses 16-bit spread multiplicities)."""
    import torch
    n = 3
    cfg, res, rng = _batch(pkg, [64], n, 62, num_bits_lookup=16)
    info = cfg.lookup_info()
    assert info["spread_table_rows"] == 1 << 16
    usable = (1 << 17) - 6
    n_r, n_s = info["n_range_lookups"], info["n_spread_lookups"]
    L = pkg.load_library()
    mult = torch.zeros((n, info["mult_words_per_instance"]), dtype=torch.int32, device=res.lookup.device)
    assert L.h2sha_lookup_multiplicities(cfg._h, n, res.lookup.data_ptr(), None, usable, mult.data_ptr(), None,
                                         torch.cuda.current_stream(0).cuda_stream) == 0
    lay = cfg.layout
    cols = lay.n_spread_cols // 2
    for i in range(n):
        for c in range(cols):
            used = (lay.n_spread_limbs - c + cols - 1) // cols
            m = np.bincount(np.array(MP.canon_all(res.spread[i, c, :used].cpu().numpy().view(np.uint64)), dtype=np.int64), minlength=1 << 16)
            m[0] += usable - used
            mult[i, (n_r << 16) + (c << 16):(n_r << 16) + ((c + 1) << 16)] = torch.from_numpy(m.astype(np.int32))
    _check_lookups(pkg, cfg, res, mult, usable, (0, n_r, n_r + n_s - 1), rng)
    cfg.close()


@pytest.mark.gpu
def test_pairs_from_the_raw_value_lists(pkg):
    """permute_lookup_from_raw_per_instance == permute_lookup_per_instance, for the whole batch and for a slice from instance 1"""
    import torch
    n = 5
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0)
    info = cfg.lookup_info()
    usable = info["min_usable_rows"] + 5
    rng = np.random.default_rng(63)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, 56)), dtype=np.uint8))] for _ in range(n)]
    blob, offs, lens = pkg.pack_messages(msgs)
    gate, lookup, spread = cfg.alloc_outputs(n)
    cfg.digest_batch_raw(n, blob.ctypes.data if blob.size else 0, False, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                         spread_ptr=spread.data_ptr(), keep_lookup_raw=True, stream=torch.cuda.current_stream(0).cuda_stream)
    torch.cuda.synchronize()
    mult, bad = cfg.lookup_multiplicities(pkg.BatchResult(None, None, gate, lookup, spread), usable)
    assert bad == 0
    thetas = _rows(rng, n)
    for l in range(info["n_range_lookups"] + info["n_spread_lookups"]):
        th = None if l < info["n_range_lookups"] else thetas
        wa, ws, err = cfg.permute_lookup_per_instance(mult, l, usable, th)
        assert not err.any()
        ga, gs, err = cfg.permute_lookup_from_raw_per_instance(0, n, l, usable, th)
        assert not err.any() and torch.equal(ga, wa) and torch.equal(gs, ws), f"lookup {l}"
        ga, gs, err = cfg.permute_lookup_from_raw_per_instance(1, n - 1, l, usable, None if th is None else th[1:])
        assert not err.any() and torch.equal(ga, wa[1:]) and torch.equal(gs, ws[1:]), f"lookup {l}, instances 1.."
    cfg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [
    dict(sizes=[64], n=4, bind=False),        # config 2: 7 columns
    dict(sizes=[128, 128], n=3, bind=True),   # the TestCircuit with its instance column
], ids=["cfg2", "128x128"])
def test_permutation_product_matches_the_shared_call_per_instance(pkg, kw):
    import torch
    sizes, n, bind = kw["sizes"], kw["n"], kw["bind"]
    cfg, res, rng = _batch(pkg, sizes, n, 64, build_shape=True)
    columns = _columns(cfg.layout, bind)
    if not bind:
        assert len(columns) == 7
    usable = (1 << 17) - 6
    betas, gammas = _rows(rng, n), _rows(rng, n)
    D = cfg.layout.n_digests
    kw = dict(columns_per_chunk=2, bind_output_bytes=bind)
    z, err = cfg.permutation_product_per_instance(res, columns, usable, betas, gammas, digests=res.digests if bind else None, **kw)
    assert not err.any()
    for i in range(n):
        one = pkg.BatchResult(res.digests[i * D:(i + 1) * D], None, res.gate[i:i + 1], res.lookup[i:i + 1], res.spread[i:i + 1])
        want, e = cfg.permutation_product(one, columns, usable, betas[i], gammas[i], digests=one.digests if bind else None, **kw)
        assert e == 0 and torch.equal(z[i], want[0]), f"instance {i}"
    cfg.close()


@pytest.mark.gpu
def test_equal_rows_give_the_shared_batch_call(pkg):
    """all rows equal: bit-identical to the shared call on the whole batch, and the per-instance errors sum to its counter (one S'
    row of instance 3 is corrupted so that the counters have something to count)"""
    import torch
    n = 6
    cfg, res, rng = _batch(pkg, [64], n, 65, build_shape=True)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    theta, beta, gamma = (O.int_to_mont(_rand(rng)) for _ in range(3))
    rows = lambda x: np.tile(x, (n, 1))
    for l in (0, info["n_range_lookups"]):
        th = None if l < info["n_range_lookups"] else theta
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        ga, gs, err = cfg.permute_lookup_per_instance(mult, l, usable, None if th is None else rows(th))
        assert not err.any() and torch.equal(ga, a_p) and torch.equal(gs, s_p), f"lookup {l}"
        s_p[3, 1000] = s_p[3, int(torch.nonzero((s_p[3] != s_p[3, 1000]).any(-1))[0])]
        want, werr = cfg.lookup_product(res, l, a_p, s_p, usable, beta, gamma, th)
        got, err = cfg.lookup_product_per_instance(res, l, a_p, s_p, usable, rows(beta), rows(gamma), None if th is None else rows(th))
        assert torch.equal(got, want) and int(err.sum()) == werr == 1 and err[3] == 1, f"lookup {l}"
    columns = _columns(cfg.layout, False)
    want, werr = cfg.permutation_product(res, columns, usable, beta, gamma, columns_per_chunk=2)
    got, err = cfg.permutation_product_per_instance(res, columns, usable, rows(beta), rows(gamma), columns_per_chunk=2)
    assert torch.equal(got, want) and int(err.sum()) == werr == 0
    res.lookup[4, 0, 100, 0] ^= 1                             # a lookup cell no longer equals the gate cell it copies
    want, werr = cfg.permutation_product(res, columns, usable, beta, gamma, columns_per_chunk=2)
    got, err = cfg.permutation_product_per_instance(res, columns, usable, rows(beta), rows(gamma), columns_per_chunk=2)
    assert torch.equal(got, want) and int(err.sum()) == werr == 1 and err[4] == 1
    cfg.close()


@pytest.mark.gpu
def test_failures_stay_with_their_instance(pkg):
    import torch
    n = 5
    cfg, res, rng = _batch(pkg, [64], n, 66)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    n_r = info["n_range_lookups"]
    # theta = p - 3: spread-table rows 1 and 2 compress to the same value (1 * theta + 1 == 2 * theta + 4)
    thetas = _rows(rng, n)
    thetas[2] = O.int_to_mont(P - 3)
    a_p, s_p, err = cfg.permute_lookup_per_instance(mult, n_r, usable, thetas)
    assert err.tolist() == [0, 0, 1, 0, 0]
    for i in (0, 1, 3, 4):
        wa, ws = cfg.permute_lookup(mult[i:i + 1], n_r, usable, thetas[i])
        assert torch.equal(a_p[i], wa[0]) and torch.equal(s_p[i], ws[0]), f"instance {i}"
    with pytest.raises(pkg.EngineError):
        cfg.permute_lookup(mult[2:3], n_r, usable, thetas[2])
    # beta_1 = -A'[r] of instance 1: a zero denominator zeroes the rest of its column, and only its column
    a_p, s_p, err = cfg.permute_lookup_per_instance(mult, 0, usable)
    assert not err.any()
    ap1 = MP.canon_all(a_p[1].cpu().numpy().view(np.uint64).reshape(-1, 4))
    r = next(i for i in range(usable - 1, 0, -1) if ap1[i] != 0 and ap1[i] != ap1[i - 1])   # first row of the largest value's run
    betas, gammas = _rows(rng, n), _rows(rng, n)
    betas[1] = O.int_to_mont((P - ap1[r]) % P)
    z, err = cfg.lookup_product_per_instance(res, 0, a_p, s_p, usable, betas, gammas)
    assert err.tolist() == [0, 1, 0, 0, 0]
    want, e = cfg.lookup_product(_one(pkg, res, 1), 0, a_p[1:2], s_p[1:2], usable, betas[1], gammas[1])
    assert e == 1 and torch.equal(z[1], want[0])
    assert not bool(z[1, r + 1:].any())
    cfg.close()


@pytest.mark.gpu
def test_chunked_instances_give_the_same_columns(pkg, monkeypatch):
    """launches of two instances (lkchunk / pmchunk): the challenge rows follow their instances across the chunk boundaries"""
    import torch
    n = 5
    cfg, res, rng = _batch(pkg, [128], n, 67, build_shape=True)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    thetas, betas, gammas = _rows(rng, n), _rows(rng, n), _rows(rng, n)
    columns = _columns(cfg.layout, False)

    def run():
        out = []
        for l in (0, info["n_range_lookups"]):
            th = None if l < info["n_range_lookups"] else thetas
            a_p, s_p, err = cfg.permute_lookup_per_instance(mult, l, usable, th)
            z, zerr = cfg.lookup_product_per_instance(res, l, a_p, s_p, usable, betas, gammas, th)
            out += [a_p, s_p, z, err, zerr]
        z, err = cfg.permutation_product_per_instance(res, columns, usable, betas, gammas, columns_per_chunk=2)
        return out + [z, err]

    want = run()
    monkeypatch.setenv("H2SHA_TUNE", "lkchunk=2,pmchunk=2")   # three launches per call share the workspaces
    got = run()
    monkeypatch.delenv("H2SHA_TUNE")
    for k, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, np.ndarray):
            assert not w.any() and not g.any(), k
        else:
            assert torch.equal(g, w), k
    cfg.close()


@pytest.mark.gpu
def test_writes_stay_inside_their_buffers(pkg):
    """guard bands around A', S', z and the errors array stay untouched; the rows of an instance whose theta collides stay unwritten"""
    import torch
    rng = np.random.default_rng(68)
    usable = (1 << 16) + 777                                 # not a multiple of the 256-row tiles
    n = 5
    cfg, res, _ = _batch(pkg, [64], n, 68, build_shape=True)
    info = cfg.lookup_info()
    L = pkg.load_library()
    dev = res.gate.device
    st = torch.cuda.current_stream(0).cuda_stream
    G = 4096
    SENT, ESENT = 0x6B6B6B6B6B6B6B6B, 0x5A5A5A5A
    mult, _ = cfg.lookup_multiplicities(res, usable)
    thetas, betas, gammas = _rows(rng, n), _rows(rng, n), _rows(rng, n)
    thetas[3] = O.int_to_mont(P - 3)
    cells = n * usable * 4

    def guarded(count, fill, dtype):
        return torch.full((count + 2 * G,), fill, dtype=dtype, device=dev)

    def intact(t, count, fill):
        return bool((t[:G] == fill).all()) and bool((t[G + count:] == fill).all())

    for l in range(info["n_range_lookups"] + info["n_spread_lookups"]):
        spread_l = l >= info["n_range_lookups"]
        a, s = guarded(cells, SENT, torch.int64), guarded(cells, SENT, torch.int64)
        err = guarded(n, ESENT, torch.int32)
        err[G:G + n] = 0
        th = thetas.ctypes.data if spread_l else None
        assert L.h2sha_permute_lookup_per_instance(cfg._h, n, l, mult.data_ptr(), usable, th, a[G:].data_ptr(), s[G:].data_ptr(), err[G:].data_ptr(), st) == 0
        torch.cuda.synchronize()
        assert intact(a, cells, SENT) and intact(s, cells, SENT) and intact(err, n, ESENT), f"lookup {l}: guard band overwritten"
        assert err[G:G + n].tolist() == ([0, 0, 0, 1, 0] if spread_l else [0] * n)
        for t in (a, s):
            rows = t[G:G + cells].view(n, usable, 4)
            written = ~(rows == SENT).all(-1)
            for i in range(n):
                assert bool(written[i].all()) if not (spread_l and i == 3) else not bool(written[i].any()), f"lookup {l}, instance {i}"
        if spread_l:
            continue
        zc = n * (usable + 1) * 4
        z = guarded(zc, SENT, torch.int64)
        err = guarded(n, ESENT, torch.int32)
        err[G:G + n] = 0
        assert L.h2sha_lookup_product_per_instance(cfg._h, n, l, res.lookup.data_ptr(), None, a[G:].data_ptr(), s[G:].data_ptr(), usable, None,
                                                   betas.ctypes.data, gammas.ctypes.data, z[G:].data_ptr(), err[G:].data_ptr(), st) == 0
        torch.cuda.synchronize()
        assert intact(z, zc, SENT) and intact(err, n, ESENT) and err[G:G + n].tolist() == [0] * n, f"lookup {l}"
    usable = (1 << 17) - 6                                   # the permutation needs every copied cell (gate rows up to ~70 k) below usable_rows
    columns = _columns(cfg.layout, False)
    d, cols = cfg._perm_desc(columns, 1, 2, False, 0)
    zc = n * 4 * (usable + 1) * 4
    z = guarded(zc, SENT, torch.int64)
    err = guarded(n, ESENT, torch.int32)
    err[G:G + n] = 0
    rc = L.h2sha_permutation_product_per_instance(cfg._h, n, C.byref(d), usable, res.gate.data_ptr(), res.lookup.data_ptr(), res.spread.data_ptr(), None,
                                                  betas.ctypes.data, gammas.ctypes.data, z[G:].data_ptr(), err[G:].data_ptr(), st)
    assert rc == 0, L.h2sha_last_error().decode()
    torch.cuda.synchronize()
    assert intact(z, zc, SENT) and intact(err, n, ESENT) and err[G:G + n].tolist() == [0] * n
    assert not bool((z[G:G + zc].view(-1, 4) == SENT).all(-1).any()), "a row of z was not written"
    cfg.close()
