"""Grand-product column z of the lookup argument (halo2's `Permuted::commit_product`, restated below as `lookup_product`)
for the chip's range and spread lookups, on the device: h2sha_lookup_product.

CPU part: the restatement itself (z[0] = z[U] = 1 and the row constraint for a valid pair, z[U] != 1 for a broken one; the
tile algorithm the kernels use gives the same column, zero denominators included) and the host side of the C-ABI.
GPU part: h2sha_lookup_product against that restatement (and A', S' against the oracle) on the witness of real batches."""
import ctypes as C

import numpy as np
import pytest

from oracle import lookup_prework as LP
from oracle import mock_prover as MP
from oracle import oracle as O

P = O.P


def batch_invert(values):
    """ff `BatchInvertIter::batch_invert` in place: Montgomery's trick with one inversion; a zero is skipped and stays zero."""
    acc = 1
    tmp = []
    for p in values:
        tmp.append(acc)
        if p:
            acc = acc * p % P
    acc = pow(acc, P - 2, P)
    for i in range(len(values) - 1, -1, -1):
        p = values[i]
        if p:
            values[i] = tmp[i] * acc % P
            acc = acc * p % P


def lookup_product(a, s, a_p, s_p, beta, gamma, usable_rows):
    """halo2 lookup prover `Permuted::commit_product` without the trailing blinding rows (those are random): the grand-product
    column z[0 .. usable_rows] of one lookup from the compressed input / table expressions (a, s) and the permuted pair (a_p, s_p),
    canonical ints.  Same dependency as `permute_expression_pair` in oracle/lookup_prework.py (absent from the reference crate):
    a restatement of the published algorithm, **parity unpinned** against halo2_proofs itself."""
    # denominators (A'(x) + beta)(S'(x) + gamma), inverted together; a zero denominator stays zero
    product = [(beta + a_p[i]) * (gamma + s_p[i]) % P for i in range(usable_rows)]
    batch_invert(product)
    # numerators (A(x) + beta)(S(x) + gamma)
    for i in range(usable_rows):
        product[i] = product[i] * ((a[i] + beta) % P) % P * ((s[i] + gamma) % P) % P
    # iter::once(1).chain(lookup_product).scan(1, |state, cur| { state *= cur; Some(state) }).take(usable_rows + 1)
    z = []
    state = 1
    for cur in [1] + product:
        state = state * cur % P
        z.append(state)
    return z[:usable_rows + 1]


def _rand(rng):
    return int.from_bytes(rng.bytes(32), "little") % P


def _prod(xs):
    r = 1
    for x in xs:
        r = r * x % P
    return r


def _tiled(a, s, a_p, s_p, beta, gamma, usable, tile, seg):
    """What k_product_tiles + k_product_fold + k_product_fill compute: tile products, one inversion, per tile
    C_t = U_<t / V_<=t, then per segment of `seg` rows the constant times the products inside the segment."""
    u, v = [], []
    for i in range(usable):
        vi = (a_p[i] + beta) * (s_p[i] + gamma) % P
        ui = (a[i] + beta) * (s[i] + gamma) % P
        u.append(0 if vi == 0 else ui)
        v.append(1 if vi == 0 else vi)
    n_tiles = -(-usable // tile)
    pu = [_prod(u[t * tile:(t + 1) * tile]) for t in range(n_tiles)]
    pv = [_prod(v[t * tile:(t + 1) * tile]) for t in range(n_tiles)]
    inv = pow(_prod(pv), P - 2, P)
    z = [0] * (usable + 1)
    z[usable] = _prod(pu) * inv % P
    for t in range(n_tiles):
        c_t = _prod(pu[:t]) * inv % P * _prod(pv[t + 1:]) % P
        t0, t1 = t * tile, min((t + 1) * tile, usable)
        for s0 in range(t0, t1, seg):
            s1 = min(s0 + seg, t1)
            k = c_t * _prod(u[t0:s0]) % P * _prod(v[s1:t1]) % P
            for j in range(s0, s1):
                z[j] = k * _prod(u[s0:j]) % P * _prod(v[j:s1]) % P
    return z


def _range_case(rng, bits, usable):
    n = 1 << bits
    hot = rng.integers(0, n, size=max(1, n // 3))
    col = [int(hot[i]) for i in rng.integers(0, len(hot), size=int(rng.integers(0, usable + 1)))]
    a, s = LP.range_lookup_columns(col, usable, bits)
    return (a, s) + LP.permute_expression_pair(a, s, usable)


def _spread_case(rng, bits, usable):
    n = 1 << bits
    theta = _rand(rng)
    dense = [int(x) for x in rng.integers(0, n, size=int(rng.integers(0, usable + 1)))]
    a, s = LP.spread_lookup_columns(dense, [LP.spread_bits(d, bits) for d in dense], usable, bits, theta)
    return (a, s) + LP.permute_expression_pair(a, s, usable)


@pytest.mark.parametrize("seed", range(6))
def test_restated_product_closes_and_holds_the_row_constraint(seed):
    rng = np.random.default_rng(200 + seed)
    bits = int(rng.integers(2, 7))
    usable = (1 << bits) + int(rng.integers(0, 3 << bits))
    a, s, a_p, s_p = (_range_case if seed % 2 else _spread_case)(rng, bits, usable)
    beta, gamma = _rand(rng), _rand(rng)
    z = lookup_product(a, s, a_p, s_p, beta, gamma, usable)
    assert len(z) == usable + 1 and z[0] == 1 and z[usable] == 1
    for i in range(usable):
        assert z[i + 1] * (a_p[i] + beta) * (s_p[i] + gamma) % P == z[i] * (a[i] + beta) * (s[i] + gamma) % P, f"row {i}"
    # one S' row replaced by another table value: S' is no longer a permutation of S
    r = int(rng.integers(0, usable))
    other = next(t for t in s if t != s_p[r])
    s_bad = list(s_p)
    s_bad[r] = other
    assert lookup_product(a, s, a_p, s_bad, beta, gamma, usable)[usable] != 1


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("zero_row", [False, True])
def test_tile_algorithm_matches_the_literal_restatement(seed, zero_row):
    rng = np.random.default_rng(300 + seed)
    bits = int(rng.integers(2, 6))
    usable = (1 << bits) + int(rng.integers(0, 5 << bits))
    a, s, a_p, s_p = (_range_case if seed % 2 else _spread_case)(rng, bits, usable)
    beta, gamma = _rand(rng), _rand(rng)
    if zero_row:   # v_r = 0: batch_invert leaves it 0, every later z is 0
        r = int(rng.integers(0, usable))
        beta = (P - a_p[r]) % P
    want = lookup_product(a, s, a_p, s_p, beta, gamma, usable)
    if zero_row:
        assert want[r + 1:] == [0] * (usable - r)
    for tile, seg in ((4, 1), (8, 4), (16, 4), (7, 3), (usable, 8), (usable + 5, usable)):
        assert _tiled(a, s, a_p, s_p, beta, gamma, usable, tile, seg) == want, (tile, seg)


def test_argument_checks_without_a_device(pkg):
    cfg = pkg.Sha256DynamicConfig.configure([64], device=-1)
    L = pkg.load_library()
    buf = (C.c_uint64 * 8)()
    one = O.int_to_mont(1)
    usable = 1 << 17
    # no CPU path: a plan-only engine refuses the call
    assert L.h2sha_lookup_product(cfg._h, 1, 0, buf, buf, buf, buf, usable, None, one.ctypes.data, one.ctypes.data, buf, None, None) == pkg.H2SHA_ECUDA
    assert L.h2sha_lookup_product(cfg._h, 1, 0, buf, buf, buf, buf, usable, None, None, one.ctypes.data, buf, None, None) == pkg.H2SHA_EINVAL
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------
def _canon(t):
    return MP.canon_all(t.cpu().numpy().view(np.uint64).reshape(-1, 4))


def _expressions(cfg, res, inst, l, usable, theta, max_rows):
    """oracle (A, S) of lookup l of one instance, from the canonical ints of its assigned cells"""
    lay, info = cfg.layout, cfg.lookup_info()
    n_r = info["n_range_lookups"]
    if l < n_r:
        used = max(0, min(max_rows, lay.n_lookup_cells - l * max_rows))
        return LP.range_lookup_columns(_canon(res.lookup[inst, l, :used]), usable, info["range_table_rows"].bit_length() - 1)
    c, cols = l - n_r, lay.n_spread_cols // 2
    used = (lay.n_spread_limbs - c + cols - 1) // cols if lay.n_spread_limbs > c else 0
    return LP.spread_lookup_columns(_canon(res.spread[inst, c, :used]), _canon(res.spread[inst, cols + c, :used]), usable,
                                    info["spread_table_rows"].bit_length() - 1, theta)


def _batch(pkg, sizes, n, seed, **kw):
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0, **kw)
    rng = np.random.default_rng(seed)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, s - 8)), dtype=np.uint8)) for s in sizes] for _ in range(n)]
    return cfg, cfg.digest_batch(msgs), rng


def _challenges(rng):
    return [O.int_to_mont(_rand(rng)) for _ in range(3)]   # theta, beta, gamma


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [
    dict(sizes=[64], n=48),                                                        # config 2 shape
    dict(sizes=[128, 128], n=3),                                                   # the reference's TestCircuit
    dict(sizes=[320], n=4, max_rows=9973),                                         # two range lookups
    dict(sizes=[192], n=3, lookup_bits=9, num_bits_lookup=4, num_advice_columns=3),
], ids=["cfg2", "128x128", "320_wraps", "9bit-3cols"])
def test_product_matches_the_restatement(pkg, kw):
    kw = dict(kw)
    sizes, n = kw.pop("sizes"), kw.pop("n")
    max_rows = kw.get("max_rows", (1 << 17) - 9)
    cfg, res, rng = _batch(pkg, sizes, n, 41, **kw)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6 if kw.get("lookup_bits", 16) == 16 else info["min_usable_rows"] + 11
    n_r = info["n_range_lookups"]
    if "max_rows" in kw:
        assert n_r == 2
    mult, bad = cfg.lookup_multiplicities(res, usable)
    assert bad == 0
    theta_m, beta_m, gamma_m = _challenges(rng)
    theta, beta, gamma = (O.mont_to_int(x) for x in (theta_m, beta_m, gamma_m))
    for l in range(n_r + info["n_spread_lookups"]):
        th = None if l < n_r else theta_m
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        z, errors = cfg.lookup_product(res, l, a_p, s_p, usable, beta_m, gamma_m, th)
        assert errors == 0, f"lookup {l}: {errors} instance(s) with z[U] != 1"
        assert z.shape == (n, usable + 1, 4)
        for inst in (0, n - 1):
            a, s = _expressions(cfg, res, inst, l, usable, theta, max_rows)
            want_ap, want_sp = LP.permute_expression_pair(a, s, usable)
            got_ap, got_sp = _canon(a_p[inst]), _canon(s_p[inst])
            assert got_ap == want_ap and got_sp == want_sp, f"lookup {l}, instance {inst}: permuted pair"
            assert _canon(z[inst]) == lookup_product(a, s, want_ap, want_sp, beta, gamma, usable), f"lookup {l}, instance {inst}"
    cfg.close()


@pytest.mark.gpu
def test_product_of_pairs_from_the_raw_value_lists(pkg):
    """A', S' from h2sha_permute_lookup_from_raw, for the whole batch and for a slice from instance 1 (every pointer offset): same z"""
    import torch
    sizes, n = [64], 5
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0)
    info = cfg.lookup_info()
    usable = info["min_usable_rows"] + 5
    rng = np.random.default_rng(42)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, 56)), dtype=np.uint8))] for _ in range(n)]
    blob, offs, lens = pkg.pack_messages(msgs)
    gate, lookup, spread = cfg.alloc_outputs(n)
    cfg.digest_batch_raw(n, blob.ctypes.data if blob.size else 0, False, int(blob.size), offs, lens, None, gate_ptr=gate.data_ptr(), lookup_ptr=lookup.data_ptr(),
                         spread_ptr=spread.data_ptr(), keep_lookup_raw=True, stream=torch.cuda.current_stream(0).cuda_stream)
    torch.cuda.synchronize()
    res = pkg.BatchResult(None, None, gate, lookup, spread)
    mult, bad = cfg.lookup_multiplicities(res, usable)
    assert bad == 0
    theta, beta, gamma = _challenges(rng)
    sl = pkg.BatchResult(None, None, gate[1:], lookup[1:], spread[1:])
    for l in range(info["n_range_lookups"] + info["n_spread_lookups"]):
        th = None if l < info["n_range_lookups"] else theta
        want, err = cfg.lookup_product(res, l, *cfg.permute_lookup(mult, l, usable, th), usable, beta, gamma, th)
        assert err == 0
        got, err = cfg.lookup_product(res, l, *cfg.permute_lookup_from_raw(0, n, l, usable, th), usable, beta, gamma, th)
        assert err == 0 and torch.equal(got, want), f"lookup {l}"
        got, err = cfg.lookup_product(sl, l, *cfg.permute_lookup_from_raw(1, n - 1, l, usable, th), usable, beta, gamma, th)
        assert err == 0 and torch.equal(got, want[1:]), f"lookup {l}, instances 1.."
    cfg.close()


@pytest.mark.gpu
def test_corrupted_table_row_is_counted_for_its_instance_only(pkg):
    import torch
    cfg, res, rng = _batch(pkg, [64], 6, 43)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    theta, beta, gamma = _challenges(rng)
    for l in (0, info["n_range_lookups"]):   # a range and a spread lookup
        th = None if l < info["n_range_lookups"] else theta
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        want, err = cfg.lookup_product(res, l, a_p, s_p, usable, beta, gamma, th)
        assert err == 0
        r = 1000
        other = int(torch.nonzero((s_p[3] != s_p[3, r]).any(-1))[0])
        s_p[3, r] = s_p[3, other]                             # another table value in row r of instance 3
        got, err = cfg.lookup_product(res, l, a_p, s_p, usable, beta, gamma, th)
        assert err == 1, f"lookup {l}"
        keep = [i for i in range(6) if i != 3]
        assert torch.equal(got[keep], want[keep])
        assert torch.equal(got[3, :r + 1], want[3, :r + 1]) and not torch.equal(got[3, -1], want[3, -1])
    cfg.close()


@pytest.mark.gpu
def test_zero_denominator_zeroes_the_rest_of_the_column(pkg):
    """beta = -A'[r] makes v_r = 0: like ff's batch_invert, the fraction of row r is 0 and so is every later z"""
    cfg, res, rng = _batch(pkg, [64], 3, 44)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    theta_m, _, gamma_m = _challenges(rng)
    theta, gamma = O.mont_to_int(theta_m), O.mont_to_int(gamma_m)
    for l in (0, info["n_range_lookups"]):
        th = None if l < info["n_range_lookups"] else theta_m
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        ap0 = _canon(a_p[0])
        r = next(i for i in range(usable - 1, 0, -1) if ap0[i] != 0 and ap0[i] != ap0[i - 1])   # first row of the largest value's run
        beta = (P - ap0[r]) % P
        z, errors = cfg.lookup_product(res, l, a_p, s_p, usable, O.int_to_mont(beta), gamma_m, th)
        hit = sum(bool((a_p[i] == a_p[0, r]).all(-1).any()) for i in range(3))   # instances with that value in A' get a zero denominator too
        assert errors == hit >= 1
        a, s = _expressions(cfg, res, 0, l, usable, theta, (1 << 17) - 9)
        want = lookup_product(a, s, ap0, _canon(s_p[0]), beta, gamma, usable)
        assert want[r + 1:] == [0] * (usable - r)
        assert _canon(z[0]) == want, f"lookup {l}"
    cfg.close()


@pytest.mark.gpu
def test_sixteen_bit_limbs(pkg):
    """num_bits_lookup = 16: range multiplicities from the engine (spread = NULL), spread multiplicities counted on the host (the engine
    keeps no 2^16-bin histograms in shared memory); the permutation of the 2^16-row spread table against the oracle, z against the restatement"""
    import torch
    sizes, n = [64], 2
    cfg, res, rng = _batch(pkg, sizes, n, 45, num_bits_lookup=16)
    info = cfg.lookup_info()
    assert info["spread_table_rows"] == 1 << 16
    usable = (1 << 17) - 6
    n_r, n_s = info["n_range_lookups"], info["n_spread_lookups"]
    L = pkg.load_library()
    mult = torch.zeros((n, info["mult_words_per_instance"]), dtype=torch.int32, device=res.lookup.device)
    bad = torch.zeros(1, dtype=torch.int32, device=res.lookup.device)
    assert L.h2sha_lookup_multiplicities(cfg._h, n, res.lookup.data_ptr(), None, usable, mult.data_ptr(), bad.data_ptr(),
                                         torch.cuda.current_stream(0).cuda_stream) == 0
    lay = cfg.layout
    cols = lay.n_spread_cols // 2
    for i in range(n):
        for c in range(cols):
            used = (lay.n_spread_limbs - c + cols - 1) // cols
            m = np.bincount(np.array(_canon(res.spread[i, c, :used]), dtype=np.int64), minlength=1 << 16)
            m[0] += usable - used
            mult[i, (n_r << 16) + (c << 16):(n_r << 16) + ((c + 1) << 16)] = torch.from_numpy(m.astype(np.int32))
    assert int(bad.item()) == 0
    theta_m, beta_m, gamma_m = _challenges(rng)
    theta, beta, gamma = (O.mont_to_int(x) for x in (theta_m, beta_m, gamma_m))
    for l in (0, n_r, n_r + n_s - 1):
        th = None if l < n_r else theta_m
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        z, errors = cfg.lookup_product(res, l, a_p, s_p, usable, beta_m, gamma_m, th)
        assert errors == 0
        a, s = _expressions(cfg, res, 1, l, usable, theta, (1 << 17) - 9)
        want_ap, want_sp = LP.permute_expression_pair(a, s, usable)
        assert _canon(a_p[1]) == want_ap and _canon(s_p[1]) == want_sp, f"lookup {l}: permuted pair"
        assert _canon(z[1]) == lookup_product(a, s, want_ap, want_sp, beta, gamma, usable), f"lookup {l}"
    cfg.close()


@pytest.mark.gpu
def test_chunked_instances_give_the_same_column(pkg, monkeypatch):
    import torch
    cfg, res, rng = _batch(pkg, [128], 5, 46)
    info = cfg.lookup_info()
    usable = (1 << 17) - 6
    mult, _ = cfg.lookup_multiplicities(res, usable)
    theta, beta, gamma = _challenges(rng)
    for l in (0, info["n_range_lookups"]):
        th = None if l < info["n_range_lookups"] else theta
        a_p, s_p = cfg.permute_lookup(mult, l, usable, th)
        want, _ = cfg.lookup_product(res, l, a_p, s_p, usable, beta, gamma, th)
        monkeypatch.setenv("H2SHA_TUNE", "lkchunk=2")        # three launches share the workspace
        got, err = cfg.lookup_product(res, l, a_p, s_p, usable, beta, gamma, th)
        monkeypatch.delenv("H2SHA_TUNE")
        assert err == 0 and torch.equal(got, want), f"lookup {l}"
    cfg.close()
