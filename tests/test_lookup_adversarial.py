"""The lookup- and permutation-argument kernels on adversarial inputs: synthetic multiplicities, spread-table thetas whose canonical
values tie on their top limbs, field values on the carry and reduction edges of the Montgomery arithmetic, row counts on the edges
of the grand product's tiles, and near misses of table membership.

The chip's own witness never reaches most of these: its multiplicities have a huge m[0] and a few hundred distinct values, random
thetas give every spread-table row its own top limb, and random 256-bit operands hit a carry edge with probability ~2^-64.  So
every call here is driven with synthetic device inputs and compared with a plain big-integer restatement:
  * A', S'  against `permuted_from_counts`, a vectorised literal restatement of halo2's `permute_expression_pair` (checked on the
            CPU against oracle/lookup_prework.py itself, not against the scan formulation the kernels use);
  * z       against `lookup_product` (tests/test_lookup_product.py) and `permutation_commit` (tests/test_permutation_product.py);
  * table membership against the canonical value of each replaced cell.

CPU part: the restatement, the edge-value generator and the theta classifier.  GPU part: the five groups of the module's
sections below."""
import numpy as np
import pytest

from oracle import lookup_prework as LP
from oracle import mock_prover as MP
from oracle import oracle as O

try:
    from tests.test_lookup_product import lookup_product
    from tests.test_permutation_product import _check_instances, assemble, column_list, facade_copies, sigma_value, _instance_values
except ImportError:   # another installed distribution named `tests` shadows this directory; pytest has put the directory itself on sys.path
    from test_lookup_product import lookup_product
    from test_permutation_product import _check_instances, assemble, column_list, facade_copies, sigma_value, _instance_values

P = O.P
R = O.R
R_INV = pow(R, -1, P)
M64 = (1 << 64) - 1
P3 = P >> 192
GP_TILE = 2048                                   # rows of a grand-product tile (grand_product.cuh)
SENT = 0x6B6B6B6B6B6B6B6B                        # guard fill of A', S'
SPREAD = 3

# configurations the planner accepts, one table size each ([64]-byte digests); minimum usable rows come from lookup_info()
RANGE_CFGS = {8: dict(lookup_bits=8, max_rows=1000), 11: dict(lookup_bits=11), 12: dict(lookup_bits=12), 13: dict(lookup_bits=13),
              16: dict(), 20: dict(lookup_bits=20)}
SPREAD_CFGS = {2: dict(lookup_bits=8, max_rows=1000, num_bits_lookup=2), 4: dict(lookup_bits=8, max_rows=1000, num_bits_lookup=4),
               8: dict(lookup_bits=8, max_rows=1000), 16: dict(num_bits_lookup=16)}


# ----------------------------------------------------------------------------------------------------------------
# restatements and generators
# ----------------------------------------------------------------------------------------------------------------
def permuted_from_counts(table_vals, counts, usable, order=None):
    """halo2 `permute_expression_pair`, literally, for an input column that holds table row r counts[r] times (sum == usable) against
    the table column `table_vals` (distinct canonical ints, in table-row order) padded to `usable` rows with its first row.
    The input sorted (np.repeat over the rows in ascending value), the first row of each run takes its own value, the leftover table
    elements in ascending order go to the repeated rows popped from the back.  Returns (A', S') as table-row indices.
    `order`: the table rows sorted by value, when the caller has it already."""
    n = len(table_vals)
    counts = np.asarray(counts, dtype=np.int64)
    assert counts.sum() == usable and len(counts) == n
    if order is None:
        order = np.array(sorted(range(n), key=table_vals.__getitem__), dtype=np.int64)   # sorted position -> table row
    mk = counts[order]
    a_pos = np.repeat(np.arange(n), mk)                  # sorted input, as sorted positions
    first = np.ones(usable, dtype=bool)
    first[1:] = a_pos[1:] != a_pos[:-1]
    table_mult = np.ones(n, dtype=np.int64)
    table_mult[np.flatnonzero(order == 0)] += usable - n   # the padding rows repeat table row 0
    leftover = np.repeat(np.arange(n), table_mult - (mk > 0))
    repeated = np.flatnonzero(~first)
    assert len(leftover) == len(repeated)
    s_pos = a_pos.copy()
    s_pos[repeated[::-1]] = leftover                     # repeated_rows.pop() while walking the leftover elements upwards
    return order[a_pos], order[s_pos]


def _mont_array(vals):
    """canonical ints -> [n, 4] u64 Montgomery limbs"""
    return np.frombuffer(b"".join((v * R % P).to_bytes(32, "little") for v in vals), dtype=np.uint64).reshape(-1, 4).copy()


def _int_of_limbs(x):
    return int(x[0]) | int(x[1]) << 64 | int(x[2]) << 128 | int(x[3]) << 192


# Montgomery representations (what the device adds and multiplies) on the edges of fr_add_dev / mont_mul_dev: p - 1, all-ones limbs,
# [~0, ~0, ~0, p3 - 1], R mod p (= 1), and pairs m, p - m whose sum lands exactly on p
EDGE_MONT = [0, 1, 2, P - 1, P - 2, M64, 1 << 64, P - M64, (1 << 128) - 1, 1 << 128, (1 << 192) - 1, 1 << 192, P - (1 << 192),
             ((P3 - 1) << 192) | ((1 << 192) - 1), R % P, P - R % P, (P - 1) // 2, (P + 1) // 2]
EDGE_CANON = [0, 1, 2, P - 1, P - 2, M64, 1 << 64, (1 << 64) + 1, 1 << 128, (P - 1) // 2, (P + 1) // 2]


def edge_values():
    """canonical ints < p: the values whose Montgomery form is in EDGE_MONT, then canonical edges"""
    out = []
    for v in [m * R_INV % P for m in EDGE_MONT] + EDGE_CANON:
        if v not in out:
            out.append(v)
    return out


EDGES = edge_values()
EDGES_M = _mont_array(EDGES)


def _rand(rng):
    return int.from_bytes(rng.bytes(32), "little") % P


def field_column(rng, n, avoid=(), edge_share=0.25):
    """n field elements: ([n, 4] u64 Montgomery limbs, canonical ints); a share of the rows (at random) an edge value, the rest random.
    No value is in `avoid` (a value that would make a term zero where the test does not want one)."""
    m = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    m[:, 3] %= np.uint64(P3)                               # < p3 * 2^192 < p
    e = rng.random(n) < edge_share
    m[e] = EDGES_M[rng.integers(0, len(EDGES), size=int(e.sum()))]
    vals = MP.canon_all(m)
    avoid = set(avoid)
    for i, v in enumerate(vals):
        while v in avoid:
            v = _rand(rng)
        if v != vals[i]:
            vals[i] = v
            m[i] = O.int_to_mont(v)
    return m, vals


def spread_table(theta, bits):
    """compressed spread table dense * theta + spread (halo2 `compress_expressions`), canonical, in table-row order"""
    return [(i * theta + LP.spread_bits(i, bits)) % P for i in range(1 << bits)]


def classify_theta(theta, bits):
    """rows of the compressed spread table that share limb 3, limbs 3..2, limbs 3..1 with another row; and whether two rows collide"""
    vals = spread_table(theta, bits)
    out = {}
    for name, shift in (("tie3", 192), ("tie32", 128), ("tie321", 64)):
        keys = [v >> shift for v in vals]
        cnt = {}
        for k in keys:
            cnt[k] = cnt.get(k, 0) + 1
        out[name] = sum(1 for k in keys if cnt[k] > 1)
    out["collide"] = len(set(vals)) < len(vals)
    return out


# candidate thetas that tie the top limbs of most rows (only the lower sort passes decide), and a random-looking one
TIE_THETAS = [0, 1, 2, 1 << 32, 1 << 64, (1 << 64) + 1, 1 << 128, 1 << 192, P - (1 << 64), P - (1 << 128), P - 5, P - 19,
              0x1D2C3B4A59687786 ** 4 % P]


def tie_thetas(bits):
    """the candidates that make no two rows of the 2^bits-row table collide (p - 5 does at 8 and 16 bits)"""
    return [t for t in TIE_THETAS if not classify_theta(t, bits)["collide"]]


def collision_thetas(bits):
    """thetas solved from i * theta + spread(i) == j * theta + spread(j): rows (0, 1), (0, n/2 + 1) (row 0 compresses to 0) and (n - 2, n - 1)"""
    n = 1 << bits
    sp = lambda x: LP.spread_bits(x, bits)
    return [(sp(j) - sp(i)) * pow((i - j) % P, -1, P) % P for i, j in ((0, 1), (0, n // 2 + 1), (n - 2, n - 1))]


def distributions(rng, n, usable):
    """name -> multiplicities of the n table rows summing to usable ('short': one row short)"""
    uni = lambda k, total: np.bincount(rng.integers(0, k, size=total), minlength=k).astype(np.int64)
    d = {}
    m = np.zeros(n, np.int64)
    m[1:] = uni(n - 1, usable)
    d["m0_zero"] = m
    m = np.ones(n, np.int64)
    m[0] += usable - n
    d["every_row_once"] = m
    m = np.zeros(n, np.int64)
    m[n - 1] = usable
    d["last_row_hot"] = m
    m = np.zeros(n, np.int64)
    m[n // 2] = usable
    d["middle_row_hot"] = m
    m = np.zeros(n, np.int64)
    m[1::2] = uni(n // 2, usable)
    d["alternating"] = m
    d["uniform"] = uni(n, usable)
    d["short"] = uni(n, usable - 1)
    return d


# ----------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------
def _literal(table_vals, counts, usable, rng):
    a = [table_vals[r] for r in np.repeat(np.arange(len(table_vals)), counts)]
    rng.shuffle(a)
    s = list(table_vals) + [table_vals[0]] * (usable - len(table_vals))
    return LP.permute_expression_pair(a, s, usable)


@pytest.mark.parametrize("seed", range(20))
def test_counts_restatement_equals_permute_expression_pair(seed):
    rng = np.random.default_rng(700 + seed)
    bits = int(rng.integers(1, 6))
    n = 1 << bits
    usable = n + int(rng.integers(0, 3 * n)) if seed % 4 else n   # every fourth case without padding rows
    if seed % 2:
        table = list(range(n))
    else:                                                         # a spread table: not sorted by row
        theta = _rand(rng)
        table = spread_table(theta, bits)
    dists = list(distributions(rng, n, usable).items())
    name, counts = dists[seed % len(dists)]
    if name == "short":
        counts = counts.copy()
        counts[int(rng.integers(0, n))] += 1
    a_rows, s_rows = permuted_from_counts(table, counts, usable)
    a_p, s_p = _literal(table, counts, usable, rng)
    assert [table[r] for r in a_rows] == a_p, name
    assert [table[r] for r in s_rows] == s_p, name


def test_edge_values_round_trip_through_montgomery_form():
    assert all(0 <= v < P for v in EDGES)
    for m, v in zip(EDGE_MONT, EDGES):
        if m * R_INV % P == v:
            assert _int_of_limbs(O.int_to_mont(v)) == m
    for v in EDGES:
        assert O.mont_to_int(O.int_to_mont(v)) == v
    limbs = [[int(x) for x in O.int_to_mont(v)] for v in EDGES]
    assert [M64, M64, M64, P3 - 1] in limbs and [M64, 0, 0, 0] in limbs
    assert _mont_array(EDGES).tolist() == limbs
    rng = np.random.default_rng(3)
    m, vals = field_column(rng, 4000, avoid=(1, 0))
    assert all(0 < v < P and v != 1 for v in vals) and MP.canon_all(m) == vals
    assert len({int(x) for x in m[:, 3]}) > 10 and any(v in EDGES for v in vals)


@pytest.mark.parametrize("bits", [8, 16])
def test_theta_classifier_backs_the_choices(bits):
    n = 1 << bits
    chosen = tie_thetas(bits)
    assert P - 5 not in chosen and len(chosen) == len(TIE_THETAS) - 1
    monotone = 0
    for theta in chosen:
        assert not classify_theta(theta, bits)["collide"], hex(theta)
        vals = spread_table(theta, bits)
        monotone += sorted(range(n), key=vals.__getitem__) == list(range(n))
    # the structured thetas leave only limb 0, 1 or 2 to decide for (almost) every row
    for theta in (0, 1, 2, 1 << 32, 1 << 64, (1 << 64) + 1, 1 << 128, P - (1 << 64), P - (1 << 128), P - 19):
        assert classify_theta(theta, bits)["tie3"] >= n - 2, hex(theta)
    for theta in (0, 1, 2, 1 << 32, P - 19):
        assert classify_theta(theta, bits)["tie321"] >= n - 2, hex(theta)
    # and some of them (p - 2^64, p - 2^128, p - 19) order the tied rows against their row index: a missing or wrong lower pass
    # changes the order
    assert monotone <= len(chosen) - 3
    for theta in collision_thetas(bits):
        assert classify_theta(theta, bits)["collide"], hex(theta)


# ----------------------------------------------------------------------------------------------------------------
# GPU helpers
# ----------------------------------------------------------------------------------------------------------------
_TABLES = {}


def _table(kind, bits, theta=None):
    """(canonical values in table-row order, their Montgomery limbs, the rows sorted by value) of a range or compressed spread table"""
    key = (kind, bits, theta)
    if key not in _TABLES:
        tv = list(range(1 << bits)) if kind == "range" else spread_table(theta, bits)
        _TABLES[key] = (tv, _mont_array(tv), np.array(sorted(range(1 << bits), key=tv.__getitem__), dtype=np.int64))
    return _TABLES[key]


def _np(t):
    return t.cpu().numpy().view(np.uint64)


def _mult_off(info, l):
    n_r = info["n_range_lookups"]
    return l * info["range_table_rows"] if l < n_r else n_r * info["range_table_rows"] + (l - n_r) * info["spread_table_rows"]


def _permute(pkg, cfg, mult, l, usable, thetas, per_inst):
    """h2sha_permute_lookup(_per_instance) into guard-filled A', S': (a, s) as [n, usable, 4] views, errors, and both guard bands intact"""
    import torch
    n = mult.shape[0]
    G = 1024
    dev = mult.device
    cells = n * usable * 4
    a = torch.full((cells + 2 * G,), SENT, dtype=torch.int64, device=dev)
    s = torch.full((cells + 2 * G,), SENT, dtype=torch.int64, device=dev)
    err = torch.zeros(n if per_inst else 1, dtype=torch.int32, device=dev)
    th = None
    if thetas is not None:
        th = np.ascontiguousarray(np.stack([O.int_to_mont(t) for t in thetas]) if per_inst else O.int_to_mont(thetas[0]), dtype=np.uint64)
    L = pkg.load_library()
    fn = L.h2sha_permute_lookup_per_instance if per_inst else L.h2sha_permute_lookup
    rc = fn(cfg._h, n, l, mult.data_ptr(), usable, th.ctypes.data if th is not None else None, a[G:].data_ptr(), s[G:].data_ptr(), err.data_ptr(),
            torch.cuda.current_stream(0).cuda_stream)
    assert rc == 0, L.h2sha_last_error().decode()
    torch.cuda.synchronize()
    guards = all(bool((t[:G] == SENT).all()) and bool((t[G + cells:] == SENT).all()) for t in (a, s))
    return a[G:G + cells].view(n, usable, 4), s[G:G + cells].view(n, usable, 4), err.cpu().numpy(), guards


def _expect_pair(table, counts, usable):
    tv, tm, order = table
    a_rows, s_rows = permuted_from_counts(tv, counts, usable, order)
    return tm[a_rows], tm[s_rows]


def _first_diff(got, want):
    bad = np.flatnonzero((got != want).any(-1))
    return int(bad[0]) if len(bad) else None


# ----------------------------------------------------------------------------------------------------------------
# GPU 1: permuted pair from synthetic multiplicities
# ----------------------------------------------------------------------------------------------------------------
_PERMUTE_CASES = [("range", b) for b in RANGE_CFGS] + [("spread", b) for b in SPREAD_CFGS]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,bits", _PERMUTE_CASES, ids=[f"{k}{b}" for k, b in _PERMUTE_CASES])
def test_permuted_pair_from_synthetic_multiplicities(pkg, kind, bits, monkeypatch):
    import torch
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0, **(RANGE_CFGS if kind == "range" else SPREAD_CFGS)[bits])
    info = cfg.lookup_info()
    n_r, n_s = info["n_range_lookups"], info["n_spread_lookups"]
    n_vals = info["range_table_rows" if kind == "range" else "spread_table_rows"]
    assert n_vals == 1 << bits
    l = n_r - 1 if kind == "range" else n_r + n_s - 1       # the last lookup of its kind: a nonzero offset in the multiplicity row
    off = _mult_off(info, l)
    # no padding rows where the planner allows it, padding otherwise
    usables = ([n_vals] if info["min_usable_rows"] <= n_vals else []) + ([info["min_usable_rows"] + 3] if bits < 20 else [])
    rng = np.random.default_rng(800 + bits + (0 if kind == "range" else 100))
    for usable in usables:
        dists = distributions(rng, n_vals, usable)
        names = list(dists)
        n = len(names)
        mult = torch.zeros((n, info["mult_words_per_instance"]), dtype=torch.int32, device=torch.device("cuda", 0))
        for i, name in enumerate(names):
            mult[i, off:off + n_vals] = torch.from_numpy(dists[name].astype(np.int32))
        if kind == "range":
            thetas_shared = thetas_pi = None
        else:
            thetas_pi = [_rand(rng) for _ in range(n)]
            thetas_shared = [thetas_pi[0]] * n
            assert not any(classify_theta(t, bits)["collide"] for t in thetas_pi)
        tune = [None, "lkinv=0,lktab=0"] if kind == "range" and bits == 16 else [None]
        for per_inst, thetas in ((False, thetas_shared), (True, thetas_pi)):
            if per_inst:   # a different distribution per instance than in the shared call: rotate the rows
                rot = [(i + 3) % n for i in range(n)]
                mult = mult[rot].contiguous()
                dist_of = [names[r] for r in rot]
            else:
                dist_of = names
            for t in (tune if not per_inst else [None]):
                if t:
                    monkeypatch.setenv("H2SHA_TUNE", t)   # the 2^16 range table through the generic two-level search of the spread tables
                a, s, err, guards = _permute(pkg, cfg, mult, l, usable, thetas, per_inst)
                if t:
                    monkeypatch.delenv("H2SHA_TUNE")
                what = f"usable {usable}, per_inst {per_inst}, tune {t}"
                assert guards, f"{what}: guard band overwritten"
                i_short = dist_of.index("short")
                if per_inst:
                    assert err.tolist() == [int(i == i_short) for i in range(n)], what
                else:
                    assert int(err[0]) == 1, what
                a_np, s_np = _np(a), _np(s)
                for i, name in enumerate(dist_of):
                    if name == "short":
                        assert (a_np[i] == SENT).all() and (s_np[i] == SENT).all(), f"{what}: the short instance was written"
                        continue
                    table = _table(kind, bits, None if kind == "range" else thetas[i])
                    want_a, want_s = _expect_pair(table, dists[name], usable)
                    d = _first_diff(a_np[i], want_a)
                    assert d is None, f"{what}, {name}: A' differs first at row {d}"
                    d = _first_diff(s_np[i], want_s)
                    assert d is None, f"{what}, {name}: S' differs first at row {d}"
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU 2: the per-instance spread sort at tied-limb thetas
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("bits", [8, 16])
def test_per_instance_spread_sort_at_tied_limb_thetas(pkg, bits):
    import torch
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0, **SPREAD_CFGS[bits])
    info = cfg.lookup_info()
    n_r = info["n_range_lookups"]
    l = n_r
    n_vals = 1 << bits
    usable = info["min_usable_rows"] + 1
    rng = np.random.default_rng(900 + bits)
    ties = tie_thetas(bits)
    collide = collision_thetas(bits)
    assert all(classify_theta(t, bits)["collide"] for t in collide)
    thetas = ties[:6] + collide[:1] + ties[6:] + collide[1:]
    bad = {i for i, t in enumerate(thetas) if t in collide}
    n = len(thetas)
    mult = torch.zeros((n, info["mult_words_per_instance"]), dtype=torch.int32, device=torch.device("cuda", 0))
    counts = [np.bincount(rng.integers(0, n_vals, size=usable), minlength=n_vals) for _ in range(n)]
    off = _mult_off(info, l)
    for i in range(n):
        mult[i, off:off + n_vals] = torch.from_numpy(counts[i].astype(np.int32))
    a, s, err = cfg.permute_lookup_per_instance(mult, l, usable, np.stack([O.int_to_mont(t) for t in thetas]))
    assert err.tolist() == [int(i in bad) for i in range(n)], "exactly the colliding thetas are counted"
    a_np, s_np = _np(a), _np(s)
    for i, theta in enumerate(thetas):
        if i in bad:
            continue
        want_a, want_s = _expect_pair(_table("spread", bits, theta), counts[i], usable)
        d = _first_diff(a_np[i], want_a)
        assert d is None, f"theta {theta:#x}: A' differs first at row {d}"
        d = _first_diff(s_np[i], want_s)
        assert d is None, f"theta {theta:#x}: S' differs first at row {d}"
        sa, ss = cfg.permute_lookup(mult[i:i + 1], l, usable, O.int_to_mont(theta))   # the host-sorted table of the shared call
        assert torch.equal(sa[0], a[i]) and torch.equal(ss[0], s[i]), f"theta {theta:#x}: shared call differs"
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU 3: the lookup grand product on synthetic columns
# ----------------------------------------------------------------------------------------------------------------
_PRODUCT_CASES = [("range", u, False) for u in ("min", 4095, 4096, 4097, 32 * GP_TILE, 33 * GP_TILE + 1, 65 * GP_TILE - 1)]
_PRODUCT_CASES += [("spread", 4097, False), ("spread", 33 * GP_TILE + 1, False), ("spread", "min", True), ("spread", 65 * GP_TILE - 1, True),
                   ("range", 4096, True)]
_SWEEP = ("min", 4097, 33 * GP_TILE + 1, 4096)                 # one instance per zero-denominator row at these sizes


def _challenge_pool(rng):
    return [1, P - 1, EDGES[3], EDGES[5], EDGES[7], EDGES[11], EDGES[13], _rand(rng)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,usable,per_inst", _PRODUCT_CASES, ids=[f"{k}-{u}-{'pi' if p else 'shared'}" for k, u, p in _PRODUCT_CASES])
def test_lookup_product_on_synthetic_columns(pkg, kind, usable, per_inst):
    """z of every instance == lookup_product in Python ints; errors == instances whose restated z[U] != 1.  Instance 0 holds a
    consistent pair (A' = A, S' = S under one row permutation: z[U] == 1), instance 1 random and edge values, instance 2 a zero
    numerator and three zero denominators, the others one zero denominator each at a segment (8 rows), warp (256), tile (2048)
    edge, row 0 or row U - 1."""
    import torch
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0, lookup_bits=8, max_rows=1000)
    info = cfg.lookup_info()
    n_r = info["n_range_lookups"]
    U = info["min_usable_rows"] if usable == "min" else usable
    assert U >= info["min_usable_rows"]
    l = n_r - 1 if kind == "range" else n_r
    lay = cfg.layout
    rng = np.random.default_rng(1000 + U + (7 if kind == "spread" else 0) + (3 if per_inst else 0))
    zero_rows = [r for r in (0, 7, 8, 255, 256, 2047, 2048, U - 1) if r < U]
    n = 3 + (len(zero_rows) if usable in _SWEEP else 0)
    pool = _challenge_pool(rng)
    if per_inst:   # a different (beta, gamma, theta) per instance, edges included; beta = 0 and gamma = 0 zero every row from the first 0 of A / S
        betas = [pool[(i + 1) % len(pool)] for i in range(n)]
        gammas = [pool[(i + 3) % len(pool)] for i in range(n)]
        thetas = [pool[(i + 5) % len(pool)] for i in range(n)]
        betas[-1], gammas[-2] = 0, 0
    else:
        betas, gammas, thetas = [EDGES[5]] * n, [EDGES[11]] * n, [EDGES[13]] * n
    bits = 8
    gate, lookup, spread = cfg.alloc_outputs(n)
    a_p = torch.empty((n, U, 4), dtype=torch.int64, device=gate.device)
    s_p = torch.empty_like(a_p)
    want_z, want_err = [], 0
    if kind == "range":
        used = min(lay.n_lookup_cells - l * 1000, 1000)
        table = list(range(1 << bits))
    else:
        nc = lay.n_spread_cols // 2
        used = (lay.n_spread_limbs + nc - 1) // nc
    for i in range(n):
        beta, gamma, theta = betas[i], gammas[i], thetas[i]
        if kind == "spread":
            table = spread_table(theta, bits)
        s = table + [0] * (U - len(table))
        avoid_a = [(-beta) % P]
        if kind == "range":
            am, av = field_column(rng, used, avoid=avoid_a)
            lookup[i, l, :used] = torch.from_numpy(am.view(np.int64))
            a = av + [0] * (U - used)
        else:   # dense and spread cells: A = dense * theta + spread
            dm, dv = field_column(rng, used)
            sm, sv = field_column(rng, used)
            for r in range(used):
                while (dv[r] * theta + sv[r] + beta) % P == 0:
                    sv[r] = _rand(rng)
                    sm[r] = O.int_to_mont(sv[r])
            if i == 2:   # a zero numerator: the spread cell that makes A + beta = 0
                sv[used // 2] = (-(dv[used // 2] * theta) - beta) % P
                sm[used // 2] = O.int_to_mont(sv[used // 2])
            spread[i, 0, :used] = torch.from_numpy(dm.view(np.int64))
            spread[i, nc, :used] = torch.from_numpy(sm.view(np.int64))
            a = [(d * theta + x) % P for d, x in zip(dv, sv)] + [0] * (U - used)
        if i == 0:
            perm = rng.permutation(U)
            ap = [a[j] for j in perm]
            sp = [s[j] for j in perm]
            apm, spm = _mont_array(ap), _mont_array(sp)
        else:
            apm, ap = field_column(rng, U, avoid=avoid_a)
            spm, sp = field_column(rng, U, avoid=[(-gamma) % P])
        zs = [] if i < 2 else ([zero_rows[2], zero_rows[4], zero_rows[-1]] if i == 2 else [zero_rows[i - 3]])
        for r in zs:
            ap[r] = (-beta) % P
            apm[r] = O.int_to_mont(ap[r])
        if i == 2 and kind == "range":   # a zero numerator: the lookup cell that makes A + beta = 0
            a[used // 2] = (-beta) % P
            lookup[i, l, used // 2] = torch.from_numpy(O.int_to_mont(a[used // 2]).view(np.int64))
        a_p[i] = torch.from_numpy(apm.view(np.int64))
        s_p[i] = torch.from_numpy(spm.view(np.int64))
        want = lookup_product(a, s, ap, sp, beta, gamma, U)
        if i == 0:
            assert want[U] == 1 or any(w == 0 for w in want)
        want_z.append(want)
        want_err += want[U] != 1
    res = pkg.BatchResult(None, None, gate, lookup, spread)
    mont = lambda xs: np.stack([O.int_to_mont(x) for x in xs])
    if per_inst:
        z, err = cfg.lookup_product_per_instance(res, l, a_p, s_p, U, mont(betas), mont(gammas), mont(thetas) if kind == "spread" else None)
        assert err.tolist() == [int(w[U] != 1) for w in want_z]
    else:
        z, err = cfg.lookup_product(res, l, a_p, s_p, U, O.int_to_mont(betas[0]), O.int_to_mont(gammas[0]),
                                    O.int_to_mont(thetas[0]) if kind == "spread" else None)
        assert err == want_err
    assert tuple(z.shape) == (n, U + 1, 4)
    z_np = _np(z)
    for i in range(n):
        got = MP.canon_all(z_np[i])
        if got != want_z[i]:
            d = next(j for j, (x, y) in enumerate(zip(got, want_z[i])) if x != y)
            pytest.fail(f"instance {i}: z differs first at row {d} of {U + 1}")
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU 4: the permutation product on a synthetic witness
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("usable", [35 * GP_TILE - 1, 35 * GP_TILE], ids=["U+1=35tiles", "U+1=35tiles+1"])
def test_permutation_product_on_a_synthetic_witness(pkg, usable):
    """edge and random values in every gate, lookup and spread cell: every copy is broken, most rows hold no moved cell (the constant
    store of k_product_fill), and instance 2 has a zero denominator at a moved cell on a tile edge, a sum that lands exactly on p"""
    import torch
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0, build_shape=True)
    lay = cfg.layout
    columns = column_list(lay, False)
    m, k = 3, 17
    try:
        cfg.permutation_mapping(columns, usable, columns_per_chunk=m)
    except pkg.EngineError as ex:
        pytest.skip(f"the permutation mapping refuses usable_rows = {usable}: {ex}")
    n = 3
    rng = np.random.default_rng(1100 + usable)
    gate, lookup, spread = cfg.alloc_outputs(n)
    for buf in (gate, lookup, spread):
        vals, _ = field_column(rng, buf.numel() // 4)
        buf.copy_(torch.from_numpy(vals.view(np.int64)).view(buf.shape))
    res = pkg.BatchResult(None, None, gate, lookup, spread)
    asm = assemble(columns, usable, facade_copies(cfg, False))
    betas = [EDGES[5], _rand(rng), EDGES[11]]
    gammas = [EDGES[13], _rand(rng), 0]
    c, r = columns.index((SPREAD, 1)), GP_TILE - 1           # the only column of the last chunk: v of that row is one sum, not a product
    assert asm.mapping[c * usable + r] != c * usable + r
    values = _instance_values(cfg, res, 2, columns, usable)
    gammas[2] = (-(values[c][r] + betas[2] * sigma_value(asm, c, r, k))) % P
    mont = lambda xs: np.stack([O.int_to_mont(x) for x in xs])
    z, err = cfg.permutation_product_per_instance(res, columns, usable, mont(betas), mont(gammas), columns_per_chunk=m)
    assert tuple(z.shape) == (n, -(-len(columns) // m), usable + 1, 4)
    for i in range(n):
        _check_instances(cfg, res, z, (i,), columns, usable, k, m, betas[i], gammas[i], asm)
    last = [_int_of_limbs(x) * R_INV % P for x in _np(z[:, -1, usable])]
    assert err.tolist() == [int(x != 1) for x in last]
    assert last[2] == 0
    zs, e = cfg.permutation_product(res, columns, usable, O.int_to_mont(betas[0]), O.int_to_mont(gammas[0]), columns_per_chunk=m)
    assert torch.equal(zs[0], z[0]), "shared call with instance 0's challenges"
    assert e == n                                             # random cells break every copy
    cfg.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU 5: near misses of table membership
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_near_miss_table_membership(pkg):
    """cells right in limb 0 and wrong above it, p - v, n_vals, and spread halves off by 2^64 or one bit, each in its own instance of a
    real cfg2 batch: the multiplicities bin exactly the valid ones, not_in_table and the MockProver's lookup classes count the rest"""
    import torch
    n_vals = 1 << 16
    range_cases = [(n_vals - 1, True), (n_vals, False), (1 << 64, False), ((1 << 64) + 3, False), (P - 1, False), (P - 3, False)]
    sp = lambda x: LP.spread_bits(x, 9)
    d = 0x5B
    spread_cases = [((d, sp(d)), True), ((d, sp(d) + (1 << 64)), False), ((d + (1 << 64), sp(d)), False), ((256, sp(256)), False),
                    ((d, sp(d) ^ 1), False)]
    n = len(range_cases) + len(spread_cases)
    rng = np.random.default_rng(1200)
    cfg = pkg.Sha256DynamicConfig.configure([64], device=0)
    res = cfg.digest_batch([[bytes(rng.integers(0, 256, size=int(rng.integers(0, 56)), dtype=np.uint8))] for _ in range(n)])
    info = cfg.lookup_info()
    nc = cfg.layout.n_spread_cols // 2
    usable = (1 << 17) - 6
    m0, bad0 = cfg.lookup_multiplicities(res, usable)
    counts0, _ = cfg.check_batch_per_instance(res)
    assert bad0 == 0 and not counts0[:, 2:4].any()
    want = m0.cpu().numpy().astype(np.int64)
    cell = lambda v: torch.from_numpy(O.int_to_mont(v).view(np.int64)).to(res.lookup.device)
    row = 17
    for i, (v, ok) in enumerate(range_cases):
        old = O.mont_to_int(_np(res.lookup[i, 0, row]))
        res.lookup[i, 0, row] = cell(v)
        want[i, old] -= 1
        if ok:
            want[i, v] += 1
    off = info["n_range_lookups"] * n_vals
    row = 9
    for j, ((dv, sv), ok) in enumerate(spread_cases):
        i = len(range_cases) + j
        old = O.mont_to_int(_np(res.spread[i, 0, row]))
        res.spread[i, 0, row] = cell(dv)
        res.spread[i, nc, row] = cell(sv)
        want[i, off + old] -= 1
        if ok:
            want[i, off + dv] += 1
    m1, bad1 = cfg.lookup_multiplicities(res, usable)
    n_bad = sum(not ok for _, ok in range_cases + spread_cases)
    assert bad1 == n_bad
    got = m1.cpu().numpy().astype(np.int64)
    for i in range(n):
        assert (got[i] == want[i]).all(), f"instance {i}: multiplicities"
    counts, _ = cfg.check_batch_per_instance(res)
    want_range = [int(not ok) for _, ok in range_cases] + [0] * len(spread_cases)
    want_spread = [0] * len(range_cases) + [int(not ok) for _, ok in spread_cases]
    assert counts[:, 2].tolist() == want_range and counts[:, 3].tolist() == want_spread
    cfg.close()
