"""Permutation argument (copy constraints) of the chip: the keygen mapping (h2sha_get_permutation) and the product columns z on the
device (h2sha_permutation_product).  halo2_proofs `permutation::keygen::Assembly::{new, copy}`, the sigma values and
`permutation::prover` `Argument::commit` are restated below over canonical ints (`Assembly`, `sigma_value`, `permutation_commit`,
ff's `batch_invert`); that restatement is the reference.  Parity against the halo2_proofs crate itself is unpinned.

CPU part: the constants, the restatement closes on an oracle witness, the engine's mapping equals the restatement fed with the
copy / instance calls the C++ facade (tests/cpp/test_chip_api.cc, keygen case) records, other column orders and chunk sizes,
argument refusals.  GPU part: z bit-exact against the restatement on five configurations, batch slices, corruption, zero terms,
the instance binding."""
import bisect
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import mock_prover as MP
from oracle import oracle as O

P = O.P
DELTA = 0x09226B6E22C6F0CA64EC26AAD4C86E715B5F898E5E963F25870E56BBE533E9A2          # 7^(2^28), halo2curves bn256::Fr::DELTA
ROOT_OF_UNITY = 0x03DDB9F5166D18B798865EA93DD31F743215CF6DD39329C8D34F1ED960C37C9C  # 7^((p - 1) / 2^28), S = 28
GATE, LOOKUP, DENSE, SPREAD, FIXED, INSTANCE = 0, 1, 2, 3, 4, 6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_ROWS = (1 << 17) - 9


# ----------------------------------------------------------------------------------------------------------------
# the restatement
# ----------------------------------------------------------------------------------------------------------------
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


class Assembly:
    """halo2_proofs plonk/permutation/keygen.rs `Assembly` over `n` rows; a cell (column position c, row r) is the int c * n + r."""

    def __init__(self, columns, n):
        self.columns = [tuple(c) for c in columns]
        self.n = n
        self.mapping = list(range(len(columns) * n))   # mapping[c][r] = (c, r)
        self.aux = list(self.mapping)                   # aux[c][r] = (c, r)
        self.sizes = [1] * (len(columns) * n)

    def cell(self, column, row):
        assert row < self.n, "BoundsFailure"
        return self.columns.index(tuple(column)) * self.n + row   # ColumnNotInPermutation raises here

    def copy(self, left_column, left_row, right_column, right_row):
        l, r = self.cell(left_column, left_row), self.cell(right_column, right_row)
        left_cycle, right_cycle = self.aux[l], self.aux[r]
        if left_cycle == right_cycle:
            return
        if self.sizes[left_cycle] < self.sizes[right_cycle]:
            left_cycle, right_cycle = right_cycle, left_cycle
        self.sizes[left_cycle] += self.sizes[right_cycle]
        i = right_cycle
        while True:
            self.aux[i] = left_cycle
            i = self.mapping[i]
            if i == right_cycle:
                break
        self.mapping[l], self.mapping[r] = self.mapping[r], self.mapping[l]


def omega_of(k):
    return pow(ROOT_OF_UNITY, 1 << (28 - k), P)


def sigma_value(asm, c, r, k):
    """sigma_c(w^r) = delta^c' w^r' with (c', r') = mapping[c][r] (keygen `build_pk`)"""
    t = asm.mapping[c * asm.n + r]
    return pow(DELTA, t // asm.n, P) * pow(omega_of(k), t % asm.n, P) % P


def permutation_commit(values, asm, m, beta, gamma, k):
    """halo2 `permutation::prover` `Argument::commit` without the blinding rows: the z column of every chunk of m columns,
    rows 0 .. U (U = asm.n usable rows).  values[c]: U canonical ints of column c."""
    U = asm.n
    omega = omega_of(k)
    wpow = [1] * U
    for i in range(1, U):
        wpow[i] = wpow[i - 1] * omega % P
    dpow = [pow(DELTA, c, P) for c in range(len(values))]
    zs, last_z, deltaomega = [], 1, 1
    for c0 in range(0, len(values), m):
        cols = range(c0, min(len(values), c0 + m))
        modified = [1] * U
        for c in cols:   # denominators
            vals, mp = values[c], asm.mapping
            for i in range(U):
                t = mp[c * U + i]
                perm = dpow[t // U] * wpow[t % U]
                modified[i] = modified[i] * ((beta * perm + gamma + vals[i]) % P) % P
        batch_invert(modified)
        for c in cols:   # numerators
            vals, do = values[c], deltaomega
            for i in range(U):
                modified[i] = modified[i] * ((do * beta + gamma + vals[i]) % P) % P
                do = do * omega % P
            deltaomega = deltaomega * DELTA % P
        z = [last_z]
        for row in range(1, U + 1):
            z.append(z[row - 1] * modified[row - 1] % P)
        zs.append(z)
        last_z = z[U]
    return zs


# ----------------------------------------------------------------------------------------------------------------
# the chip's copy calls in facade order (csrc/chip_api.hpp assign_digest / RangeConfig::finalize, test_chip_api.cc instance binding)
# ----------------------------------------------------------------------------------------------------------------
def facade_copies(cfg, bind, num_fixed=1, max_rows=MAX_ROWS):
    lay, sh, rg = cfg.layout, cfg.shape(), cfg.digest_ranges()
    br = [int(b) for b in cfg.breaks()]
    nc = lay.n_spread_cols // 2

    def gate(s):
        c = bisect.bisect_right(br, s) - 1
        return (GATE, c, s - br[c])

    fixed = lambda k: (FIXED, k % num_fixed, k // num_fixed)
    out = []
    for d in range(len(rg)):
        for a_kind, a, b_kind, b in sh.copies.tolist():
            if a_kind == 0 and rg[d][0] <= a < rg[d][1]:
                out.append((gate(a), gate(b) if b_kind == 0 else fixed(b)))
        for n in range(int(rg[d][4]), int(rg[d][5])):
            out.append(((DENSE, n % nc, n // nc), gate(int(sh.limb_dense_src[n]))))
            out.append(((SPREAD, n % nc, n // nc), gate(int(sh.limb_spread_src[n]))))
    for k, src in enumerate(sh.lookup_src.tolist()):
        out.append(((LOOKUP, k // max_rows, k % max_rows), gate(src)))
    if bind:
        for d in range(len(rg)):
            for i, s in enumerate(cfg.handles(d).output_bytes.tolist()):
                out.append((gate(s), (INSTANCE, 0, 32 * d + i)))
    return out


def assemble(columns, usable, copies):
    asm = Assembly(columns, usable)
    for (lk, li, lr), (rk, ri, rr) in copies:
        asm.copy((lk, li), lr, (rk, ri), rr)
    return asm


def column_list(lay, bind, order=0):
    g = [(GATE, i) for i in range(lay.n_gate_cols)]
    lk = [(LOOKUP, i) for i in range(lay.n_lookup_cols)]
    nc = lay.n_spread_cols // 2
    de, sp = [(DENSE, i) for i in range(nc)], [(SPREAD, i) for i in range(nc)]
    inst = [(INSTANCE, 0)] if bind else []
    if order == 0:
        return g + lk + [(FIXED, 0)] + de + sp + inst
    return inst + sp[::-1] + [(FIXED, 0)] + de + lk + g[::-1]


def needed_rows(cfg, max_rows=MAX_ROWS):
    lay = cfg.layout
    br = [int(b) for b in cfg.breaks()] + [lay.n_gate_cells]
    nc = lay.n_spread_cols // 2
    return max(max(b - a for a, b in zip(br, br[1:])), min(lay.n_lookup_cells, max_rows), -(-lay.n_spread_limbs // nc),
               lay.n_fixed, 32 * lay.n_digests)


def usable_for(cfg, max_rows=MAX_ROWS):
    """(usable_rows, k): the smallest domain with 5 blinding rows that holds every assigned cell"""
    need, k = needed_rows(cfg, max_rows), 1
    while (1 << k) - 6 < need:
        k += 1
    return (1 << k) - 6, k


def witness_columns(columns, usable, gate, lookup, dense, spread, consts, digest_bytes, max_rows=MAX_ROWS, num_fixed=1):
    """values[c] (U canonical ints) of every listed column from one instance's cells: gate [cols][rows], lookup [cols][rows],
    dense / spread [cols][rows] canonical ints, consts canonical (first-use order), digest_bytes (the instance column)"""
    out = []
    for kind, idx in columns:
        v = [0] * usable
        if kind == GATE:
            src = gate[idx]
        elif kind == LOOKUP:
            src = lookup[idx]
        elif kind == DENSE:
            src = dense[idx]
        elif kind == SPREAD:
            src = spread[idx]
        elif kind == FIXED:
            src = consts[idx::num_fixed]
        else:
            src = list(digest_bytes)
        v[:len(src)] = src[:usable]
        out.append(v)
    return out


def _rand(rng):
    return int.from_bytes(rng.bytes(32), "little") % P


def _engine_mapping(cfg, columns, usable, **kw):
    m = cfg.permutation_mapping(columns, usable, **kw).astype(np.int64)
    return (m[..., 0] * usable + m[..., 1]).reshape(-1).tolist()


# ----------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------
def test_constants():
    assert DELTA == pow(7, 1 << 28, P)
    assert ROOT_OF_UNITY == pow(7, (P - 1) >> 28, P) and (P - 1) % (1 << 28) == 0
    assert pow(ROOT_OF_UNITY, 1 << 28, P) == 1 and pow(ROOT_OF_UNITY, 1 << 27, P) != 1
    assert pow(DELTA, 1 << 28, P) != 1   # DELTA generates no subgroup of the 2-adic roots: the cosets delta^j H are distinct


def _oracle_witness(cfg, sizes, msgs, columns, usable, bind):
    reg = O.synthesize(O.OracleConfig(max_variable_byte_sizes=tuple(sizes)), msgs)
    lay = cfg.layout
    canon = MP.canon_all
    g = canon(reg.gate)
    br = [int(b) for b in reg.breaks] + [len(g)]
    gate = [g[br[c]:br[c + 1]] for c in range(lay.n_gate_cols)]
    lk = [g[i] for i in reg.lookup_idx.tolist()]
    lookup = [lk[c * MAX_ROWS:(c + 1) * MAX_ROWS] for c in range(lay.n_lookup_cols)]
    nc = lay.n_spread_cols // 2
    dn, sp = canon(reg.dense), canon(reg.spread)
    dense = [dn[c::nc] for c in range(nc)]
    spread = [sp[c::nc] for c in range(nc)]
    bts = b"".join(reg.digests) if bind else b""
    return witness_columns(columns, usable, gate, lookup, dense, spread, canon(reg.consts), bts), reg


def test_restatement_closes_on_an_oracle_witness(pkg):
    sizes = [64]
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=-1, build_shape=True)
    usable, k = (1 << 17) - 6, 17
    columns = column_list(cfg.layout, False)
    asm = assemble(columns, usable, facade_copies(cfg, False))
    values, _ = _oracle_witness(cfg, sizes, [b"abc"], columns, usable, False)
    rng = np.random.default_rng(7)
    beta, gamma = _rand(rng), _rand(rng)
    zs = permutation_commit(values, asm, 3, beta, gamma, k)
    assert len(zs) == 3 and zs[0][0] == 1 and zs[-1][usable] == 1
    assert all(zs[h][usable] == zs[h + 1][0] for h in range(2))
    # one copied cell changed: a lookup-column cell no longer equals the gate cell it copies
    c = columns.index((LOOKUP, 0))
    values[c][100] = (values[c][100] + 1) % P
    assert permutation_commit(values, asm, 3, beta, gamma, k)[-1][usable] != 1
    cfg.close()


def _build_chip_api(pkg):
    exe = os.path.join(ROOT, "tests", "cpp", "_build", "test_chip_api")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    libdir = os.path.dirname(pkg.LIB_PATH)
    subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-std=c++17", "-O1", "-o", exe, os.path.join(ROOT, "tests", "cpp", "test_chip_api.cc"),
                           "-L" + libdir, "-lh2sha_b200", "-Xlinker", "-rpath," + libdir, "-cudart", "shared"])
    return exe


def _recorded_copies(path):
    """the constrain_equal (tag 4) and instance (tag 6) events of the recorder, in call order"""
    w = np.fromfile(path, dtype=np.uint32)
    out, i = [], 0
    while i < len(w):
        t = int(w[i])
        if t == 1:
            i += 5 + (8 if int(w[i + 4]) else 0)
        elif t == 2:
            i += 11
        elif t == 3:
            i += 3
        elif t == 4:
            a = [int(x) for x in w[i + 1:i + 7]]
            out.append(((a[0], a[1], a[2]), (a[3], a[4], a[5]))); i += 7
        elif t == 5:
            ln, nc, nr = (int(x) for x in w[i + 1:i + 4]); i += 4 + ln + 2 * nc * nr
        elif t == 6:
            kind, idx, row, j = (int(x) for x in w[i + 1:i + 5])
            out.append(((kind, idx, row), (INSTANCE, 0, j))); i += 5   # layouter.constrain_instance(cell, instance, j)
        else:
            raise AssertionError(f"bad event tag {t} at word {i}")
    return out


def test_keygen_mapping_equals_the_restatement_of_the_recorded_facade_calls(pkg, tmp_path):
    """the TestCircuit through the C++ facade (plan-only keygen replay): its recorded constrain_equal / constrain_instance calls fed
    to the restated Assembly give the mapping h2sha_get_permutation computes, and the Python facade order here is that order"""
    exe = _build_chip_api(pkg)
    out = subprocess.run([exe, str(tmp_path / "k.bin"), "0"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    recorded = _recorded_copies(tmp_path / "k.bin")
    cfg = pkg.Sha256DynamicConfig.configure([128, 128], device=-1, build_shape=True)
    assert facade_copies(cfg, True) == recorded
    usable = (1 << 17) - 6
    columns = column_list(cfg.layout, True)
    asm = assemble(columns, usable, recorded)
    assert _engine_mapping(cfg, columns, usable, columns_per_chunk=2, bind_output_bytes=True) == asm.mapping
    moved = sum(1 for i, t in enumerate(asm.mapping) if t != i)
    assert moved == 326255
    cfg.close()


@pytest.mark.parametrize("kw", [
    dict(sizes=[64], bind=False, order=1, chunk=1),
    dict(sizes=[64], bind=True, order=0, chunk=3),
    dict(sizes=[128, 128], bind=True, order=1, chunk=2),
    dict(sizes=[320], bind=False, order=0, chunk=2, max_rows=9973),
    dict(sizes=[192], bind=False, order=1, chunk=3, lookup_bits=9, num_bits_lookup=4, num_advice_columns=3),
], ids=["cfg2-order1-m1", "cfg2-bind-m3", "128x128-order1-m2", "320_wraps", "9bit-3cols"])
def test_mapping_for_other_column_orders_and_chunks(pkg, kw):
    kw = dict(kw)
    sizes, bind, order, chunk = kw.pop("sizes"), kw.pop("bind"), kw.pop("order"), kw.pop("chunk")
    max_rows = kw.get("max_rows", MAX_ROWS)
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=-1, build_shape=True, **kw)
    usable, k = usable_for(cfg, max_rows)
    columns = column_list(cfg.layout, bind, order)
    asm = assemble(columns, usable, facade_copies(cfg, bind, max_rows=max_rows))
    assert _engine_mapping(cfg, columns, usable, columns_per_chunk=chunk, bind_output_bytes=bind) == asm.mapping
    if sizes == [64] and not bind:
        assert sum(1 for i, t in enumerate(asm.mapping) if t != i) == 81862
    cfg.close()


def test_two_fixed_columns_take_the_constants_round_robin(pkg):
    cfg = pkg.Sha256DynamicConfig.configure([64], device=-1, build_shape=True)
    usable = (1 << 17) - 6
    columns = column_list(cfg.layout, False) + [(FIXED, 1)]
    asm = assemble(columns, usable, facade_copies(cfg, False, num_fixed=2))
    assert _engine_mapping(cfg, columns, usable, columns_per_chunk=3, num_fixed=2) == asm.mapping
    with pytest.raises(pkg.EngineError):   # constants in fixed column 1, which is not listed
        cfg.permutation_mapping(column_list(cfg.layout, False), usable, columns_per_chunk=3, num_fixed=2)
    cfg.close()


def test_argument_refusals(pkg):
    cfg = pkg.Sha256DynamicConfig.configure([128, 128], device=-1, build_shape=True)
    lay = cfg.layout
    usable = (1 << 17) - 6
    cols = column_list(lay, False)
    ok = dict(columns_per_chunk=2)
    cfg.permutation_mapping(cols, usable, **ok)
    bad = [
        (cols[1:], ok),                                        # gate column 0 missing
        ([c for c in cols if c[0] != SPREAD], ok),             # spread columns missing
        ([c for c in cols if c[0] != FIXED], ok),              # the constants column missing
        (cols + [cols[0]], ok),                                # listed twice
        (cols + [(GATE, lay.n_gate_cols)], ok),                # index out of range
        (cols + [(DENSE, lay.n_spread_cols // 2)], ok),
        (cols + [(5, 0)], ok),                                 # selector columns have no equality
        (cols, dict(columns_per_chunk=0)),
        (cols, dict(columns_per_chunk=2, bind_output_bytes=True)),            # binding without the instance column
        (cols + [(INSTANCE, 0)], ok),                                         # instance column without the binding
        (cols, dict(columns_per_chunk=2, k=16)),                              # 2^k too small for usable_rows
    ]
    for columns, kw in bad:
        with pytest.raises(pkg.EngineError) as ex:
            cfg.permutation_mapping(columns, usable, **kw)
        assert ex.value.code == pkg.H2SHA_EINVAL, (columns, kw)
    with pytest.raises(pkg.EngineError):                       # a copied cell above usable_rows
        cfg.permutation_mapping(cols, 1000, **ok)
    # the device product: argument checks first, then no CPU path
    L = pkg.load_library()
    d, keep = cfg._perm_desc(cols, 1, 2, False, 0)
    buf = (C.c_uint64 * 8)()
    one = O.int_to_mont(1)
    unreduced = np.array([0xFFFFFFFFFFFFFFFF] * 4, dtype=np.uint64)
    args = lambda b: (cfg._h, 1, C.byref(d), usable, buf, buf, buf, None, b.ctypes.data, one.ctypes.data, buf, None, None)
    assert L.h2sha_permutation_product(*args(unreduced)) == pkg.H2SHA_EINVAL
    assert L.h2sha_permutation_product(*args(one)) == pkg.H2SHA_ECUDA
    d0, keep0 = cfg._perm_desc(cols, 1, 0, False, 0)
    assert L.h2sha_permutation_product(cfg._h, 1, C.byref(d0), usable, buf, buf, buf, None, one.ctypes.data, one.ctypes.data, buf, None,
                                       None) == pkg.H2SHA_EINVAL
    cfg.close()
    plain = pkg.Sha256DynamicConfig.configure([64], device=-1)   # no build_shape: no copy constraints to replay
    with pytest.raises(pkg.EngineError):
        plain.permutation_mapping(column_list(plain.layout, False), usable, columns_per_chunk=2)
    plain.close()


# ----------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------
def _canon(t):
    return MP.canon_all(t.cpu().numpy().view(np.uint64).reshape(-1, 4))


def _batch(pkg, sizes, n, seed, **kw):
    cfg = pkg.Sha256DynamicConfig.configure(sizes, device=0, build_shape=True, **kw)
    rng = np.random.default_rng(seed)
    msgs = [[bytes(rng.integers(0, 256, int(rng.integers(0, s - 8)), dtype=np.uint8)) for s in sizes] for _ in range(n)]
    return cfg, cfg.digest_batch(msgs), rng


def _instance_values(cfg, res, inst, columns, usable, max_rows=MAX_ROWS, num_fixed=1):
    lay = cfg.layout
    br = [int(b) for b in cfg.breaks()] + [lay.n_gate_cells]
    gate = [_canon(res.gate[inst, c, :br[c + 1] - br[c]]) for c in range(lay.n_gate_cols)]
    lookup = []
    for c in range(lay.n_lookup_cols):
        used = max(0, min(max_rows, lay.n_lookup_cells - c * max_rows))
        lookup.append(_canon(res.lookup[inst, c, :used]))
    nc = lay.n_spread_cols // 2
    used = lambda c: (lay.n_spread_limbs - c + nc - 1) // nc if lay.n_spread_limbs > c else 0
    dense = [_canon(res.spread[inst, c, :used(c)]) for c in range(nc)]
    spread = [_canon(res.spread[inst, nc + c, :used(c)]) for c in range(nc)]
    consts = [int(x[0]) | int(x[1]) << 64 | int(x[2]) << 128 | int(x[3]) << 192 for x in cfg.shape().fixed]
    D = lay.n_digests
    bts = res.digests[inst * D:(inst + 1) * D].reshape(-1).tolist() if res.digests is not None else []
    return witness_columns(columns, usable, gate, lookup, dense, spread, consts, bts, max_rows, num_fixed)


def _check_instances(cfg, res, z, insts, columns, usable, k, m, beta, gamma, asm, max_rows=MAX_ROWS):
    for inst in insts:
        values = _instance_values(cfg, res, inst, columns, usable, max_rows)
        want = permutation_commit(values, asm, m, beta, gamma, k)
        got = _canon(z[inst])
        flat = [x for zc in want for x in zc]
        assert got == flat, f"instance {inst}: z differs (first at {next(i for i, (a, b) in enumerate(zip(got, flat)) if a != b)})"


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [
    dict(sizes=[64], n=48, bind=False, m=3, check=(0, 47)),                                  # config 2 shape
    dict(sizes=[128, 128], n=3, bind=True, m=2, check=(1,)),                                 # the reference's TestCircuit
    dict(sizes=[320], n=3, bind=False, m=2, check=(2,), max_rows=9973),                      # two lookup columns
    dict(sizes=[192], n=3, bind=False, m=3, check=(0,), lookup_bits=9, num_bits_lookup=4, num_advice_columns=3),
    dict(sizes=[64], n=2, bind=True, m=4, check=(1,), num_bits_lookup=16),                   # 16-bit limbs
], ids=["cfg2", "128x128", "320_wraps", "9bit-3cols", "16bit-limbs"])
def test_product_matches_the_restatement(pkg, kw):
    kw = dict(kw)
    sizes, n, bind, m, check = (kw.pop(x) for x in ("sizes", "n", "bind", "m", "check"))
    max_rows = kw.get("max_rows", MAX_ROWS)
    cfg, res, rng = _batch(pkg, sizes, n, 51, **kw)
    usable, k = usable_for(cfg, max_rows)
    columns = column_list(cfg.layout, bind, order=len(sizes) % 2)
    beta, gamma = _rand(rng), _rand(rng)
    z, errors = cfg.permutation_product(res, columns, usable, O.int_to_mont(beta), O.int_to_mont(gamma), columns_per_chunk=m,
                                        bind_output_bytes=bind, digests=res.digests if bind else None)
    assert errors == 0
    assert tuple(z.shape) == (n, -(-len(columns) // m), usable + 1, 4)
    asm = assemble(columns, usable, facade_copies(cfg, bind, max_rows=max_rows))
    _check_instances(cfg, res, z, check, columns, usable, k, m, beta, gamma, asm, max_rows)
    cfg.close()


@pytest.mark.gpu
def test_batch_slice_gives_the_same_columns(pkg):
    import torch
    cfg, res, rng = _batch(pkg, [128, 128], 5, 52)
    usable, _ = usable_for(cfg)
    columns = column_list(cfg.layout, True)
    beta, gamma = O.int_to_mont(_rand(rng)), O.int_to_mont(_rand(rng))
    kw = dict(columns_per_chunk=2, bind_output_bytes=True)
    want, err = cfg.permutation_product(res, columns, usable, beta, gamma, digests=res.digests, **kw)
    assert err == 0
    sl = pkg.BatchResult(res.digests[2:], None, res.gate[1:], res.lookup[1:], res.spread[1:])
    got, err = cfg.permutation_product(sl, columns, usable, beta, gamma, digests=res.digests[2:], **kw)
    assert err == 0 and torch.equal(got, want[1:])
    cfg.close()


@pytest.mark.gpu
def test_corrupted_copied_cell_is_counted_for_its_instance_only(pkg):
    import torch
    cfg, res, rng = _batch(pkg, [64], 6, 53)
    usable, _ = usable_for(cfg)
    columns = column_list(cfg.layout, False)
    beta, gamma = O.int_to_mont(_rand(rng)), O.int_to_mont(_rand(rng))
    want, err = cfg.permutation_product(res, columns, usable, beta, gamma, columns_per_chunk=3)
    assert err == 0
    res.lookup[3, 0, 100, 0] ^= 1                             # a lookup cell no longer equals the gate cell it copies
    got, err = cfg.permutation_product(res, columns, usable, beta, gamma, columns_per_chunk=3)
    assert err == 1
    keep = [i for i in range(6) if i != 3]
    assert torch.equal(got[keep], want[keep])
    h = columns.index((LOOKUP, 0)) // 3
    assert torch.equal(got[3, :h], want[3, :h]) and torch.equal(got[3, h, :101], want[3, h, :101])
    assert not torch.equal(got[3, -1, -1], want[3, -1, -1])
    cfg.close()


@pytest.mark.gpu
def test_zero_denominator_at_a_moved_cell_zeroes_the_rest(pkg):
    """gamma = -(p + beta sigma) of one moved cell of instance 0: like ff's batch_invert, that row's fraction is 0, and so is the rest
    of that chunk and every later chunk"""
    cfg, res, rng = _batch(pkg, [64], 3, 54)
    usable, k = usable_for(cfg)
    columns = column_list(cfg.layout, False)
    m = 3
    asm = assemble(columns, usable, facade_copies(cfg, False))
    c = columns.index((LOOKUP, 0))
    r = 500
    assert asm.mapping[c * usable + r] != c * usable + r
    values = _instance_values(cfg, res, 0, columns, usable)
    beta = _rand(rng)
    gamma = (-(values[c][r] + beta * sigma_value(asm, c, r, k))) % P
    z, errors = cfg.permutation_product(res, columns, usable, O.int_to_mont(beta), O.int_to_mont(gamma), columns_per_chunk=m)
    assert errors >= 1
    want = permutation_commit(values, asm, m, beta, gamma, k)
    h = c // m
    assert want[h][r + 1:] == [0] * (usable - r) and all(x == 0 for zc in want[h + 1:] for x in zc)
    assert _canon(z[0]) == [x for zc in want for x in zc]
    cfg.close()


@pytest.mark.gpu
def test_corrupted_digest_bytes_are_caught_by_the_instance_binding(pkg):
    import torch
    cfg, res, rng = _batch(pkg, [128, 128], 3, 55)
    usable, _ = usable_for(cfg)
    columns = column_list(cfg.layout, True)
    beta, gamma = O.int_to_mont(_rand(rng)), O.int_to_mont(_rand(rng))
    kw = dict(columns_per_chunk=2, bind_output_bytes=True)
    want, err = cfg.permutation_product(res, columns, usable, beta, gamma, digests=res.digests, **kw)
    assert err == 0
    bad = res.digests.copy()
    bad[3, 5] ^= 0x40                                          # instance 1, second digest, byte 5
    got, err = cfg.permutation_product(res, columns, usable, beta, gamma, digests=bad, **kw)
    assert err == 1
    assert torch.equal(got[0], want[0]) and torch.equal(got[2], want[2]) and not torch.equal(got[1], want[1])
    cfg.close()
