"""Geometry of the lookup input columns (csrc/lookup_geom.h), restated from the reference and compared with what the
engine reports on plan-only configurations (no GPU needed):

- range.finalize copies the looked-up cells into the lookup advice columns in push order and wraps at max_rows
  (reference src/lib.rs:469): column c holds cells [c * max_rows, min(n_lookup, (c + 1) * max_rows));
- spread limb n sits in column pair n % num_advice_columns, row n // num_advice_columns (src/spread.rs:202,228-231);
- the multiplicity row of an instance holds one bin per table row of every lookup: range lookups first, then spread lookups;
- the lookup arguments need usable_rows >= every assigned lookup input column and every table.
"""
import pytest

MAX_ROWS = (1 << 17) - 9


def _up8(x):
    return (x + 7) // 8 * 8


def _range_used(n_lookup, max_rows, c):
    return max(0, min(max_rows, n_lookup - c * max_rows))


def _spread_used(n_limb, cols, c):
    return len(range(c, n_limb, cols))


def _max_rows(n_lookup, split):
    """max_rows giving one column holding every cell, two columns (exactly full when n_lookup is even), or three"""
    return {"one": n_lookup, "two": (n_lookup + 1) // 2, "three": (n_lookup + 2) // 3}[split]


# [64, 64]: an even number of looked-up cells (two exactly full columns), a limb count that 3 does not divide;
# [192]: an odd number of looked-up cells, a limb count that 1, 2 and 3 all divide
@pytest.mark.parametrize("sizes", [[64, 64], [192]])
@pytest.mark.parametrize("lookup_bits", [8])   # a range table smaller than the columns: min_usable_rows follows the cells
@pytest.mark.parametrize("num_bits_lookup", [1, 8, 16])
@pytest.mark.parametrize("spread_cols", [1, 2, 3])
@pytest.mark.parametrize("split", ["one", "two", "three"])
def test_lookup_geometry_matches_the_reference_layout(pkg, sizes, lookup_bits, num_bits_lookup, spread_cols, split):
    kw = dict(device=-1, lookup_bits=lookup_bits, num_bits_lookup=num_bits_lookup, num_advice_columns=spread_cols)
    base = pkg.Sha256DynamicConfig.configure(sizes, max_rows=MAX_ROWS, **kw)
    max_rows = _max_rows(base.layout.n_lookup_cells, split)
    base.close()
    cfg = pkg.Sha256DynamicConfig.configure(sizes, max_rows=max_rows, **kw)
    lay, info = cfg.layout, cfg.lookup_info()
    n_lookup, n_limb = lay.n_lookup_cells, lay.n_spread_limbs

    n_cols = max(1, -(-n_lookup // max_rows))
    assert n_cols == {"one": 1, "two": 2, "three": 3}[split]
    assert lay.n_lookup_cols == info["n_range_lookups"] == n_cols
    lk_used = [_range_used(n_lookup, max_rows, c) for c in range(n_cols)]
    assert sum(lk_used) == n_lookup and min(lk_used) > 0
    assert lay.lookup_col_rows == _up8(max(lk_used))

    sp_used = [_spread_used(n_limb, spread_cols, c) for c in range(spread_cols)]
    assert sum(sp_used) == n_limb
    assert lay.n_spread_cols == 2 * spread_cols and info["n_spread_lookups"] == spread_cols
    assert lay.spread_rows == _up8(max(sp_used))

    assert info["range_table_rows"] == 1 << lookup_bits and info["spread_table_rows"] == 1 << num_bits_lookup
    assert info["mult_words_per_instance"] == n_cols * (1 << lookup_bits) + spread_cols * (1 << num_bits_lookup)
    assert info["min_usable_rows"] == max(lk_used + sp_used + [1 << lookup_bits, 1 << num_bits_lookup])
    cfg.close()


def test_extra_lookup_columns_and_widened_strides(pkg):
    """num_lookup_advice adds lookup columns that hold no cell; wider strides change no count"""
    kw = dict(device=-1, max_rows=5000, num_advice_columns=3)
    plain = pkg.Sha256DynamicConfig.configure([128, 128], **kw)
    wide = pkg.Sha256DynamicConfig.configure([128, 128], num_lookup_advice=5, lookup_col_rows=6000, spread_rows=9000, **kw)
    p, w = plain.layout, wide.layout
    assert p.n_lookup_cols == 3 and w.n_lookup_cols == 5
    assert (w.lookup_col_rows, w.spread_rows) == (6000, 9000)
    pi, wi = plain.lookup_info(), wide.lookup_info()
    assert wi["n_range_lookups"] == 5
    assert wi["mult_words_per_instance"] == pi["mult_words_per_instance"] + 2 * (1 << 16)
    assert wi["min_usable_rows"] == pi["min_usable_rows"]
    plain.close()
    wide.close()
