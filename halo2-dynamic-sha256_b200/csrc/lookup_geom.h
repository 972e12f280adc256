// lookup_geom.h -- where the input cells of the chip's two lookups sit, and where their table-row multiplicities go.
// One definition for the planner (strides, zero ranges), the permutation replay, the batch checker, the hand-off and the
// lookup kernels (lookup_prework.cuh, lookup_product.cuh, k_mult_from_raw); the members compile for host and device.
//
//   range lookup   range.finalize copies the looked-up cells into the lookup advice columns in push order and wraps at
//                  max_rows: column c holds stream cells [c * max_rows, min(n_lookup, (c + 1) * max_rows)) (reference
//                  src/lib.rs:469).  Its other usable rows hold 0, which is table row 0.
//   spread lookup  limb n sits in column pair n % spread_cols, row n / spread_cols (spread.rs:202,228-231); the dense
//                  column of pair c is spread column c, its spread column is spread column spread_cols + c.
//   multiplicities one row of mult_words() u32 per instance: [n_lookup_cols << lookup_bits | spread_cols << limb_bits].
//   lookup_idx     range lookups first (one per lookup column), then one spread lookup per column pair.
#pragma once
#include <stdint.h>

#include "planner.h"

#if defined(__CUDACC__)
#define H2SHA_HD __host__ __device__ __forceinline__
#else
#define H2SHA_HD
#endif

namespace h2sha {

struct LookupCell {
  uint32_t col, row;
};

struct LookupGeom {
  uint64_t lookup_inst_cells, spread_inst_cells;   // Fr per instance in the lookup / spread buffers
  uint32_t n_lookup, max_rows, n_lookup_cols, lookup_col_rows, lookup_bits;
  uint32_t n_limb, spread_cols, spread_rows, limb_bits;
  uint32_t usable_rows;                            // rows of a lookup input column in the proof (0 where no call gives one)

  // range lookup column c: first stream cell (when range_used(c) > 0) and assigned rows
  H2SHA_HD uint32_t range_first(uint32_t c) const { return c * max_rows; }
  H2SHA_HD uint32_t range_used(uint32_t c) const {
    const uint64_t first = (uint64_t)c * max_rows;
    return first < n_lookup ? (n_lookup - first < max_rows ? (uint32_t)(n_lookup - first) : max_rows) : 0u;
  }
  H2SHA_HD LookupCell range_cell(uint32_t k) const {
    const uint32_t col = k / max_rows;
    return {col, k - col * max_rows};
  }
  // lookup advice columns the looked-up cells need (the engine may configure more)
  H2SHA_HD uint32_t range_cols_needed() const {
    const uint32_t c = (n_lookup + max_rows - 1) / max_rows;
    return c > 1u ? c : 1u;
  }
  // spread column pair c: assigned rows
  H2SHA_HD uint32_t spread_used(uint32_t c) const { return n_limb > c ? (n_limb - c + spread_cols - 1) / spread_cols : 0u; }
  H2SHA_HD LookupCell spread_cell(uint32_t n) const {
    const uint32_t row = n / spread_cols;
    return {n - row * spread_cols, row};
  }
  // multiplicity row of an instance: u32 words, and the first word of lookup l
  H2SHA_HD uint64_t range_words() const { return (uint64_t)n_lookup_cols << lookup_bits; }
  H2SHA_HD uint64_t mult_words() const { return range_words() + ((uint64_t)spread_cols << limb_bits); }
  H2SHA_HD uint64_t mult_off(uint32_t l) const {
    return l < n_lookup_cols ? (uint64_t)l << lookup_bits : range_words() + ((uint64_t)(l - n_lookup_cols) << limb_bits);
  }
  // rows of the largest assigned lookup input column, and the fewest usable rows the lookup arguments accept
  H2SHA_HD uint32_t max_range_used() const { return range_used(0); }
  H2SHA_HD uint32_t max_spread_used() const { return spread_used(0); }
  H2SHA_HD uint32_t min_usable_rows() const {
    const uint32_t lk = max_range_used(), sp = max_spread_used(), rt = 1u << lookup_bits, st = 1u << limb_bits;
    const uint32_t a = lk > sp ? lk : sp, t = rt > st ? rt : st;
    return a > t ? a : t;
  }
};

// The geometry of a plan (its strides as they are now: the engine may widen them after planning).
inline LookupGeom lookup_geom(const Plan& P, uint32_t usable_rows = 0) {
  LookupGeom G{};
  G.n_lookup = P.n_lookup; G.max_rows = P.cfg.max_rows; G.n_lookup_cols = P.n_lookup_cols; G.lookup_col_rows = P.lookup_col_rows;
  G.lookup_bits = P.cfg.lookup_bits;
  G.n_limb = P.n_limb; G.spread_cols = P.cfg.spread_cols; G.spread_rows = P.spread_rows; G.limb_bits = P.cfg.limb_bits;
  G.lookup_inst_cells = (uint64_t)P.n_lookup_cols * P.lookup_col_rows;
  G.spread_inst_cells = (uint64_t)2 * P.cfg.spread_cols * P.spread_rows;
  G.usable_rows = usable_rows;
  return G;
}

// One lookup of the argument, by lookup_idx.
struct LookupSel {
  bool valid;            // lookup_idx names a lookup
  bool is_range;
  uint32_t col;          // range: lookup column; spread: column pair
  uint32_t n_vals;       // table rows
  uint64_t mult_off;     // first word of its multiplicities in an instance's row
  uint64_t inst_cells;   // Fr per instance in the witness buffer it reads (lookup or spread)
  uint64_t col_off;      // Fr offset of the looked-up column (range) / the dense column (spread) inside an instance
  uint64_t spread_off;   // spread: Fr distance from a dense cell to its spread cell
  uint32_t used;         // assigned rows of that column; the rows above hold 0
  template <class T>
  T* buffer(T* lookup, T* spread) const { return is_range ? lookup : spread; }
};

inline LookupSel select_lookup(const LookupGeom& G, uint32_t lookup_idx) {
  LookupSel L{};
  L.is_range = lookup_idx < G.n_lookup_cols;
  L.valid = lookup_idx < G.n_lookup_cols + G.spread_cols;
  if (!L.valid) return L;
  L.mult_off = G.mult_off(lookup_idx);
  if (L.is_range) {
    L.col = lookup_idx;
    L.n_vals = 1u << G.lookup_bits;
    L.inst_cells = G.lookup_inst_cells;
    L.col_off = (uint64_t)L.col * G.lookup_col_rows;
    L.used = G.range_used(L.col);
  } else {
    L.col = lookup_idx - G.n_lookup_cols;
    L.n_vals = 1u << G.limb_bits;
    L.inst_cells = G.spread_inst_cells;
    L.col_off = (uint64_t)L.col * G.spread_rows;
    L.spread_off = (uint64_t)G.spread_cols * G.spread_rows;
    L.used = G.spread_used(L.col);
  }
  return L;
}

}  // namespace h2sha
