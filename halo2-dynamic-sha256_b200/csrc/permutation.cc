// permutation.cc -- the permutation mapping of the chip's copy constraints (PSE halo2_proofs plonk/permutation/keygen.rs
// `Assembly::{new, copy}`), replayed in the order the chip API issues them.
//
// The order decides the cycle order in `mapping` and so every intermediate value of the product column z.  It is the order
// halo2 sees through this project's facades: chip_api.hpp `Sha256DynamicConfig::assign_digest` / `RangeConfig::finalize` and
// the TestCircuit's instance binding (tests/cpp/test_chip_api.cc, reference lib.rs:480-482), the same in rust/src/lib.rs:
//   per digest() call d:  (2) the shape copies whose newer cell lies in d's gate range, shape order:
//                             constrain_equal(gate(a), gate(b) | fixed(k))
//                         (3) per spread limb n of d: constrain_equal(dense cell, gate(limb_dense_src[n])), then the spread cell
//   range.finalize:       constrain_equal(lookup cell k, gate(lookup_src[k])), push order (LookupGeom::range_cell)
//   bind_output_bytes:    constrain_instance(output_bytes[i], instance, i), i < 32 * n_digests
// A change to that order in chip_api.hpp has to be made here too (tests/test_permutation_product.py replays the recorded calls of
// the C++ facade against h2sha_get_permutation).
#include "permutation.h"

#include <algorithm>

#include "lookup_geom.h"

namespace h2sha {

bool perm_columns(const Plan& P, const h2sha_perm_desc_t& d, uint32_t U, PermColumns* out, std::string* err) {
  auto fail = [&](const std::string& m) { *err = m; return false; };
  if (!P.cfg.record_shape) return fail("engine was created without build_shape");
  if (d.columns_per_chunk == 0) return fail("columns_per_chunk must be >= 1 (cs.degree() - 2)");
  if (d.n_columns == 0 || !d.columns) return fail("the column list is empty");
  if (U == 0) return fail("usable_rows must be > 0");
  PermColumns& C = *out;
  C = PermColumns();
  C.n_cols = d.n_columns; C.usable_rows = U; C.m = d.columns_per_chunk;
  C.n_chunks = (C.n_cols + C.m - 1) / C.m;
  C.num_fixed = d.num_fixed ? d.num_fixed : 1;
  C.bind = d.bind_output_bytes ? 1 : 0;
  if ((uint64_t)C.n_cols * U >= (1ull << 32)) return fail("n_columns * usable_rows must be < 2^32");
  if (d.k) {
    if (d.k > 28 || (1ull << d.k) < (uint64_t)U + 2) return fail("k: 2^k must exceed usable_rows + 1 and k <= 28 (two-adicity of Fr)");
    C.k = d.k;
  } else {
    while ((1ull << C.k) < (uint64_t)U + 2) C.k++;
    if (C.k > 28) return fail("usable_rows needs a domain larger than 2^28");
  }
  const LookupGeom G = lookup_geom(P);
  const uint32_t nc = G.spread_cols;
  const uint32_t limit[7] = {P.n_gate_cols, P.n_lookup_cols, nc, nc, C.num_fixed, 0, 1};
  for (int k = 0; k < 7; k++) C.pos[k].assign(limit[k], -1);
  for (uint32_t c = 0; c < C.n_cols; c++) {
    const uint32_t kind = d.columns[2 * c], idx = d.columns[2 * c + 1];
    const std::string name = "column (" + std::to_string(kind) + ", " + std::to_string(idx) + ")";
    if (kind > H2SHA_COL_INSTANCE || idx >= limit[kind]) return fail(name + " is out of range");
    if (C.pos[kind][idx] >= 0) return fail(name + " is listed twice");
    C.pos[kind][idx] = (int32_t)c;
    C.kind.push_back(kind); C.index.push_back(idx);
  }
  if ((C.pos[H2SHA_COL_INSTANCE][0] >= 0) != (C.bind != 0)) return fail("the instance column is listed exactly when bind_output_bytes is set");
  // every column the chip copies from or to (the replay checks each cell again)
  for (uint32_t c = 0; c < P.n_gate_cols; c++)
    if (C.pos[H2SHA_COL_GATE][c] < 0) return fail("gate advice column " + std::to_string(c) + " holds copied cells but is not listed");
  for (uint32_t c = 0; c < P.n_lookup_cols && G.range_used(c) > 0; c++)
    if (C.pos[H2SHA_COL_LOOKUP][c] < 0) return fail("lookup advice column " + std::to_string(c) + " holds copied cells but is not listed");
  for (uint32_t c = 0; c < nc && G.spread_used(c) > 0; c++)
    if (C.pos[H2SHA_COL_DENSE][c] < 0 || C.pos[H2SHA_COL_SPREAD][c] < 0)
      return fail("spread column pair " + std::to_string(c) + " holds copied cells but is not listed");
  for (uint32_t c = 0; c < C.num_fixed && c < P.fixed_consts.size(); c++)
    if (C.pos[H2SHA_COL_FIXED][c] < 0) return fail("fixed column " + std::to_string(c) + " holds constants but is not listed");
  return true;
}

bool replay_permutation(const Plan& P, const PermColumns& C, std::vector<uint32_t>* mapping_out, std::string* err) {
  const uint32_t U = C.usable_rows;
  const uint64_t n = (uint64_t)C.n_cols * U;
  // Assembly::new: mapping[c][r] = aux[c][r] = (c, r), sizes = 1
  std::vector<uint32_t>& mapping = *mapping_out;
  mapping.resize(n);
  for (uint64_t i = 0; i < n; i++) mapping[i] = (uint32_t)i;
  std::vector<uint32_t> aux(mapping), sizes(n, 1);
  bool ok = true;
  auto cell = [&](uint32_t kind, uint32_t idx, uint32_t row) -> uint32_t {
    const int32_t p = idx < C.pos[kind].size() ? C.pos[kind][idx] : -1;
    if (p < 0) { *err = "column (" + std::to_string(kind) + ", " + std::to_string(idx) + ") holds a copied cell but is not listed"; ok = false; return 0; }
    if (row >= U) { *err = "a copied cell lies at row " + std::to_string(row) + " >= usable_rows"; ok = false; return 0; }
    return (uint32_t)p * U + row;
  };
  auto gate = [&](uint32_t s) {
    const uint32_t c = (uint32_t)(std::upper_bound(P.breaks.begin(), P.breaks.end(), s) - P.breaks.begin()) - 1;
    return cell(H2SHA_COL_GATE, c, s - P.breaks[c]);
  };
  auto fixed = [&](uint32_t k) { return cell(H2SHA_COL_FIXED, k % C.num_fixed, k / C.num_fixed); };   // Context::assign_fixed
  // Assembly::copy(left, right)
  auto copy = [&](uint32_t l, uint32_t r) {
    if (!ok) return;
    uint32_t left = aux[l], right = aux[r];
    if (left == right) return;
    if (sizes[left] < sizes[right]) std::swap(left, right);
    sizes[left] += sizes[right];
    uint32_t i = right;
    do { aux[i] = left; i = mapping[i]; } while (i != right);
    std::swap(mapping[l], mapping[r]);
  };
  const LookupGeom G = lookup_geom(P);
  const uint32_t D = (uint32_t)P.digests.size();
  for (uint32_t d = 0; d < D && ok; d++) {
    const bool last = d + 1 == D;
    const uint32_t g0 = P.digests[d].gate_base, g1 = last ? P.n_gate : P.digests[d + 1].gate_base;
    const uint32_t n0 = P.digests[d].limb_base, n1 = last ? P.n_limb : P.digests[d + 1].limb_base;
    for (const CopyPair& cp : P.copies) {   // (2) a is always the newer gate cell
      if (cp.a_kind != CP_GATE || cp.a_idx < g0 || cp.a_idx >= g1) continue;
      const uint32_t a = gate(cp.a_idx), b = cp.b_kind == CP_GATE ? gate(cp.b_idx) : fixed(cp.b_idx);
      copy(a, b);
    }
    for (uint32_t l = n0; l < n1; l++) {    // (3)
      const LookupCell c = G.spread_cell(l);
      copy(cell(H2SHA_COL_DENSE, c.col, c.row), gate(P.limb_gate_dense[l]));
      copy(cell(H2SHA_COL_SPREAD, c.col, c.row), gate(P.limb_gate_spread[l]));
    }
  }
  for (uint32_t k = 0; k < P.n_lookup && ok; k++) {   // range.finalize
    const LookupCell c = G.range_cell(k);
    copy(cell(H2SHA_COL_LOOKUP, c.col, c.row), gate(P.lookup_cells[k]));
  }
  if (C.bind)
    for (uint32_t d = 0; d < D && ok; d++)
      for (uint32_t i = 0; i < 32; i++) copy(gate(P.handles[d].output_bytes_idx[i]), cell(H2SHA_COL_INSTANCE, 0, 32 * d + i));
  return ok;
}

U256 perm_delta_mont() {
  static const U256 delta = {{0x870e56bbe533e9a2ull, 0x5b5f898e5e963f25ull, 0x64ec26aad4c86e71ull, 0x09226b6e22c6f0caull}};
  return fr::to_mont(delta);
}

U256 perm_omega_mont(uint32_t k) {
  static const U256 root = {{0xd34f1ed960c37c9cull, 0x3215cf6dd39329c8ull, 0x98865ea93dd31f74ull, 0x03ddb9f5166d18b7ull}};
  U256 w = fr::to_mont(root);
  for (uint32_t i = k; i < 28; i++) w = fr::mont_mul(w, w);
  return w;
}

}  // namespace h2sha
