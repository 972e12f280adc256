// lookup_prework.cuh -- lookup-argument pre-work on the witness that is already in HBM (SURVEY.md §8f #4).
// Included at the end of engine.cu (one translation unit: it uses the engine struct, c_fr and mont_from_u32).
//
// What it replaces: the first step of halo2's lookup prover for the chip's two lookups --
//   * "spread lookup" per column pair (reference src/spread.rs:53-62, table src/spread.rs:165-194),
//   * the range lookup on the lookup advice column(s) filled by range.finalize (reference src/lib.rs:409-418, 469;
//     halo2-base RangeConfig, dependency not vendored),
// i.e. PSE halo2_proofs plonk/lookup/prover.rs `permute_expression_pair`: A' = the input column sorted, S' = the table
// column permuted so that A'[i] == S'[i] or A'[i] == A'[i-1].  Both are functions of the table-row *multiplicities*
// of the input, so the work is split into
//   k_range_mult / k_spread_mult   cells (Montgomery Fr) -> canonical value (REDC) -> histogram over the table rows,
//   k_permute_scan                 per (instance, lookup): exclusive scans over the table rows in sorted order,
//   k_permute_fill                 one thread per row: two-level search in the scans, 2 x 256-bit stores.
// HBM-bound like the rest of the path: the fill writes 64 B per usable row and reads only the (L2-resident) scans.
// oracle/lookup_prework.py is the CPU restatement the tests compare against.  Where the input cells sit, the layout of the
// multiplicity buffer and the meaning of lookup_idx: LookupGeom and select_lookup (lookup_geom.h).
#pragma once

#include <cub/device/device_segmented_sort.cuh>

#include "lookup_geom.h"

namespace {

// Table membership of the chip's two lookups, from Montgomery cells: REDC, then the range table 0 .. n_vals - 1, or a row
// (dense, spread32(dense)) of the spread table with dense < n_vals.  *row = the table row a member hits.  The multiplicity kernels
// and the constraint check (batch_check.cuh) share them.
__device__ __forceinline__ bool range_table_row(const uint64_t* cell, uint32_t n_vals, uint32_t* row) {
  uint64_t x[4], v[4];
  load_cell(cell, x);
  mont_reduce(x, v);
  *row = (uint32_t)v[0];
  return (v[1] | v[2] | v[3]) == 0 && v[0] < n_vals;
}
__device__ __forceinline__ bool spread_table_row(const uint64_t* dense_cell, const uint64_t* spread_cell, uint32_t n_vals, uint32_t* row) {
  uint64_t x[4], d[4], s[4];
  load_cell(dense_cell, x);
  mont_reduce(x, d);
  load_cell(spread_cell, x);
  mont_reduce(x, s);
  *row = (uint32_t)d[0];
  bool ok = (d[1] | d[2] | d[3]) == 0 && d[0] < n_vals && (s[1] | s[2] | s[3]) == 0;
  if (ok) ok = spread32(d[0]) == s[0];   // the pair has to be a table row, not just the dense half
  return ok;
}

// range lookup: one thread per assigned cell of the lookup advice column(s).  grid = (tiles, instances).
__global__ void __launch_bounds__(256) k_range_mult(const LookupGeom G, const uint64_t* __restrict__ lookup, uint32_t* __restrict__ mult,
                                                   uint32_t* __restrict__ bad) {
  const uint64_t inst = blockIdx.y;
  const uint64_t* base = lookup + inst * G.lookup_inst_cells * 4;
  uint32_t* m_inst = mult + inst * G.mult_words();
  const uint32_t n_vals = 1u << G.lookup_bits;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < G.n_lookup; i += gridDim.x * blockDim.x) {
    const LookupCell c = G.range_cell(i);
    uint32_t v;
    if (range_table_row(base + ((uint64_t)c.col * G.lookup_col_rows + c.row) * 4, n_vals, &v)) atomicAdd(&m_inst[(uint64_t)c.col * n_vals + v], 1u);
    else if (bad) atomicAdd(bad, 1u);
  }
  // never-assigned rows of a column hold 0
  if (blockIdx.x == 0 && threadIdx.x < G.n_lookup_cols) {
    const uint32_t col = threadIdx.x, used = G.range_used(col);
    if (G.usable_rows > used) atomicAdd(&m_inst[(uint64_t)col * n_vals], G.usable_rows - used);
  }
}

// spread lookups, one histogram per column pair.  Block-local histograms in
// shared memory, flushed with one global atomic per non-empty bin.  grid = (tiles, instances); dynamic smem = cols * 2^bits * 4.
__global__ void __launch_bounds__(256) k_spread_mult(const LookupGeom G, const uint64_t* __restrict__ spread, uint32_t* __restrict__ mult,
                                                    uint32_t* __restrict__ bad) {
  extern __shared__ uint32_t s_hist[];   // [spread_cols << limb_bits]
  const uint32_t n_vals = 1u << G.limb_bits, n_bins = G.spread_cols * n_vals;
  for (uint32_t i = threadIdx.x; i < n_bins; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  const uint64_t inst = blockIdx.y;
  const uint64_t* base = spread + inst * G.spread_inst_cells * 4;
  uint32_t* m_inst = mult + inst * G.mult_words() + G.range_words();
  uint32_t n_bad = 0;
  for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < G.n_limb; n += gridDim.x * blockDim.x) {
    const LookupCell c = G.spread_cell(n);
    uint32_t d;
    if (spread_table_row(base + ((uint64_t)c.col * G.spread_rows + c.row) * 4, base + ((uint64_t)(G.spread_cols + c.col) * G.spread_rows + c.row) * 4,
                         n_vals, &d))
      atomicAdd(&s_hist[c.col * n_vals + d], 1u);
    else n_bad++;
  }
  if (n_bad && bad) atomicAdd(bad, n_bad);
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < n_bins; i += blockDim.x)
    if (s_hist[i]) atomicAdd(&m_inst[i], s_hist[i]);
  if (blockIdx.x == 0 && threadIdx.x < G.spread_cols) {
    const uint32_t col = threadIdx.x, used = G.spread_used(col);
    if (G.usable_rows > used) atomicAdd(&m_inst[col * n_vals], G.usable_rows - used);
  }
}

struct PermuteArgs {
  const uint32_t* mult;        // this lookup's multiplicities of instance 0; instance i at + i * mult_stride
  uint64_t mult_stride;
  const uint32_t* order;       // sorted position -> table row, or null (identity: the range table is already sorted)
  const uint32_t* vals;        // [n_vals][8]: Montgomery value at each sorted position, or null (value = position, range table)
  uint32_t n_vals, usable_rows;
  uint32_t* scan;              // workspace [n_inst][3][n_vals]: start | distinct-before | leftover-before   (+ [n_inst] totals after)
  uint32_t* totals;            // [n_inst][4]: distinct inputs, sum of multiplicities, m[first sorted row], leftover copies of the first sorted row
  // identity order only (range table): the two searches of the fill kernel inverted by the scan kernel --
  uint32_t* vrow;              // [n_inst][usable_rows]: sorted position of the value in row r of A', for r >= m[0] (rows below are the run of 0)
  uint32_t* llist;             // [n_inst][n_vals]: the unused table rows > 0 in increasing order (leftover element j >= lf0 is llist[j - lf0])
  uint32_t* errors;            // may be null
  uint32_t err_stride;         // 0: errors is one counter for the batch; 1: errors[inst] (the *_per_instance calls)
  uint32_t tab_stride;         // per-instance spread tables: sorted positions per instance in order / vals (0: one table for the batch)
  const uint32_t* skip;        // per-instance spread tables: [n_inst] nonzero when theta_i makes two table rows collide, or null
  uint64_t* out_input;         // [n_inst][usable_rows] Fr
  uint64_t* out_table;
};

// one CTA per instance: exclusive scans, in sorted order, of m (-> first row of each value's run in A'), of [m > 0]
// (-> how many runs start before it) and of the leftover table multiplicity t - [m > 0]
// (t = 1 per table row; the row holding the padding value -- table row 0 -- also takes the usable_rows - n_vals padded rows)
// VPT = consecutive sorted positions per thread and round: 1 (any order / size), or 4 with 128-bit loads and stores when the order is the
// identity and the table size allows.  (16 per thread -- four rounds instead of sixteen for the 2^16-row range table -- was measured
// slower in round 2: 0.593 vs 0.504 ms per 256 instances; 64-byte strides per lane and spills cost more than the saved barriers.)
template <int VPT>
__global__ void __launch_bounds__(1024) k_permute_scan(const PermuteArgs A) {
  __shared__ uint32_t s_part[2][3][32];   // double-buffered by round: two barriers per round
  const uint32_t inst = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (A.skip && A.skip[inst]) {   // colliding table rows: counted once, the pair is not written
    if (tid == 0 && A.errors) atomicAdd(A.errors + (uint64_t)inst * A.err_stride, 1u);
    return;
  }
  const uint32_t* order = A.order ? A.order + (uint64_t)inst * A.tab_stride : nullptr;
  const uint32_t* m = A.mult + (uint64_t)inst * A.mult_stride;
  uint32_t* start = A.scan + (uint64_t)inst * 3 * A.n_vals;
  uint32_t* dpre = start + A.n_vals;
  uint32_t* lpre = dpre + A.n_vals;
  const uint32_t pad = A.usable_rows - A.n_vals;
  constexpr bool vec = VPT > 1;
  uint32_t base[3] = {0, 0, 0};
  uint32_t round = 0;
  for (uint32_t k0 = 0; k0 < A.n_vals; k0 += 1024u * VPT, round++) {
    const uint32_t k = k0 + tid * VPT;
    uint32_t mk[VPT], lf[VPT];
    if constexpr (vec) {
#pragma unroll
      for (int q4 = 0; q4 < VPT / 4; q4++) {
        const uint4 q = *reinterpret_cast<const uint4*>(m + k + 4 * q4);
        mk[4 * q4] = q.x; mk[4 * q4 + 1] = q.y; mk[4 * q4 + 2] = q.z; mk[4 * q4 + 3] = q.w;
      }
#pragma unroll
      for (int i = 0; i < VPT; i++) lf[i] = 1u + ((k + i) == 0 ? pad : 0u) - (mk[i] ? 1u : 0u);
    } else {
      mk[0] = 0; lf[0] = 0;
      if (k < A.n_vals) {
        const uint32_t row = order ? order[k] : k;
        mk[0] = m[row];
        lf[0] = 1u + (row == 0 ? pad : 0u) - (mk[0] ? 1u : 0u);
      }
    }
    uint32_t v[3] = {0, 0, 0};
#pragma unroll
    for (int i = 0; i < VPT; i++) { v[0] += mk[i]; v[1] += mk[i] ? 1u : 0u; v[2] += lf[i]; }
    uint32_t (*part)[32] = s_part[round & 1u];
    uint32_t incl[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
      uint32_t x = v[q];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if ((int)lane >= o) x += y;
      }
      incl[q] = x;
      if (lane == 31) part[q][warp] = x;
    }
    __syncthreads();
    if (warp < 3) {
      uint32_t x = part[warp][lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if ((int)lane >= o) x += y;
      }
      part[warp][lane] = x;   // inclusive over warps
    }
    __syncthreads();
    uint32_t ex[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
      ex[q] = base[q] + (warp ? part[q][warp - 1] : 0u) + incl[q] - v[q];
      base[q] += part[q][31];
    }
    if constexpr (vec) {
      uint32_t o0 = ex[0], o1 = ex[1], o2 = ex[2];
#pragma unroll
      for (int q4 = 0; q4 < VPT / 4; q4++) {
        uint4 a, b, c;
        a.x = o0; o0 += mk[4 * q4]; a.y = o0; o0 += mk[4 * q4 + 1]; a.z = o0; o0 += mk[4 * q4 + 2]; a.w = o0; o0 += mk[4 * q4 + 3];
        b.x = o1; o1 += mk[4 * q4] ? 1u : 0u; b.y = o1; o1 += mk[4 * q4 + 1] ? 1u : 0u; b.z = o1; o1 += mk[4 * q4 + 2] ? 1u : 0u; b.w = o1; o1 += mk[4 * q4 + 3] ? 1u : 0u;
        c.x = o2; o2 += lf[4 * q4]; c.y = o2; o2 += lf[4 * q4 + 1]; c.z = o2; o2 += lf[4 * q4 + 2]; c.w = o2; o2 += lf[4 * q4 + 3];
        *reinterpret_cast<uint4*>(start + k + 4 * q4) = a; *reinterpret_cast<uint4*>(dpre + k + 4 * q4) = b; *reinterpret_cast<uint4*>(lpre + k + 4 * q4) = c;
      }
    } else if (k < A.n_vals) {
      start[k] = ex[0]; dpre[k] = ex[1]; lpre[k] = ex[2];
    }
    if (A.vrow && order == nullptr) {
      // inverse maps for the fill kernel (identity order: sorted position == table row).  Position 0 is implicit in both:
      // its run is rows [0, m[0]) of A' and its leftover copies are elements [0, lf0) of the leftover sequence.
      uint32_t* vr = A.vrow + (uint64_t)inst * A.usable_rows;
      uint32_t* ll = A.llist + (uint64_t)inst * A.n_vals;
      const uint32_t lf0 = 1u + pad - (m[0] ? 1u : 0u);
      uint32_t st_k = ex[0], lp_k = ex[2];
#pragma unroll
      for (uint32_t q = 0; q < (uint32_t)VPT; q++) {
        if (k + q < A.n_vals && k + q > 0) {
          for (uint32_t r = 0; r < mk[q]; r++) vr[st_k + r] = k + q;
          if (lf[q]) ll[lp_k - lf0] = k + q;   // leftover element j >= lf0 of the sequence is ll[j - lf0]
        }
        st_k += mk[q]; lp_k += lf[q];
      }
    }
  }
  if (tid == 0) {
    A.totals[4 * inst] = base[1];
    A.totals[4 * inst + 1] = base[0];
    const uint32_t m_first = m[order ? order[0] : 0];
    A.totals[4 * inst + 2] = m_first;
    A.totals[4 * inst + 3] = 1u + ((order ? order[0] : 0u) == 0u ? pad : 0u) - (m_first ? 1u : 0u);
    if (base[0] != A.usable_rows && A.errors) atomicAdd(A.errors + (uint64_t)inst * A.err_stride, 1u);   // multiplicities do not cover the usable rows
  }
}

// Multiplicities of ONE lookup of instances [first, first + gridDim.x) from the raw value lists k_expand<.., MODE 1> left in the engine
// (h2sha_permute_lookup_from_raw): one CTA per instance, out[blockIdx.x][n_vals].  Hot values (< 4096: zeros, bytes) are binned in
// shared memory, the bins are written once (coalesced), the rest follows with global atomics on lines that are L2-resident by then.
struct MultOneArgs {
  const uint32_t* lookup_raw;   // [n][n_lookup]
  const uint8_t* dense_raw;     // [n][n_limb]
  uint32_t* out;                // [gridDim.x][n_vals]
  uint32_t* bad;                // may be null
  uint64_t first;
  uint32_t n_vals, is_range, col;
  LookupGeom G;
};
__global__ void __launch_bounds__(512) k_mult_one(const MultOneArgs A) {
  __shared__ uint32_t s_small[MULT_SMALL_BINS];
  const LookupGeom& G = A.G;
  const uint64_t inst = A.first + blockIdx.x;
  uint32_t* bins = A.out + (uint64_t)blockIdx.x * A.n_vals;
  const uint32_t n_small = min((uint32_t)MULT_SMALL_BINS, A.n_vals);
  for (uint32_t i = threadIdx.x; i < n_small; i += blockDim.x) s_small[i] = 0;
  __syncthreads();
  uint32_t n_bad = 0, used = 0;
  const uint32_t* lr = A.lookup_raw + inst * G.n_lookup;
  const uint8_t* dr = A.dense_raw + inst * G.n_limb;
  uint32_t k0 = 0, k1 = 0;
  if (A.is_range) {
    used = G.range_used(A.col);
    k0 = G.range_first(A.col); k1 = k0 + used;
    for (uint32_t k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
      const uint32_t v = lr[k];
      if (v < n_small) atomicAdd(&s_small[v], 1u);
    }
  } else {
    used = G.spread_used(A.col);
    for (uint32_t n = A.col + threadIdx.x * G.spread_cols; n < G.n_limb; n += blockDim.x * G.spread_cols) atomicAdd(&s_small[dr[n]], 1u);   // dense limbs are < 2^8 <= n_small
  }
  if (threadIdx.x == 0 && G.usable_rows > used) atomicAdd(&s_small[0], G.usable_rows - used);   // never-assigned rows hold 0 = table row 0
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < A.n_vals; i += blockDim.x) bins[i] = i < n_small ? s_small[i] : 0u;
  __syncthreads();
  if (A.is_range) {
    for (uint32_t k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
      const uint32_t v = lr[k];
      if (v >= A.n_vals) n_bad++;
      else if (v >= n_small) atomicAdd(&bins[v], 1u);
    }
  }
  if (n_bad && A.bad) atomicAdd(A.bad, n_bad);
}

// last index k in [lo, hi) with a[k] <= x (a non-decreasing, a[lo] <= x)
__device__ __forceinline__ uint32_t last_leq(const uint32_t* __restrict__ a, uint32_t lo, uint32_t hi, uint32_t x) {
  while (hi - lo > 1) {   // invariant: a[lo] <= x, (hi == end or a[hi] > x)
    const uint32_t mid = (lo + hi) >> 1;
    if (a[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ void permuted_value(const uint32_t* vals, uint32_t k, uint32_t x[8]) {
  if (vals) {
    const uint4 lo = __ldg(reinterpret_cast<const uint4*>(vals + (uint64_t)k * 8)), hi = __ldg(reinterpret_cast<const uint4*>(vals + (uint64_t)k * 8) + 1);
    x[0] = lo.x; x[1] = lo.y; x[2] = lo.z; x[3] = lo.w; x[4] = hi.x; x[5] = hi.y; x[6] = hi.z; x[7] = hi.w;
  } else {
    mont_from_u32(k, x);
  }
}

// grid = (tiles, instances), one thread per row.  The two searches (run of the row in A'; leftover table element of a
// repeated row) are two-level: a <= 256-entry sample of each scan sits in shared memory, so only log2(n_vals / 256)
// dependent global loads remain per search (8 for the range table, none for the spread table) and neighbouring rows
// touch the same few cache lines.
__global__ void __launch_bounds__(256) k_permute_fill(const PermuteArgs A) {
  __shared__ uint32_t s_start[256], s_lpre[256];
  const uint32_t inst = blockIdx.y;
  if (A.skip && A.skip[inst]) return;   // colliding table rows: counted by the scan kernel
  const uint32_t* start = A.scan + (uint64_t)inst * 3 * A.n_vals;
  const uint32_t* dpre = start + A.n_vals;
  const uint32_t* lpre = dpre + A.n_vals;
  const uint32_t* vals = A.vals ? A.vals + (uint64_t)inst * A.tab_stride * 8 : nullptr;
  const uint32_t n_distinct = A.totals[4 * inst];
  if (A.totals[4 * inst + 1] != A.usable_rows) return;   // inconsistent multiplicities: reported by the scan kernel
  const uint32_t n_rep = A.usable_rows - n_distinct;
  uint32_t* out_a = reinterpret_cast<uint32_t*>(A.out_input) + (uint64_t)inst * A.usable_rows * 8;
  uint32_t* out_s = reinterpret_cast<uint32_t*>(A.out_table) + (uint64_t)inst * A.usable_rows * 8;
  if (A.vrow && A.order == nullptr) {
    // identity order (range table): the scan kernel has inverted both searches.  Rows below m[0] are the run of value 0 (the
    // never-assigned rows: almost all of them), whose repeated rows take leftover elements with ONE dependent load.
    const uint32_t m0 = A.totals[4 * inst + 2], lf0 = A.totals[4 * inst + 3];
    const uint32_t* vr = A.vrow + (uint64_t)inst * A.usable_rows;
    const uint32_t* ll = A.llist + (uint64_t)inst * A.n_vals;
    for (uint32_t row = blockIdx.x * 256u + threadIdx.x; row < A.usable_rows; row += gridDim.x * 256u) {
      uint32_t k = 0, st = 0, dp = 0;
      if (row >= m0) { k = __ldg(vr + row); st = __ldg(start + k); dp = __ldg(dpre + k); }
      uint32_t x[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // value 0 is 0 in Montgomery form as well
      if (k) permuted_value(vals, k, x);
      store_cell2(out_a + (uint64_t)row * 8, make_uint4(x[0], x[1], x[2], x[3]), make_uint4(x[4], x[5], x[6], x[7]));
      if (row != st) {
        const uint32_t j = n_rep - 1u - (row - dp - 1u);
        const uint32_t w = j < lf0 ? 0u : __ldg(ll + (j - lf0));
        if (w) permuted_value(vals, w, x);
        else {
#pragma unroll
          for (int q = 0; q < 8; q++) x[q] = 0;
        }
      }
      store_cell2(out_s + (uint64_t)row * 8, make_uint4(x[0], x[1], x[2], x[3]), make_uint4(x[4], x[5], x[6], x[7]));
    }
    return;
  }
  const uint32_t stride = max(1u, A.n_vals >> 8), n_coarse = A.n_vals / stride;
  for (uint32_t i = threadIdx.x; i < n_coarse; i += 256) { s_start[i] = __ldg(start + i * stride); s_lpre[i] = __ldg(lpre + i * stride); }
  __syncthreads();
  for (uint32_t row = blockIdx.x * 256u + threadIdx.x; row < A.usable_rows; row += gridDim.x * 256u) {
    const uint32_t c = last_leq(s_start, 0, n_coarse, row) * stride;
    const uint32_t k = last_leq(start, c, c + stride, row);
    uint32_t x[8];
    permuted_value(vals, k, x);
    store_cell2(out_a + (uint64_t)row * 8, make_uint4(x[0], x[1], x[2], x[3]), make_uint4(x[4], x[5], x[6], x[7]));
    if (row != __ldg(start + k)) {
      // a repeated row: halo2 pops the repeated rows from the back while walking the leftover table elements upwards.
      // rows <= row: row + 1, first occurrences among them: dpre[k] + 1 -> zero-based rank among the repeated rows
      const uint32_t rank = row - __ldg(dpre + k) - 1u;
      const uint32_t j = n_rep - 1u - rank;
      const uint32_t c2 = last_leq(s_lpre, 0, n_coarse, j) * stride;
      const uint32_t w = last_leq(lpre, c2, c2 + stride, j);
      permuted_value(vals, w, x);
    }
    store_cell2(out_s + (uint64_t)row * 8, make_uint4(x[0], x[1], x[2], x[3]), make_uint4(x[4], x[5], x[6], x[7]));
  }
}

// Montgomery form of 0 .. n-1: the range table's values, kept in HBM (2 MB for 16 bits, L2-resident while the fill runs)
__global__ void k_range_table(uint32_t* tab, uint32_t n) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x[8];
  mont_from_u32(i, x);
  store_cell2(tab + (uint64_t)i * 8, make_uint4(x[0], x[1], x[2], x[3]), make_uint4(x[4], x[5], x[6], x[7]));
}

// Spread table per instance (h2sha_permute_lookup_per_instance): the host path below (compressed_spread_table, std::stable_sort by
// canonical value, collision check) on the device for every (instance, table row).  The rows are sorted by four stable segmented
// sorts on the 64-bit limbs of the canonical value, least significant limb first (one segment per instance, the row index as the
// value): equal to std::stable_sort on the whole 256-bit value for any theta.

// dense * theta + spread of spread-table row i (halo2 `compress_expressions`), Montgomery form: compressed_spread_table on the device
__device__ __forceinline__ void compressed_spread_row(const uint64_t theta[4], uint32_t i, uint64_t r[4]) {
  uint64_t d[4], s[4], t[4];
  mont_from_u64(i, d);
  mont_from_u64(spread32(i), s);
  mont_mul_dev(theta, d, t);
  fr_add_dev(t, s, r);
}

struct SpreadSort {
  const uint64_t* chal;   // [n][3][4]: theta_i first
  uint32_t n_vals;
  uint64_t* canon;        // [n][4][n_vals]: canonical value of each table row, limb-major
  uint64_t* key;          // [n][n_vals]: the limb the next sort pass orders by
  uint32_t* idx;          // [n][n_vals]: table row at each position
  int* seg;               // [n + 1] segment offsets
  uint32_t* vals;         // [n][n_vals][8]: Montgomery value at each sorted position
  uint32_t* skip;         // [n]: two sorted neighbours are equal
};

// grid (tiles, instances)
__global__ void __launch_bounds__(256) k_spread_rows(const SpreadSort S) {
  const uint32_t inst = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) {
    S.seg[inst] = (int)(inst * S.n_vals);
    S.skip[inst] = 0;
    if (inst + 1 == gridDim.y) S.seg[inst + 1] = (int)((inst + 1) * S.n_vals);
  }
  if (i >= S.n_vals) return;
  uint64_t th[4], cm[4], c[4];
  load_cell(S.chal + (uint64_t)inst * 12, th);
  compressed_spread_row(th, i, cm);
  mont_reduce(cm, c);   // canonical value: what `impl Ord for Fr` compares
#pragma unroll
  for (int l = 0; l < 4; l++) S.canon[((uint64_t)inst * 4 + l) * S.n_vals + i] = c[l];
  S.key[(uint64_t)inst * S.n_vals + i] = c[0];
  S.idx[(uint64_t)inst * S.n_vals + i] = i;
}

// the next sort key: limb `limb` of the row at each position
__global__ void __launch_bounds__(256) k_spread_key(const SpreadSort S, const uint32_t* __restrict__ idx, uint64_t* __restrict__ key, uint32_t limb) {
  const uint32_t inst = blockIdx.y, k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= S.n_vals) return;
  const uint64_t p = (uint64_t)inst * S.n_vals + k;
  key[p] = S.canon[((uint64_t)inst * 4 + limb) * S.n_vals + idx[p]];
}

// values in sorted order, and the flag of an instance in which two neighbouring sorted values are equal (row 0 compresses to 0, so
// a row that also compresses to 0 is caught too)
__global__ void __launch_bounds__(256) k_spread_sorted(const SpreadSort S, const uint32_t* __restrict__ order) {
  const uint32_t inst = blockIdx.y, k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= S.n_vals) return;
  const uint64_t p = (uint64_t)inst * S.n_vals + k;
  const uint32_t row = order[p];
  uint64_t th[4], cm[4];
  load_cell(S.chal + (uint64_t)inst * 12, th);
  compressed_spread_row(th, row, cm);
  store_cell2(S.vals + p * 8, make_uint4((uint32_t)cm[0], (uint32_t)(cm[0] >> 32), (uint32_t)cm[1], (uint32_t)(cm[1] >> 32)),
              make_uint4((uint32_t)cm[2], (uint32_t)(cm[2] >> 32), (uint32_t)cm[3], (uint32_t)(cm[3] >> 32)));
  if (k == 0) return;
  const uint32_t prev = order[p - 1];
  const uint64_t* c = S.canon + (uint64_t)inst * 4 * S.n_vals;
  bool eq = true;
#pragma unroll
  for (int l = 0; l < 4; l++) eq = eq && c[(uint64_t)l * S.n_vals + row] == c[(uint64_t)l * S.n_vals + prev];
  if (eq) atomicOr(S.skip + inst, 1u);
}

// bytes of the SpreadSort arrays of `ni` instances, and their place in `base` (256-byte aligned each)
uint64_t spread_sort_layout(uint64_t ni, uint32_t n_vals, uint64_t cub_bytes, uint8_t* base, SpreadSort* S, void** cub_tmp, uint64_t** key_alt, uint32_t** idx_alt) {
  uint64_t off = 0;
  auto take = [&](uint64_t bytes) { uint8_t* p = base ? base + off : nullptr; off += (bytes + 255) / 256 * 256; return p; };
  const uint64_t rows = ni * n_vals;
  S->vals = (uint32_t*)take(rows * 32);
  S->canon = (uint64_t*)take(rows * 32);
  S->key = (uint64_t*)take(rows * 8);
  *key_alt = (uint64_t*)take(rows * 8);
  S->idx = (uint32_t*)take(rows * 4);
  *idx_alt = (uint32_t*)take(rows * 4);
  S->seg = (int*)take((ni + 1) * 4);
  S->skip = (uint32_t*)take(ni * 4);
  *cub_tmp = take(cub_bytes);
  return off;
}

// builds, sorts and checks the spread tables of `ni` instances; returns the order (sorted position -> table row) in *order
int build_spread_tables(SpreadSort S, uint64_t ni, void* cub_tmp, uint64_t cub_bytes, uint64_t* key_alt, uint32_t* idx_alt, const uint32_t** order,
                        cudaStream_t st) {
  const dim3 grid((S.n_vals + 255) / 256, (unsigned)ni);
  k_spread_rows<<<grid, 256, 0, st>>>(S);
  CUDA_TRY(cudaGetLastError());
  cub::DoubleBuffer<uint64_t> keys(S.key, key_alt);
  cub::DoubleBuffer<uint32_t> rows(S.idx, idx_alt);
  for (uint32_t limb = 0; limb < 4; limb++) {
    if (limb) {
      k_spread_key<<<grid, 256, 0, st>>>(S, rows.Current(), keys.Current(), limb);
      CUDA_TRY(cudaGetLastError());
    }
    size_t tmp = cub_bytes;
    CUDA_TRY(cub::DeviceSegmentedSort::StableSortPairs(cub_tmp, tmp, keys, rows, (int)(ni * S.n_vals), (int)ni, S.seg, S.seg + 1, st));
  }
  k_spread_sorted<<<grid, 256, 0, st>>>(S, rows.Current());
  CUDA_TRY(cudaGetLastError());
  *order = rows.Current();
  return H2SHA_OK;
}

// per-instance challenges: every row of a host array [n][4] must be a reduced field element
int check_challenge_rows(const uint64_t* a, uint64_t n, const char* name) {
  for (uint64_t i = 0; i < n; i++)
    if (fr::geq_p(a + 4 * i)) return set_err(H2SHA_EINVAL, std::string(name) + " row " + std::to_string(i) + " is not a reduced field element");
  return H2SHA_OK;
}

// host rows [n][4] of theta, beta, gamma (each may be null: zeros) -> the engine's device array [n][3][4].  The copy goes through a
// pageable vector, so it is staged before the call returns and the caller may reuse its arrays at once.
int stage_challenges(h2sha_engine* e, uint64_t n, const uint64_t* theta, const uint64_t* beta, const uint64_t* gamma, cudaStream_t st) {
  std::vector<uint64_t> host(n * 12, 0);
  const uint64_t* src[3] = {theta, beta, gamma};
  for (uint64_t i = 0; i < n; i++)
    for (int c = 0; c < 3; c++)
      if (src[c]) memcpy(&host[i * 12 + c * 4], src[c] + 4 * i, 32);
  const uint64_t need = host.size() * 8;
  if (need > e->chal_bytes) {
    cudaFree(e->d_chal); e->d_chal = nullptr; e->chal_bytes = 0;
    CUDA_TRY(cudaMalloc(&e->d_chal, need));
    e->chal_bytes = need;
  }
  CUDA_TRY(cudaMemcpyAsync(e->d_chal, host.data(), need, cudaMemcpyHostToDevice, st));
  return H2SHA_OK;
}

bool u256_less(const U256& a, const U256& b) {
  for (int i = 3; i >= 0; i--)
    if (a.l[i] != b.l[i]) return a.l[i] < b.l[i];
  return false;
}

// the range table's values in Montgomery form (e->d_range_tab), built on first use
int ensure_range_tab(h2sha_engine* e, cudaStream_t st) {
  if (e->d_range_tab) return H2SHA_OK;
  const uint32_t n_vals = 1u << e->plan.cfg.lookup_bits;
  CUDA_TRY(cudaMalloc(&e->d_range_tab, (size_t)n_vals * 32));
  k_range_table<<<(n_vals + 255) / 256, 256, 0, st>>>(e->d_range_tab, n_vals);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(st));   // one-time: later calls may come on another stream
  return H2SHA_OK;
}

// compressed table expression dense * theta + spread of every spread-table row (halo2 `compress_expressions`), Montgomery form,
// in table-row order: 2^num_bits_lookup field multiplications, done on the host with the plan-time helpers
std::vector<U256> compressed_spread_table(const U256& theta_mont, uint32_t limb_bits) {
  static const U256 r2 = fr::to_mont(fr::mont_r());   // R^2 mod p: mont_mul(v, r2) = Montgomery form of v
  std::vector<U256> rows(1u << limb_bits);
  for (uint32_t i = 0; i < rows.size(); i++) {
    uint64_t sp = 0;
    for (uint32_t b = 0; b < limb_bits; b++) sp |= (uint64_t)((i >> b) & 1u) << (2 * b);   // spread.rs:171-180
    rows[i] = fr::add(fr::mont_mul(theta_mont, fr::mont_mul(fr::from_u64(i), r2)), fr::mont_mul(fr::from_u64(sp), r2));
  }
  return rows;
}

}  // namespace

extern "C" {

int h2sha_get_lookup_info(const h2sha_engine_t* e, h2sha_lookup_info_t* out) {
  if (!e || !out) return set_err(H2SHA_EINVAL, "null argument");
  const LookupGeom G = lookup_geom(e->plan);
  out->n_range_lookups = G.n_lookup_cols;
  out->n_spread_lookups = G.spread_cols;
  out->range_table_rows = 1u << G.lookup_bits;
  out->spread_table_rows = 1u << G.limb_bits;
  out->min_usable_rows = G.min_usable_rows();
  out->mult_words_per_instance = G.mult_words();
  return H2SHA_OK;
}

int h2sha_lookup_multiplicities(h2sha_engine_t* e, uint64_t n_instances, const void* lookup, const void* spread, uint32_t usable_rows,
                                uint32_t* mult_dev, uint32_t* not_in_table_dev, void* stream) {
  if (!e || !mult_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  if (!lookup && !spread) return set_err(H2SHA_EINVAL, "neither the lookup nor the spread buffer was given");
  const LookupGeom G = lookup_geom(e->plan, usable_rows);
  if (usable_rows < G.min_usable_rows()) return set_err(H2SHA_EINVAL, "usable_rows is smaller than an assigned column or a lookup table");
  if (n_instances == 0) return H2SHA_OK;
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t mult_words = G.mult_words(), range_words = G.range_words();
  // only the halves whose buffer was given are (re)computed
  if (lookup && spread) {
    CUDA_TRY(cudaMemsetAsync(mult_dev, 0, n_instances * mult_words * 4, st));
  } else {
    const uint64_t off = lookup ? 0 : range_words, cnt = lookup ? range_words : mult_words - range_words;
    CUDA_TRY(cudaMemset2DAsync(mult_dev + off, mult_words * 4, 0, cnt * 4, n_instances, st));
  }
  if (not_in_table_dev) CUDA_TRY(cudaMemsetAsync(not_in_table_dev, 0, 4, st));
  // grid.y = instance: at most 65535 per launch
  for (uint64_t i0 = 0; i0 < n_instances; i0 += 65535) {
    const unsigned ni = (unsigned)std::min<uint64_t>(65535, n_instances - i0);
    uint32_t* m0 = mult_dev + i0 * mult_words;
    if (lookup) {
      const unsigned tiles = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((G.n_lookup + 255) / 256, 64));
      k_range_mult<<<dim3(tiles, ni), 256, 0, st>>>(G, (const uint64_t*)lookup + i0 * G.lookup_inst_cells * 4, m0, not_in_table_dev);
      CUDA_TRY(cudaGetLastError());
    }
    if (spread) {
      const unsigned tiles = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((G.n_limb + 1023) / 1024, 32));
      const size_t smem = (size_t)G.spread_cols * (1u << G.limb_bits) * 4;
      if (smem > 48 * 1024) return set_err(H2SHA_EINVAL, "spread histogram does not fit in shared memory");
      k_spread_mult<<<dim3(tiles, ni), 256, smem, st>>>(G, (const uint64_t*)spread + i0 * G.spread_inst_cells * 4, m0, not_in_table_dev);
      CUDA_TRY(cudaGetLastError());
    }
  }
  return H2SHA_OK;
}

}  // extern "C"

namespace {
// mult_dev == null: the multiplicities come from the engine's raw value lists (instances first_raw .. of the last keep_lookup_raw batch).
// per_inst: theta_mont is [n_instances][4] (rows checked by the caller), errors_dev is [n_instances], and a spread lookup sorts one
// table per instance on the device.
int permute_lookup_impl(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint64_t first_raw, uint32_t usable_rows,
                        const uint64_t* theta_mont, bool per_inst, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !permuted_input_dev || !permuted_table_dev) return set_err(H2SHA_EINVAL, "null argument");
  const bool from_raw = mult_dev == nullptr;
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  const LookupGeom G = lookup_geom(e->plan, usable_rows);
  const LookupSel L = select_lookup(G, lookup_idx);
  if (!L.valid) return set_err(H2SHA_EINVAL, "bad lookup index");
  const bool is_range = L.is_range;
  if (!is_range && !theta_mont) return set_err(H2SHA_EINVAL, "a spread lookup has two expressions: theta is needed to compress them");
  if (usable_rows < G.min_usable_rows()) return set_err(H2SHA_EINVAL, "usable_rows is smaller than an assigned column or a lookup table");
  if (n_instances == 0) return H2SHA_OK;
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t n_vals = L.n_vals;
  // workspace: scans + totals of one chunk of instances (the chunks run one after the other on `stream` and share it)
  if (n_vals > (1u << 22)) return set_err(H2SHA_EINVAL, "lookup table too large for the permutation workspace (lookup_bits > 22)");
  // instances per pass: at most `lkchunk` (default 256) and at most ~1 GB of scans (and per-instance spread tables)
  const uint64_t per_inst_words = 3ull * n_vals + 4 + (is_range ? (uint64_t)usable_rows + n_vals : 0) + (from_raw ? align_up(n_vals, 4) : 0);   // scans, totals, inverse maps (identity order), this lookup's bins
  const bool sort_tabs = per_inst && !is_range;
  const uint64_t per_inst_bytes = per_inst_words * 4 + (sort_tabs ? 88ull * n_vals + 8 : 0);
  const uint64_t by_mem = std::max<uint64_t>(1, (1ull << 30) / per_inst_bytes);
  const uint64_t chunk = std::min<uint64_t>(std::min<uint64_t>(n_instances, by_mem), (uint64_t)std::max(1, tune_value("lkchunk", 256)));
  // workspace: [per-instance spread tables of a chunk] [bins of a chunk (from_raw)] [scans, totals, inverse maps of a chunk]
  size_t cub_bytes = 0;
  uint64_t sort_bytes = 0;
  if (sort_tabs) {
    cub::DoubleBuffer<uint64_t> k0(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> v0(nullptr, nullptr);
    CUDA_TRY(cub::DeviceSegmentedSort::StableSortPairs(nullptr, cub_bytes, k0, v0, (int)(chunk * n_vals), (int)chunk, (int*)nullptr, (int*)nullptr, st));
    SpreadSort S0{};
    void* t0; uint64_t* ka0; uint32_t* ia0;
    sort_bytes = spread_sort_layout(chunk, n_vals, cub_bytes, nullptr, &S0, &t0, &ka0, &ia0);
  }
  const uint64_t need = sort_bytes + chunk * per_inst_words * 4;
  if (need > e->lk_ws_bytes) {
    cudaFree(e->d_lk_ws); e->d_lk_ws = nullptr; e->lk_ws_bytes = 0;
    CUDA_TRY(cudaMalloc(&e->d_lk_ws, need));
    e->lk_ws_bytes = need;
  }
  PermuteArgs A{};
  SpreadSort S{};
  void* cub_tmp = nullptr;
  uint64_t* key_alt = nullptr;
  uint32_t* idx_alt = nullptr;
  if (sort_tabs) {
    spread_sort_layout(chunk, n_vals, cub_bytes, (uint8_t*)e->d_lk_ws, &S, &cub_tmp, &key_alt, &idx_alt);
    int rc = stage_challenges(e, n_instances, theta_mont, nullptr, nullptr, st);
    if (rc) return rc;
    S.n_vals = n_vals;
    A.vals = S.vals; A.tab_stride = n_vals; A.skip = S.skip;
  }
  uint32_t* raw_bins = nullptr;   // from_raw: [chunk][n_vals] (16-byte aligned rows for the vectorised scan)
  uint32_t* ws = e->d_lk_ws + sort_bytes / 4;
  if (from_raw) {
    raw_bins = ws;
    ws += chunk * (uint64_t)align_up(n_vals, 4);
    A.mult_stride = align_up(n_vals, 4);
    A.mult = raw_bins;
  } else {
    A.mult_stride = G.mult_words();
    A.mult = mult_dev + L.mult_off;
  }
  A.n_vals = n_vals; A.usable_rows = usable_rows;
  A.scan = ws; A.totals = ws + chunk * 3ull * n_vals;
  if (is_range && tune_value("lkinv", 1)) { A.vrow = A.totals + chunk * 4; A.llist = A.vrow + chunk * (uint64_t)usable_rows; }
  A.err_stride = per_inst ? 1u : 0u;
  A.out_input = (uint64_t*)permuted_input_dev; A.out_table = (uint64_t*)permuted_table_dev;
  if (is_range) {
    int rc = ensure_range_tab(e, st);
    if (rc) return rc;
    A.vals = tune_value("lktab", 1) ? e->d_range_tab : nullptr;   // lktab=0: convert each value on the fly (mont_from_u32) instead of the 32-byte gather
  } else if (!sort_tabs) {
    // the compressed table rows sorted by canonical value (`impl Ord for Fr`)
    U256 th_m; memcpy(th_m.l, theta_mont, 32);
    if (fr::geq_p(th_m.l)) return set_err(H2SHA_EINVAL, "theta is not a reduced field element");
    const std::vector<U256> cm = compressed_spread_table(th_m, G.limb_bits);
    struct Row { U256 c, cm; uint32_t row; };
    std::vector<Row> rows(n_vals);
    for (uint32_t i = 0; i < n_vals; i++) {
      rows[i].cm = cm[i];
      rows[i].c = fr::mont_mul(rows[i].cm, fr::from_u64(1));   // canonical value: what `Ord` compares
      rows[i].row = i;
    }
    std::stable_sort(rows.begin(), rows.end(), [](const Row& a, const Row& b) { return u256_less(a.c, b.c); });
    for (uint32_t i = 0; i + 1 < n_vals; i++)
      if (rows[i].c == rows[i + 1].c) return set_err(H2SHA_EINVAL, "theta makes two spread-table rows collide");
    std::vector<uint32_t> host(n_vals * 9);   // values (16-byte aligned for the 128-bit loads), then the order
    for (uint32_t i = 0; i < n_vals; i++) {
      host[8 * n_vals + i] = rows[i].row;
      memcpy(&host[8 * i], rows[i].cm.l, 32);
    }
    if (!e->d_lk_tab) CUDA_TRY(cudaMalloc(&e->d_lk_tab, host.size() * 4));   // n_vals = 2^num_bits_lookup: fixed per engine
    CUDA_TRY(cudaMemcpyAsync(e->d_lk_tab, host.data(), host.size() * 4, cudaMemcpyHostToDevice, st));   // pageable: staged before return
    A.vals = e->d_lk_tab; A.order = e->d_lk_tab + 8 * n_vals;
  }
  const uint32_t* mult0 = A.mult;
  for (uint64_t i0 = 0; i0 < n_instances; i0 += chunk) {
    const uint64_t ni = std::min<uint64_t>(chunk, n_instances - i0);
    if (from_raw) {
      MultOneArgs M{};
      M.lookup_raw = e->d_lookup_raw; M.dense_raw = e->d_dense_raw; M.out = raw_bins; M.bad = nullptr; M.first = first_raw + i0;
      M.n_vals = n_vals; M.is_range = is_range ? 1u : 0u; M.col = L.col; M.G = G;
      if (A.mult_stride != n_vals) return set_err(H2SHA_EINVAL, "lookup tables of fewer than 4 rows are not supported by the raw-list path");
      k_mult_one<<<(unsigned)ni, 512, 0, st>>>(M);
      CUDA_TRY(cudaGetLastError());
    } else {
      A.mult = mult0 + i0 * A.mult_stride;
    }
    if (sort_tabs) {
      S.chal = e->d_chal + i0 * 12;
      int rc = build_spread_tables(S, ni, cub_tmp, cub_bytes, key_alt, idx_alt, &A.order, st);
      if (rc) return rc;
    }
    A.errors = errors_dev ? errors_dev + (per_inst ? i0 : 0) : nullptr;
    A.out_input = (uint64_t*)permuted_input_dev + i0 * (uint64_t)usable_rows * 4;
    A.out_table = (uint64_t*)permuted_table_dev + i0 * (uint64_t)usable_rows * 4;
    {
      const bool aligned = A.order == nullptr && (A.mult_stride & 3u) == 0 && ((uintptr_t)A.mult & 15u) == 0;
      if (aligned && (A.n_vals % (1024u * 4u)) == 0) k_permute_scan<4><<<(unsigned)ni, 1024, 0, st>>>(A);
      else k_permute_scan<1><<<(unsigned)ni, 1024, 0, st>>>(A);
    }
    CUDA_TRY(cudaGetLastError());
    const uint64_t min_tiles = (uint64_t)std::max(1, tune_value("lktiles", A.vrow ? 64 : 16));   // more rows in flight when a row costs one or two loads
    const unsigned tiles = (unsigned)std::min<uint64_t>((usable_rows + 255) / 256, std::max<uint64_t>(min_tiles, ((uint64_t)e->n_sms * 16 + ni - 1) / ni));
    k_permute_fill<<<dim3(tiles, (unsigned)ni), 256, 0, st>>>(A);
    CUDA_TRY(cudaGetLastError());
  }
  return H2SHA_OK;
}
}  // namespace

extern "C" {

int h2sha_permute_lookup(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows,
                         const uint64_t* theta_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
  if (!mult_dev) return set_err(H2SHA_EINVAL, "null argument");
  return permute_lookup_impl(e, n_instances, lookup_idx, mult_dev, 0, usable_rows, theta_mont, false, permuted_input_dev, permuted_table_dev, errors_dev, stream);
}

int h2sha_permute_lookup_from_raw(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, uint32_t lookup_idx, uint32_t usable_rows,
                                  const uint64_t* theta_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  if (first_instance + n_instances > e->raw_n)
    return set_err(H2SHA_EINVAL, "the engine holds no raw value lists for these instances: generate the batch with keep_lookup_raw (or lookup_mult_dev) first");
  return permute_lookup_impl(e, n_instances, lookup_idx, nullptr, first_instance, usable_rows, theta_mont, false, permuted_input_dev, permuted_table_dev, errors_dev, stream);
}

// the checks of the per-instance calls that need no device: the plan-only engine is refused after them, by permute_lookup_impl
static int check_permute_per_instance(const h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint64_t* thetas_mont) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  const LookupSel L = select_lookup(lookup_geom(e->plan), lookup_idx);
  if (L.valid && !L.is_range && !thetas_mont) return set_err(H2SHA_EINVAL, "a spread lookup has two expressions: thetas_mont is needed to compress them");
  return !L.is_range && thetas_mont ? check_challenge_rows(thetas_mont, n_instances, "thetas_mont") : H2SHA_OK;
}

int h2sha_permute_lookup_per_instance(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows,
                                      const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
  if (!mult_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (int rc = check_permute_per_instance(e, n_instances, lookup_idx, thetas_mont)) return rc;
  return permute_lookup_impl(e, n_instances, lookup_idx, mult_dev, 0, usable_rows, thetas_mont, true, permuted_input_dev, permuted_table_dev, errors_dev, stream);
}

int h2sha_permute_lookup_from_raw_per_instance(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, uint32_t lookup_idx, uint32_t usable_rows,
                                               const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
  if (int rc = check_permute_per_instance(e, n_instances, lookup_idx, thetas_mont)) return rc;
  if (first_instance + n_instances > e->raw_n)
    return set_err(H2SHA_EINVAL, "the engine holds no raw value lists for these instances: generate the batch with keep_lookup_raw (or lookup_mult_dev) first");
  return permute_lookup_impl(e, n_instances, lookup_idx, nullptr, first_instance, usable_rows, thetas_mont, true, permuted_input_dev, permuted_table_dev, errors_dev, stream);
}

}  // extern "C"
