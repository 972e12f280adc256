// lookup_product.cuh -- the lookup argument's grand-product column z on the device (SURVEY.md §8f #4), the step after
// the permutation: PSE halo2_proofs plonk/lookup/prover.rs `Permuted::commit_product`, for one lookup of every instance.
// Included at the end of engine.cu, after lookup_prework.cuh (LookupGeom, load_cell, ensure_range_tab) and batch_check.cuh
// (mont_mul_dev, fr_add_dev).
//
//   u_i = (A[i] + beta)(S[i] + gamma),  v_i = (A'[i] + beta)(S'[i] + gamma),  i < U = usable_rows
//   z[0] = 1,  z[j+1] = z[j] * u_j / v_j                                      (U + 1 values)
// commit_product inverts the v with ff's `batch_invert`, which leaves a zero as zero: a row with v_i = 0 contributes the
// fraction 0 and every later z is 0.  That is (u_i, v_i) := (0, 1) here.
//
// One field inversion per instance, no per-row inversion (rows split into tiles of LP_TILE contiguous rows):
//   k_product_tiles   grid (tiles, instances): the tile products prod u, prod v -> workspace (rows taken strided: a product
//                     does not care about order, and the loads coalesce);
//   k_product_fold    one warp per instance: exclusive prefix of the tile products of u, exclusive suffix of those of v, one
//                     Fermat inversion of prod v, per tile C_t = U_<t / V_<=t; z[U] = prod u / prod v, counted when != 1;
//   k_product_fill    grid (tiles, instances), LP_ROWS contiguous rows per thread:
//                     z[j] = C_t * (prod_{t0 <= i < j} u_i) * (prod_{j <= i < t1} v_i)
//                     (thread segment in registers, then warp shuffles of the 4-limb values, then the CTA), one 256-bit store a row.
// Bound: integer multiply-adds (about 12 Montgomery products per row, 14 for a spread lookup; DESIGN.md §4b), not HBM: 224 B of traffic per row.
#pragma once

namespace {

enum { LP_THREADS = 256, LP_ROWS = 8, LP_TILE = LP_THREADS * LP_ROWS, LP_FOLD_WARPS = 4 };

struct ProductArgs {
  const uint64_t* cells;        // the lookup's witness buffer (lookup or spread) at instance 0 of the launch
  uint64_t inst_cells;          // Fr per instance in that buffer
  uint64_t col_off;             // Fr offset of the looked-up column (range) / the dense column (spread) inside an instance
  uint64_t spread_off;          // spread lookups: Fr distance from a dense cell to its spread cell
  uint32_t used;                // assigned rows of that column; the rows above hold 0
  uint32_t is_spread;
  const uint64_t* a_p;          // [n][usable_rows] Fr: A', S'
  const uint64_t* s_p;
  const uint64_t* tab;          // [n_vals] Fr: the table expression in table-row order (padded rows hold 0)
  uint32_t n_vals, usable_rows, n_tiles;
  uint64_t theta[4], beta[4], gamma[4];   // Montgomery
  uint64_t* tiles;              // [n][n_tiles][2][4]: prod u, prod v of each tile
  uint64_t* consts;             // [n][n_tiles][4]: C_t
  uint64_t* z;                  // [n][usable_rows + 1] Fr
  uint32_t* errors;             // may be null
};

__device__ __forceinline__ void fr_one(uint64_t r[4]) { r[0] = c_fr.r1[0]; r[1] = c_fr.r1[1]; r[2] = c_fr.r1[2]; r[3] = c_fr.r1[3]; }
__device__ __forceinline__ bool fr_is_zero(const uint64_t x[4]) { return (x[0] | x[1] | x[2] | x[3]) == 0; }
__device__ __forceinline__ void fr_copy(const uint64_t x[4], uint64_t r[4]) { r[0] = x[0]; r[1] = x[1]; r[2] = x[2]; r[3] = x[3]; }
__device__ __forceinline__ void store_fr(uint64_t* p, const uint64_t x[4]) {
  store_cell2(reinterpret_cast<uint32_t*>(p), make_uint4((uint32_t)x[0], (uint32_t)(x[0] >> 32), (uint32_t)x[1], (uint32_t)(x[1] >> 32)),
              make_uint4((uint32_t)x[2], (uint32_t)(x[2] >> 32), (uint32_t)x[3], (uint32_t)(x[3] >> 32)));
}
__device__ __forceinline__ void fr_mul_into(uint64_t acc[4], const uint64_t x[4]) {
  uint64_t t[4];
  mont_mul_dev(acc, x, t);
  fr_copy(t, acc);
}
__device__ __forceinline__ void fr_shfl_up(const uint64_t x[4], uint32_t o, uint64_t r[4]) {
#pragma unroll
  for (int q = 0; q < 4; q++) r[q] = __shfl_up_sync(0xffffffffu, x[q], o);
}
__device__ __forceinline__ void fr_shfl_down(const uint64_t x[4], uint32_t o, uint64_t r[4]) {
#pragma unroll
  for (int q = 0; q < 4; q++) r[q] = __shfl_down_sync(0xffffffffu, x[q], o);
}
__device__ __forceinline__ void fr_shfl(const uint64_t x[4], uint32_t lane, uint64_t r[4]) {
#pragma unroll
  for (int q = 0; q < 4; q++) r[q] = __shfl_sync(0xffffffffu, x[q], lane);
}

// x^(p-2) (Fermat), x != 0; Montgomery in and out
__device__ void fr_inv_dev(const uint64_t x[4], uint64_t r[4]) {
  const uint64_t e[4] = {c_fr.p[0] - 2, c_fr.p[1], c_fr.p[2], c_fr.p[3]};   // p[0] is odd and > 2: no borrow
  fr_one(r);
  for (int b = 253; b >= 0; b--) {   // p < 2^254
    fr_mul_into(r, r);
    if ((e[b >> 6] >> (b & 63)) & 1u) fr_mul_into(r, x);
  }
}

// u_i and v_i of row i < usable_rows of instance `inst` (zero rule applied)
__device__ __forceinline__ void product_terms(const ProductArgs& A, uint64_t inst, uint32_t i, uint64_t u[4], uint64_t v[4]) {
  uint64_t x[4] = {0, 0, 0, 0}, y[4] = {0, 0, 0, 0}, t[4];
  if (i < A.used) {
    const uint64_t* c = A.cells + (inst * A.inst_cells + A.col_off + i) * 4;
    load_cell(c, x);
    if (A.is_spread) {   // dense * theta + spread (halo2 `compress_expressions`)
      mont_mul_dev(A.theta, x, t);
      load_cell(c + A.spread_off * 4, y);
      fr_add_dev(t, y, x);
    }
  }
  fr_add_dev(x, A.beta, t);
  if (i < A.n_vals) load_cell(A.tab + (uint64_t)i * 4, y);
  else y[0] = y[1] = y[2] = y[3] = 0;
  fr_add_dev(y, A.gamma, x);
  mont_mul_dev(t, x, u);
  const uint64_t row = inst * A.usable_rows + i;
  load_cell(A.a_p + row * 4, x);
  fr_add_dev(x, A.beta, t);
  load_cell(A.s_p + row * 4, y);
  fr_add_dev(y, A.gamma, x);
  mont_mul_dev(t, x, v);
  if (fr_is_zero(v)) {   // batch_invert leaves the zero denominator as 0: fraction 0
    u[0] = u[1] = u[2] = u[3] = 0;
    fr_one(v);
  }
}

__global__ void __launch_bounds__(LP_THREADS) k_product_tiles(const ProductArgs A) {
  __shared__ uint64_t s_w[LP_THREADS / 32][2][4];
  const uint64_t inst = blockIdx.y;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t t0 = blockIdx.x * (uint32_t)LP_TILE;
  uint64_t pu[4], pv[4], u[4], v[4];
  fr_one(pu); fr_one(pv);
  if (t0 + threadIdx.x < A.usable_rows) product_terms(A, inst, t0 + threadIdx.x, pu, pv);
#pragma unroll 1
  for (uint32_t r = 1; r < LP_ROWS; r++) {
    const uint32_t i = t0 + r * LP_THREADS + threadIdx.x;
    if (i >= A.usable_rows) break;
    product_terms(A, inst, i, u, v);
    fr_mul_into(pu, u);
    fr_mul_into(pv, v);
  }
#pragma unroll
  for (uint32_t o = 16; o > 0; o >>= 1) {
    fr_shfl_down(pu, o, u);
    fr_shfl_down(pv, o, v);
    fr_mul_into(pu, u);   // lanes >= 32 - o fold garbage, but only lane 0's result is used
    fr_mul_into(pv, v);
  }
  if (lane == 0) { fr_copy(pu, s_w[warp][0]); fr_copy(pv, s_w[warp][1]); }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < LP_THREADS / 32; w++) { fr_mul_into(pu, s_w[w][0]); fr_mul_into(pv, s_w[w][1]); }
    uint64_t* out = A.tiles + (inst * A.n_tiles + blockIdx.x) * 8;
    fr_copy(pu, out); fr_copy(pv, out + 4);
  }
}

// one warp per instance; lane l folds tiles [l*q, (l+1)*q)
__global__ void __launch_bounds__(32 * LP_FOLD_WARPS) k_product_fold(const ProductArgs A, uint32_t n_inst) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t inst = (uint64_t)blockIdx.x * LP_FOLD_WARPS + (threadIdx.x >> 5);
  if (inst >= n_inst) return;   // whole warps
  const uint64_t* tl = A.tiles + inst * A.n_tiles * 8;
  uint64_t* cs = A.consts + inst * A.n_tiles * 4;
  const uint32_t q = (A.n_tiles + 31) / 32, ta = min(lane * q, A.n_tiles), tb = min(ta + q, A.n_tiles);
  uint64_t lu[4], lv[4], x[4], y[4];
  fr_one(lu); fr_one(lv);
  for (uint32_t t = ta; t < tb; t++) { fr_mul_into(lu, tl + t * 8); fr_mul_into(lv, tl + t * 8 + 4); }
  // inclusive prefix of lu, inclusive suffix of lv over the lanes
#pragma unroll
  for (uint32_t o = 1; o < 32; o <<= 1) {
    fr_shfl_up(lu, o, x);
    fr_shfl_down(lv, o, y);
    if (lane >= o) fr_mul_into(lu, x);
    if (lane + o < 32) fr_mul_into(lv, y);
  }
  uint64_t u_all[4], v_all[4], inv[4], upre[4], vsuf[4];
  fr_shfl(lu, 31, u_all);
  fr_shfl(lv, 0, v_all);
  fr_shfl_up(lu, 1, upre);
  fr_shfl_down(lv, 1, vsuf);
  if (lane == 0) fr_one(upre);
  if (lane == 31) fr_one(vsuf);
  fr_inv_dev(v_all, inv);   // v_all != 0: every v is nonzero after the zero rule
  // C_t = U_<t * inv * prod_{t' > t} v_t'  (= U_<t / V_<=t)
  mont_mul_dev(vsuf, inv, y);
  for (uint32_t t = tb; t-- > ta;) {
    store_fr(cs + t * 4, y);
    fr_mul_into(y, tl + t * 8 + 4);
  }
  for (uint32_t t = ta; t < tb; t++) {
    load_cell(cs + t * 4, x);
    mont_mul_dev(upre, x, y);
    store_fr(cs + t * 4, y);
    fr_mul_into(upre, tl + t * 8);
  }
  if (lane == 0) {
    mont_mul_dev(u_all, inv, y);   // z[U]
    uint64_t* zu = A.z + (inst * (A.usable_rows + 1ull) + A.usable_rows) * 4;
    store_fr(zu, y);
    fr_one(x);
    if (((y[0] ^ x[0]) | (y[1] ^ x[1]) | (y[2] ^ x[2]) | (y[3] ^ x[3])) && A.errors) atomicAdd(A.errors, 1u);
  }
}

__global__ void __launch_bounds__(LP_THREADS) k_product_fill(const ProductArgs A) {
  __shared__ uint64_t s_w[LP_THREADS / 32][2][4];   // per warp: inclusive product of u, of v; then the warp's constant
  const uint64_t inst = blockIdx.y;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t s = blockIdx.x * (uint32_t)LP_TILE + threadIdx.x * LP_ROWS;
  uint64_t u[LP_ROWS][4], sv[LP_ROWS][4];   // u of each row; v, then the suffix products of v inside the segment
#pragma unroll
  for (int r = 0; r < LP_ROWS; r++) {
    if (s + r < A.usable_rows) product_terms(A, inst, s + r, u[r], sv[r]);
    else { fr_one(u[r]); fr_one(sv[r]); }
  }
#pragma unroll
  for (int r = LP_ROWS - 2; r >= 0; r--) fr_mul_into(sv[r], sv[r + 1]);
  uint64_t pu[4], pv[4], x[4], y[4];
  fr_copy(u[0], pu);
#pragma unroll
  for (int r = 1; r < LP_ROWS; r++) fr_mul_into(pu, u[r]);
  fr_copy(sv[0], pv);
  // inclusive prefix of pu, inclusive suffix of pv over the warp
#pragma unroll
  for (uint32_t o = 1; o < 32; o <<= 1) {
    fr_shfl_up(pu, o, x);
    fr_shfl_down(pv, o, y);
    if (lane >= o) fr_mul_into(pu, x);
    if (lane + o < 32) fr_mul_into(pv, y);
  }
  if (lane == 31) fr_copy(pu, s_w[warp][0]);
  if (lane == 0) fr_copy(pv, s_w[warp][1]);
  fr_shfl_up(pu, 1, x);     // exclusive
  fr_shfl_down(pv, 1, y);
  if (lane == 0) fr_one(x);
  if (lane == 31) fr_one(y);
  __syncthreads();
  if (threadIdx.x == 0) {
    // K_w = C_t * (prod u of the warps before w) * (prod v of the warps after w)
    uint64_t c[4], acc[4], k[LP_THREADS / 32][4];
    load_cell(A.consts + (inst * A.n_tiles + blockIdx.x) * 4, c);
    fr_copy(c, acc);
    for (int w = 0; w < LP_THREADS / 32; w++) { fr_copy(acc, k[w]); fr_mul_into(acc, s_w[w][0]); }
    fr_one(acc);
    for (int w = LP_THREADS / 32 - 1; w >= 0; w--) { fr_mul_into(k[w], acc); fr_mul_into(acc, s_w[w][1]); }
    for (int w = 0; w < LP_THREADS / 32; w++) fr_copy(k[w], s_w[w][0]);
  }
  __syncthreads();
  uint64_t w[4];
  mont_mul_dev(s_w[warp][0], x, pu);
  mont_mul_dev(pu, y, w);   // z[s] / sv[0]: the product of u before the segment over the product of v from its end on
  uint64_t* zr = A.z + (inst * (A.usable_rows + 1ull) + s) * 4;
#pragma unroll
  for (int r = 0; r < LP_ROWS; r++) {
    if (s + r >= A.usable_rows) break;
    mont_mul_dev(w, sv[r], x);
    store_fr(zr + r * 4, x);
    if (r + 1 < LP_ROWS) fr_mul_into(w, u[r]);
  }
}

}  // namespace

extern "C" {

int h2sha_lookup_product(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                         const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows, const uint64_t* theta_mont,
                         const uint64_t* beta_mont, const uint64_t* gamma_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !permuted_input_dev || !permuted_table_dev || !beta_mont || !gamma_mont || !z_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  const Plan& P = e->plan;
  const uint32_t n_range = P.n_lookup_cols, n_spread = P.cfg.spread_cols;
  if (lookup_idx >= n_range + n_spread) return set_err(H2SHA_EINVAL, "bad lookup index");
  const bool is_range = lookup_idx < n_range;
  if (is_range ? !lookup : !spread) return set_err(H2SHA_EINVAL, "null argument: the witness buffer this lookup reads");
  if (!is_range && !theta_mont) return set_err(H2SHA_EINVAL, "a spread lookup has two expressions: theta is needed to compress them");
  if (usable_rows < lookup_rows_needed(P)) return set_err(H2SHA_EINVAL, "usable_rows is smaller than an assigned column or a lookup table");
  if (fr::geq_p(beta_mont) || fr::geq_p(gamma_mont) || (theta_mont && !is_range && fr::geq_p(theta_mont)))
    return set_err(H2SHA_EINVAL, "beta, gamma and theta must be reduced field elements");
  const void* bufs[] = {is_range ? lookup : spread, permuted_input_dev, permuted_table_dev, z_dev};
  for (const void* b : bufs)
    if ((uintptr_t)b & 31u) return set_err(H2SHA_EINVAL, "Fr buffers must be 32-byte aligned");
  if (n_instances == 0) return H2SHA_OK;
  CUDA_TRY(cudaSetDevice(e->device));
  int rc = ensure_lookup_consts(e);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const LookupGeom G = lookup_geom(e, n_instances, usable_rows);
  ProductArgs A{};
  A.n_vals = is_range ? (1u << G.lookup_bits) : (1u << G.limb_bits);
  A.usable_rows = usable_rows;
  A.n_tiles = (uint32_t)((usable_rows + (uint64_t)LP_TILE - 1) / LP_TILE);
  memcpy(A.beta, beta_mont, 32); memcpy(A.gamma, gamma_mont, 32);
  if (is_range) {
    const uint32_t first = lookup_idx * G.max_rows;
    A.cells = (const uint64_t*)lookup; A.inst_cells = G.lookup_inst_cells;
    A.col_off = (uint64_t)lookup_idx * G.lookup_col_rows;
    A.used = G.n_lookup > first ? std::min(G.max_rows, G.n_lookup - first) : 0u;   // range.finalize wraps at max_rows
  } else {
    const uint32_t col = lookup_idx - n_range;
    A.cells = (const uint64_t*)spread; A.inst_cells = G.spread_inst_cells;
    A.col_off = (uint64_t)col * G.spread_rows; A.spread_off = (uint64_t)G.spread_cols * G.spread_rows;
    A.used = G.n_limb > col ? (G.n_limb - col + G.spread_cols - 1) / G.spread_cols : 0u;   // limb n -> column n % cols, row n / cols
    A.is_spread = 1;
    memcpy(A.theta, theta_mont, 32);
  }
  // workspace: [spread table] [tile products of a chunk] [tile constants of a chunk]
  const uint64_t chunk = std::min<uint64_t>(std::min<uint64_t>(n_instances, 65535), (uint64_t)std::max(1, tune_value("lkchunk", 256)));
  const uint64_t tab_words = is_range ? 0 : (uint64_t)A.n_vals * 4;
  const uint64_t need = (tab_words + chunk * A.n_tiles * 12ull) * 8;
  if (need > e->lp_ws_bytes) {
    cudaFree(e->d_lp_ws); e->d_lp_ws = nullptr; e->lp_ws_bytes = 0;
    CUDA_TRY(cudaMalloc(&e->d_lp_ws, need));
    e->lp_ws_bytes = need;
  }
  A.tiles = e->d_lp_ws + tab_words;
  A.consts = A.tiles + chunk * A.n_tiles * 8;
  if (is_range) {
    if ((rc = ensure_range_tab(e, st))) return rc;
    A.tab = reinterpret_cast<const uint64_t*>(e->d_range_tab);
  } else {
    U256 th_m; memcpy(th_m.l, theta_mont, 32);
    const std::vector<U256> tab = compressed_spread_table(th_m, G.limb_bits);
    CUDA_TRY(cudaMemcpyAsync(e->d_lp_ws, tab.data(), tab.size() * 32, cudaMemcpyHostToDevice, st));   // pageable: staged before return
    A.tab = e->d_lp_ws;
  }
  A.errors = errors_dev;
  const uint64_t* cells0 = A.cells;
  for (uint64_t i0 = 0; i0 < n_instances; i0 += chunk) {
    const unsigned ni = (unsigned)std::min<uint64_t>(chunk, n_instances - i0);
    A.cells = cells0 + i0 * A.inst_cells * 4;
    A.a_p = (const uint64_t*)permuted_input_dev + i0 * usable_rows * 4;
    A.s_p = (const uint64_t*)permuted_table_dev + i0 * usable_rows * 4;
    A.z = (uint64_t*)z_dev + i0 * (usable_rows + 1ull) * 4;
    k_product_tiles<<<dim3(A.n_tiles, ni), LP_THREADS, 0, st>>>(A);
    CUDA_TRY(cudaGetLastError());
    k_product_fold<<<(ni + LP_FOLD_WARPS - 1) / LP_FOLD_WARPS, 32 * LP_FOLD_WARPS, 0, st>>>(A, ni);
    CUDA_TRY(cudaGetLastError());
    k_product_fill<<<dim3(A.n_tiles, ni), LP_THREADS, 0, st>>>(A);
    CUDA_TRY(cudaGetLastError());
  }
  return H2SHA_OK;
}

}  // extern "C"
