// grand_product.cuh -- the grand-product column z of a lookup (lookup_product.cuh) or of the permutation argument
// (permutation_product.cuh) on the device, for every instance of a batch, with one field inversion per instance.
// Included at the end of engine.cu, before those two files.
//
// The rows of an instance form chunks h = 0 .. n_chunks - 1 of `rows` rows each, and every row i contributes a fraction u_i / v_i:
//   z_h[0] = z_{h-1}[last] (1 for h = 0),  z_h[i+1] = z_h[i] * u_i / v_i
// so the fractions of all chunks are ONE sequence over (chunk, row), and the closing value, the last z of the instance, is
// prod u / prod v.  ff's `batch_invert` leaves a zero denominator as zero: a row with v_i = 0 contributes the fraction 0 and every
// later z is 0.  That is (u_i, v_i) := (0, 1) here.
// The caller's row source `Rows` says what the rows contribute:
//   void setup(inst)               run by the whole CTA before any row: loads what its instance needs into shared memory
//   bool any(h, i0, i1)            does some row in [i0, i1) of chunk h contribute a fraction other than 1?
//   bool terms(inst, h, i, u, v)   the raw u_i, v_i of row i < rows of chunk h; false (u, v unset) when the row contributes 1
// Rows split into tiles of GP_TILE contiguous rows of one chunk:
//   k_product_tiles   grid (tiles of all chunks, instances): the tile products prod u, prod v -> workspace (rows taken strided: a
//                     product does not care about order, and the loads coalesce);
//   k_product_fold    one warp per instance walks the tiles of all chunks in chain order: exclusive prefix of the tile products
//                     of u, exclusive suffix of those of v, one Fermat inversion of prod v, per tile C_t = U_<t / V_<=t; the
//                     closing value prod u / prod v, counted when != 1;
//   k_product_fill    grid (tiles of all chunks, instances), GP_ROWS contiguous rows per thread:
//                     z[j] = C_t * (prod_{t0 <= i < j} u_i) * (prod_{j <= i < t1} v_i)
//                     (thread segment in registers, then warp shuffles of the 4-limb values, then the CTA), one 256-bit store a
//                     row; a warp whose rows all contribute 1 only stores its constant.
#pragma once

namespace {

enum { GP_THREADS = 256, GP_ROWS = 8, GP_TILE = GP_THREADS * GP_ROWS, GP_FOLD_WARPS = 4 };

struct GrandProduct {
  uint32_t rows;                // rows of a chunk
  uint32_t n_chunks, tiles_per_chunk;
  uint32_t z_stride;            // z values of a chunk
  uint64_t* tiles;              // [n][n_chunks * tiles_per_chunk][2][4]: prod u, prod v of each tile
  uint64_t* consts;             // [n][n_chunks * tiles_per_chunk][4]: C_t
  uint64_t* z;                  // [n][n_chunks][z_stride] Fr
  uint32_t* errors;             // may be null
  uint32_t err_stride;          // 0: errors is one counter for the batch; 1: errors[inst] (the *_per_instance calls)
};

// the challenges of the CTA's instance for the row sources of the *_per_instance calls: theta, beta, gamma (Montgomery), loaded
// once per CTA from the staged [n][3][4] array instead of once per row (the fill kernel has no registers to spare for them)
__shared__ uint64_t s_chal[3][4];
__device__ __forceinline__ void load_chal(const uint64_t* chal, uint64_t inst) {
  if (threadIdx.x < 12) s_chal[threadIdx.x / 4][threadIdx.x % 4] = chal[inst * 12 + threadIdx.x];
  __syncthreads();
}

__device__ __forceinline__ void store_fr(uint64_t* p, const uint64_t x[4]) {
  store_cell2(reinterpret_cast<uint32_t*>(p), make_uint4((uint32_t)x[0], (uint32_t)(x[0] >> 32), (uint32_t)x[1], (uint32_t)(x[1] >> 32)),
              make_uint4((uint32_t)x[2], (uint32_t)(x[2] >> 32), (uint32_t)x[3], (uint32_t)(x[3] >> 32)));
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

// u, v of row i of chunk h with the zero rule applied; false when the row contributes 1
template <class Rows>
__device__ __forceinline__ bool row_terms(const Rows& R, uint64_t inst, uint32_t h, uint32_t i, uint64_t u[4], uint64_t v[4]) {
  if (!R.terms(inst, h, i, u, v)) return false;
  if (fr_is_zero(v)) {   // batch_invert leaves the zero denominator as 0: fraction 0
    u[0] = u[1] = u[2] = u[3] = 0;
    fr_one(v);
  }
  return true;
}

template <class Rows>
__global__ void __launch_bounds__(GP_THREADS) k_product_tiles(const GrandProduct G, const Rows R) {
  __shared__ uint64_t s_w[GP_THREADS / 32][2][4];
  __shared__ uint32_t s_any[GP_THREADS / 32];
  const uint64_t inst = blockIdx.y;
  R.setup(inst);
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t h = blockIdx.x / G.tiles_per_chunk, t0 = (blockIdx.x % G.tiles_per_chunk) * (uint32_t)GP_TILE;
  uint64_t pu[4], pv[4], u[4], v[4];
  fr_one(pu); fr_one(pv);
  bool mine = false;
#pragma unroll 1
  for (uint32_t r = 0; r < GP_ROWS; r++) {
    const uint32_t i = t0 + r * GP_THREADS + threadIdx.x;
    if (i >= G.rows) break;
    if (!row_terms(R, inst, h, i, u, v)) continue;
    if (mine) { fr_mul_into(pu, u); fr_mul_into(pv, v); }
    else { fr_copy(u, pu); fr_copy(v, pv); mine = true; }
  }
  const uint32_t any = __ballot_sync(0xffffffffu, mine);
  if (any) {
#pragma unroll
    for (uint32_t o = 16; o > 0; o >>= 1) {
      fr_shfl_down(pu, o, u);
      fr_shfl_down(pv, o, v);
      fr_mul_into(pu, u);   // lanes >= 32 - o fold garbage, but only lane 0's result is used
      fr_mul_into(pv, v);
    }
  }
  if (lane == 0) { fr_copy(pu, s_w[warp][0]); fr_copy(pv, s_w[warp][1]); s_any[warp] = any; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < GP_THREADS / 32; w++)
      if (s_any[w]) { fr_mul_into(pu, s_w[w][0]); fr_mul_into(pv, s_w[w][1]); }
    uint64_t* out = G.tiles + (inst * G.n_chunks * G.tiles_per_chunk + blockIdx.x) * 8;
    fr_copy(pu, out); fr_copy(pv, out + 4);
  }
}

// one warp per instance; lane l folds tiles [l*q, (l+1)*q)
__global__ void __launch_bounds__(32 * GP_FOLD_WARPS) k_product_fold(const GrandProduct G, uint32_t n_inst) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t inst = (uint64_t)blockIdx.x * GP_FOLD_WARPS + (threadIdx.x >> 5);
  if (inst >= n_inst) return;   // whole warps
  const uint32_t n_tiles = G.n_chunks * G.tiles_per_chunk;
  const uint64_t* tl = G.tiles + inst * n_tiles * 8;
  uint64_t* cs = G.consts + inst * n_tiles * 4;
  const uint32_t q = (n_tiles + 31) / 32, ta = min(lane * q, n_tiles), tb = min(ta + q, n_tiles);
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
    mont_mul_dev(u_all, inv, y);   // the closing value: the last z of the instance
    store_fr(G.z + ((inst + 1) * G.n_chunks * G.z_stride - 1) * 4, y);
    fr_one(x);
    if (((y[0] ^ x[0]) | (y[1] ^ x[1]) | (y[2] ^ x[2]) | (y[3] ^ x[3])) && G.errors) atomicAdd(G.errors + inst * G.err_stride, 1u);
  }
}

template <class Rows>
__global__ void __launch_bounds__(GP_THREADS) k_product_fill(const GrandProduct G, const Rows R) {
  __shared__ uint64_t s_w[GP_THREADS / 32][2][4];   // per warp: inclusive product of u, of v; then the warp's constant
  const uint64_t inst = blockIdx.y;
  R.setup(inst);
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t h = blockIdx.x / G.tiles_per_chunk;
  const uint32_t s = (blockIdx.x % G.tiles_per_chunk) * (uint32_t)GP_TILE + threadIdx.x * GP_ROWS;
  const bool mine = R.any(h, s, s + GP_ROWS);
  uint64_t u[GP_ROWS][4], sv[GP_ROWS][4];   // u of each row; v, then the suffix products of v inside the segment
  uint64_t pu[4], pv[4], x[4], y[4];
  if (mine) {
#pragma unroll
    for (int r = 0; r < GP_ROWS; r++)
      if (s + r >= G.rows || !row_terms(R, inst, h, s + r, u[r], sv[r])) { fr_one(u[r]); fr_one(sv[r]); }
#pragma unroll
    for (int r = GP_ROWS - 2; r >= 0; r--) fr_mul_into(sv[r], sv[r + 1]);
    fr_copy(u[0], pu);
#pragma unroll
    for (int r = 1; r < GP_ROWS; r++) fr_mul_into(pu, u[r]);
    fr_copy(sv[0], pv);
  } else {
    fr_one(pu); fr_one(pv);
  }
  const bool warp_any = __any_sync(0xffffffffu, mine);
  if (warp_any) {
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
  } else if (lane == 0) {
    fr_one(s_w[warp][0]); fr_one(s_w[warp][1]);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // K_w = C_t * (prod u of the warps before w) * (prod v of the warps after w)
    uint64_t c[4], acc[4], k[GP_THREADS / 32][4];
    load_cell(G.consts + (inst * G.n_chunks * G.tiles_per_chunk + blockIdx.x) * 4, c);
    fr_copy(c, acc);
    for (int w = 0; w < GP_THREADS / 32; w++) { fr_copy(acc, k[w]); fr_mul_into(acc, s_w[w][0]); }
    fr_one(acc);
    for (int w = GP_THREADS / 32 - 1; w >= 0; w--) { fr_mul_into(k[w], acc); fr_mul_into(acc, s_w[w][1]); }
    for (int w = 0; w < GP_THREADS / 32; w++) fr_copy(k[w], s_w[w][0]);
  }
  __syncthreads();
  uint64_t w[4];
  if (warp_any) {
    mont_mul_dev(s_w[warp][0], x, pu);
    mont_mul_dev(pu, y, w);   // z[s] / sv[0]: the product of u before the segment over the product of v from its end on
  } else {
    fr_copy(s_w[warp][0], w);
  }
  uint64_t* zr = G.z + ((inst * G.n_chunks + h) * G.z_stride + s) * 4;
  if (mine) {
#pragma unroll
    for (int r = 0; r < GP_ROWS; r++) {
      if (s + r >= G.rows) break;
      mont_mul_dev(w, sv[r], x);
      store_fr(zr + r * 4, x);
      if (r + 1 < GP_ROWS) fr_mul_into(w, u[r]);
    }
  } else {
#pragma unroll
    for (int r = 0; r < GP_ROWS; r++) {
      if (s + r >= G.rows) break;
      store_fr(zr + r * 4, w);
    }
  }
}

// the three kernels over `ni` instances, G.z and R at the first of them
template <class Rows>
int launch_product(const GrandProduct& G, const Rows& R, unsigned ni, cudaStream_t st) {
  const uint32_t n_tiles = G.n_chunks * G.tiles_per_chunk;
  k_product_tiles<<<dim3(n_tiles, ni), GP_THREADS, 0, st>>>(G, R);
  CUDA_TRY(cudaGetLastError());
  k_product_fold<<<(ni + GP_FOLD_WARPS - 1) / GP_FOLD_WARPS, 32 * GP_FOLD_WARPS, 0, st>>>(G, ni);
  CUDA_TRY(cudaGetLastError());
  k_product_fill<<<dim3(n_tiles, ni), GP_THREADS, 0, st>>>(G, R);
  CUDA_TRY(cudaGetLastError());
  return H2SHA_OK;
}

}  // namespace
