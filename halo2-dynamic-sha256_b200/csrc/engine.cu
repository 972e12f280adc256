// engine.cu -- sm_100a kernels and the C-ABI of the SHA-256 witness-generation engine (include/h2sha_b200.h).
//
// Kernels (see DESIGN.md for the roofline of each):
//   k_trace   one thread per message: padding (lib.rs:77-117), precomputed-prefix state (lib.rs:153-160),
//             then the scalar SHA-256 of every block with register-resident state, writing the 200-word
//             per-block trace (W[64], a/e working variables) and the digest.
//   k_trace_warp  the same for batches of <= 2048 messages, one warp per message: latency instead of throughput.
//   k_expand  persistent CTAs; one job = one sha256_compression (69 348 gate + 3 184 lookup + 8 240
//             spread-column cells) or one digest prologue/epilogue.  Phase 1 runs the planner's slot
//             programs (lanes = unit instances), phase 2 expands the templates: raw value -> BN254 Fr
//             Montgomery form -> one 256-bit store per cell (st.global.v8.b32, sm_100+), checksums folded
//             from registers.
// Included at the end of this translation unit (they use the engine struct and the field helpers above):
//   lookup_prework.cuh  k_range_mult / k_spread_mult / k_permute_scan / k_permute_fill: lookup-argument pre-work
//   batch_check.cuh     k_check_gates / k_check_pairs / k_check_digest_bytes: MockProver-style pass over a whole batch; h2sha_gather
// Build-time switches (never set for the product): H2SHA_DEBUG_TIMING (1 | 2: %globaltimer prints of the producer / consumer
// hand-over).
// There is no CPU path: every entry point fails with H2SHA_ECUDA when no device is usable.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/h2sha_b200.h"
#include "h2sha_defs.h"
#include "lookup_geom.h"
#include "permutation.h"
#include "planner.h"

using namespace h2sha;

extern "C" const uint32_t H2SHA_CK_M[8] = {0x9E3779B1u, 0x85EBCA77u, 0xC2B2AE3Du, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};
static_assert(sizeof(h2sha::kCkM) == 32, "checksum multipliers");

namespace {

thread_local std::string g_err;
int set_err(int code, const std::string& m) { g_err = m; return code; }
#define CUDA_TRY(x)                                                                                         \
  do {                                                                                                      \
    cudaError_t e_ = (x);                                                                                   \
    if (e_ != cudaSuccess) return set_err(H2SHA_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_));     \
  } while (0)

// ---------------------------------------------------------------------------------------------------
// device-side plan view
// ---------------------------------------------------------------------------------------------------
struct DevDigest {
  DigestPlace dp;
  uint32_t blk_prefix;    // blocks of digests < d in one instance
  uint32_t dtrace_off;    // word offset of this digest's trace inside the instance's digest-trace area
};

struct DevPlan {
  // one contiguous blob in global memory, copied to shared memory by every CTA at start
  const uint8_t* blob;
  uint32_t blob_bytes;
  // byte offsets inside the blob (all 16-byte aligned)
  uint32_t off_fill, off_cells, off_chunks, off_items, off_table_lo, off_table_hi, off_resident, off_prog, off_groups, off_tasks, off_types, off_classes,
      off_raw, off_breaks, off_digests, off_item_dict;
  uint32_t n_breaks, n_digests, n_block_parts, n_classes;
  // dynamic shared memory layout after the blob
  uint32_t off_trace, off_scratch, off_misc, smem_bytes;
  uint32_t stage_bytes, stage_off_slots, stage_off_desc;   // per producer warp: trace | slots | StageDesc
  uint32_t max_fill, scratch_bytes, n_resident;            // per consumer warp: lo[max_fill] | hi[max_fill]
  // layout
  int32_t spread_cols_shift;   // log2(spread_cols) when it is a power of two, else -1
  uint32_t max_rows, spread_cols, n_gate_cols, gate_col_rows, n_lookup_cols, lookup_col_rows, spread_rows;
  uint32_t blocks_per_inst, dtrace_words_per_inst;
  uint64_t gate_inst_cells, lookup_inst_cells, spread_inst_cells;
};

struct JobArgs {
  uint64_t n_inst;
  const uint32_t* btrace;   // word-major: [TR_BLOCK_WORDS][blocks_per_inst][n_inst]  (coalesced writes in k_trace)
  const uint32_t* dtrace;   // word-major: [dtrace_words_per_inst][n_inst]
  uint32_t* gate;           // Fr as 8 x u32
  uint32_t* lookup;
  uint32_t* spread;
  unsigned long long* cks;  // [n_inst][4] or null
  unsigned long long* job_counter;
  uint32_t only_digest;     // 0: all; d + 1: only the jobs of digest() call d
  // lookup multiplicities (MODE 1): the raw value of every looked-up cell and of every dense spread limb, written next to the
  // cells (13.5 KB + 2 KB per block instead of a second pass over 371 KB of Montgomery cells); k_mult_from_raw bins them
  uint32_t* lookup_raw;     // [n_inst][n_lookup_total] in cells_to_lookup order; 0xffffffff = a value that does not fit 32 bits
  uint8_t* dense_raw;       // [n_inst][n_limb_total]
  uint32_t limb_bits, n_lookup_total, n_limb_total;
  // compact hand-off: every DISTINCT value of an instance, once (null: not wanted)
  uint32_t* dict;           // [n_inst][dict_inst_cells] Fr as 8 x u32
  uint64_t dict_inst_cells;
};

__constant__ uint32_t c_K[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
    0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
    0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
    0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
    0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
    0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
__constant__ uint32_t c_H0[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
__constant__ uint32_t c_CKM[8] = {0x9E3779B1u, 0x85EBCA77u, 0xC2B2AE3Du, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};

#include "fr_dev.cuh"

// bit i -> bit 2i of the low 32 bits
__device__ __forceinline__ uint64_t spread32(uint64_t x) {
  x &= 0xffffffffULL;
  x = (x | (x << 16)) & 0x0000FFFF0000FFFFULL;
  x = (x | (x << 8)) & 0x00FF00FF00FF00FFULL;
  x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0FULL;
  x = (x | (x << 2)) & 0x3333333333333333ULL;
  x = (x | (x << 1)) & 0x5555555555555555ULL;
  return x;
}
// even-position bits of a 32-bit value, packed into 16 bits
__device__ __forceinline__ uint32_t even16(uint32_t x) {
  x &= 0x55555555u;
  x = (x | (x >> 1)) & 0x33333333u;
  x = (x | (x >> 2)) & 0x0F0F0F0Fu;
  x = (x | (x >> 4)) & 0x00FF00FFu;
  x = (x | (x >> 8)) & 0x0000FFFFu;
  return x;
}
__device__ __forceinline__ uint64_t extract(uint64_t s, uint32_t sh, uint32_t w) {
  uint64_t v = s >> sh;
  return (w >= 64) ? v : (v & ((1ULL << w) - 1ULL));
}

// ---------------------------------------------------------------------------------------------------
// k_trace
// ---------------------------------------------------------------------------------------------------
struct TraceArgs {
  uint64_t n_msgs;
  uint32_t n_digests;
  const uint8_t* msgs;
  const uint64_t* offsets;
  const uint32_t* lens;
  const uint32_t* pre_lens;   // may be null
  uint32_t* btrace;
  uint32_t* dtrace;
  uint8_t* digests;           // may be null
  const DevDigest* digests_plan;
  uint32_t blocks_per_inst, dtrace_words_per_inst;
  unsigned long long* job_counter;   // zeroed here for the expansion kernel that follows (saves two memset nodes)
  unsigned long long* cks;           // [n_inst][4] or null, zeroed here
};

__device__ __forceinline__ uint32_t rotr32(uint32_t x, int n) { return __funnelshift_r(x, x, n); }

// word `i` of 64-byte block `blk` of the padded message (lib.rs:98-117): message | 0x80 | zeros | 64-bit BE bit length |
// zeros up to max.  Branch-free predicated byte loads so that all loads of a block are in flight together.
__device__ __forceinline__ uint32_t padded_word(const uint8_t* msg, uint32_t len, uint32_t num_round, uint32_t blk, int i) {
  const uint32_t pos = 64 * blk + 4 * i;
  uint32_t x = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t p = pos + k;
    uint32_t byte = (p < len) ? (uint32_t)msg[p] : 0u;
    byte = (p == len) ? 0x80u : byte;
    x = (x << 8) | byte;
  }
  if (blk + 1 == num_round) {   // the bit length occupies the last two words of the last padded block
    const uint64_t bits = 8ull * len;
    if (i == 14) x = (uint32_t)(bits >> 32);
    if (i == 15) x = (uint32_t)bits;
  }
  return x;
}

__global__ void __launch_bounds__(64) k_trace(TraceArgs A) {
  // programmatic dependent launch: the expansion kernel may be scheduled now; it waits (griddepcontrol.wait) for this
  // grid to complete before it touches the traces, the job counter or the checksums
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  uint64_t m = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (m == 0 && A.job_counter) *A.job_counter = 0ull;
  if (m >= A.n_msgs) return;
  const uint32_t d = (uint32_t)(m % A.n_digests);
  const uint64_t inst = m / A.n_digests;
  if (d == 0 && A.cks) { A.cks[inst * 4 + 0] = 0; A.cks[inst * 4 + 1] = 0; A.cks[inst * 4 + 2] = 0; A.cks[inst * 4 + 3] = 0; }
  const DevDigest dd = A.digests_plan[d];
  const uint32_t R = dd.dp.n_blocks;
  const uint8_t* msg = A.msgs + A.offsets[m];
  const uint32_t len = A.lens[m];
  const uint32_t pre = A.pre_lens ? A.pre_lens[m] : 0u;
  const uint32_t num_round = (len + 9 + 63) / 64;          // lib.rs:80-84
  const uint32_t pre_round = pre / 64;                     // lib.rs:93
  uint32_t st[8];
#pragma unroll
  for (int i = 0; i < 8; i++) st[i] = c_H0[i];
  // word-major layouts: consecutive threads (instances) write consecutive addresses
  const uint64_t n_inst = A.n_msgs / A.n_digests;
  uint32_t* dt = A.dtrace + (uint64_t)dd.dtrace_off * n_inst + inst;            // word k at dt + k * n_inst
  uint32_t* bt = A.btrace + (uint64_t)dd.blk_prefix * n_inst + inst;            // word k of block j at bt[(k * bpi + j) * n_inst]
  const uint64_t bstride = (uint64_t)A.blocks_per_inst * n_inst;
  const uint32_t words_base = TD_STATES + 8 * (R + 1);
  uint32_t hfin[8];
#pragma unroll
  for (int i = 0; i < 8; i++) hfin[i] = 0;
  // blocks [0, pre_round): un-constrained prefix (sha2::compress256, lib.rs:153-160); blocks [pre_round, pre_round+R): traced
  for (uint32_t blk = 0; blk < pre_round + R; blk++) {
    const bool traced = blk >= pre_round;
    const uint32_t j = blk - pre_round;
    uint32_t* tw = bt + (uint64_t)j * n_inst;   // word k at tw + k * bstride
    if (traced) {
#pragma unroll
      for (int i = 0; i < 8; i++) dt[(uint64_t)(TD_STATES + 8 * j + i) * n_inst] = st[i];
    }
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const uint32_t x = padded_word(msg, len, num_round, blk, i);
      w[i] = x;
      if (traced) { tw[(uint64_t)(TR_W + i) * bstride] = x; dt[(uint64_t)(words_base + 16 * j + i) * n_inst] = x; }
    }
    uint32_t a = st[0], b = st[1], c = st[2], dd_ = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
    if (traced) {
      tw[(uint64_t)(TR_A + 3) * bstride] = a; tw[(uint64_t)(TR_A + 2) * bstride] = b; tw[(uint64_t)(TR_A + 1) * bstride] = c; tw[(uint64_t)(TR_A + 0) * bstride] = dd_;
      tw[(uint64_t)(TR_E + 3) * bstride] = e; tw[(uint64_t)(TR_E + 2) * bstride] = f; tw[(uint64_t)(TR_E + 1) * bstride] = g; tw[(uint64_t)(TR_E + 0) * bstride] = h;
    }
    for (int t0 = 0; t0 < 64; t0 += 16) {
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const int t = t0 + i;
        uint32_t wt;
        if (t0 == 0) {
          wt = w[i];
        } else {
          uint32_t w15 = w[(i + 1) & 15], w2 = w[(i + 14) & 15];
          uint32_t s0 = rotr32(w15, 7) ^ rotr32(w15, 18) ^ (w15 >> 3);
          uint32_t s1 = rotr32(w2, 17) ^ rotr32(w2, 19) ^ (w2 >> 10);
          wt = w[i] + s0 + w[(i + 9) & 15] + s1;
          w[i] = wt;
          if (traced) tw[(uint64_t)(TR_W + t) * bstride] = wt;
        }
        uint32_t t1 = h + (rotr32(e, 6) ^ rotr32(e, 11) ^ rotr32(e, 25)) + ((e & f) ^ (~e & g)) + c_K[t] + wt;
        uint32_t t2 = (rotr32(a, 2) ^ rotr32(a, 13) ^ rotr32(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
        h = g; g = f; f = e; e = dd_ + t1; dd_ = c; c = b; b = a; a = t1 + t2;
        if (traced) { tw[(uint64_t)(TR_A + 4 + t) * bstride] = a; tw[(uint64_t)(TR_E + 4 + t) * bstride] = e; }
      }
    }
    st[0] += a; st[1] += b; st[2] += c; st[3] += dd_; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
    if (blk + 1 == num_round) {
#pragma unroll
      for (int i = 0; i < 8; i++) hfin[i] = st[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; i++) dt[(uint64_t)(TD_STATES + 8 * R + i) * n_inst] = st[i];
  dt[(uint64_t)(TD_LEN) * n_inst] = len; dt[(uint64_t)(TD_NUM_ROUND) * n_inst] = num_round; dt[(uint64_t)(TD_PRE_ROUND) * n_inst] = pre_round; dt[(uint64_t)(TD_TARGET) * n_inst] = num_round - pre_round;
#pragma unroll
  for (int i = 0; i < 8; i++) dt[(uint64_t)(TD_H + i) * n_inst] = hfin[i];
  if (A.digests) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      uint32_t x = hfin[i];
      A.digests[m * 32 + 4 * i + 0] = (uint8_t)(x >> 24); A.digests[m * 32 + 4 * i + 1] = (uint8_t)(x >> 16);
      A.digests[m * 32 + 4 * i + 2] = (uint8_t)(x >> 8);  A.digests[m * 32 + 4 * i + 3] = (uint8_t)x;
    }
  }
}

// Small batches (latency, not throughput: BASELINE config 1 is ONE message): one warp per message.  The chain of compressions
// cannot be shortened, so everything around it is taken off the thread that walks it: all lanes build the padded words
// (coalesced byte reads) into shared memory, lane = block expands the message schedules of up to 32 blocks at once, lane 0 then
// runs only the 64 rounds per block (schedule word + round constant from shared memory, working variables into shared memory),
// and all lanes write the traces out.  Same outputs as k_trace, bit for bit (tests/test_gpu_boundary.py compares the two).
enum { TW_PASS = 32, TW_WSTRIDE = 65 };   // blocks per pass; schedule stride in words (odd: lanes = blocks hit different banks)
__global__ void __launch_bounds__(32) k_trace_warp(TraceArgs A) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __shared__ uint32_t sW[TW_PASS * TW_WSTRIDE];   // schedule W[64] per block
  __shared__ uint32_t sA[TW_PASS * 68], sE[TW_PASS * 68];   // working variables a / e: [0..3] = input state (d,c,b,a / h,g,f,e), [4 + t] after round t
  __shared__ uint32_t sS[(TW_PASS + 1) * 8];      // chaining state before every block of the pass (+ after the last one)
  const int lane = threadIdx.x;
  const uint64_t m = blockIdx.x;
  if (m == 0 && lane == 0 && A.job_counter) *A.job_counter = 0ull;
  if (m >= A.n_msgs) return;
  const uint32_t d = (uint32_t)(m % A.n_digests);
  const uint64_t inst = m / A.n_digests;
  if (d == 0 && A.cks && lane < 4) A.cks[inst * 4 + lane] = 0;
  const DevDigest dd = A.digests_plan[d];
  const uint32_t R = dd.dp.n_blocks;
  const uint8_t* msg = A.msgs + A.offsets[m];
  const uint32_t len = A.lens[m];
  const uint32_t pre = A.pre_lens ? A.pre_lens[m] : 0u;
  const uint32_t num_round = (len + 9 + 63) / 64;          // lib.rs:80-84
  const uint32_t pre_round = pre / 64;                     // lib.rs:93
  const uint64_t n_inst = A.n_msgs / A.n_digests;
  uint32_t* dt = A.dtrace + (uint64_t)dd.dtrace_off * n_inst + inst;
  uint32_t* bt = A.btrace + (uint64_t)dd.blk_prefix * n_inst + inst;
  const uint64_t bstride = (uint64_t)A.blocks_per_inst * n_inst;
  const uint32_t words_base = TD_STATES + 8 * (R + 1);
  const uint32_t total = pre_round + R;
  uint32_t st[8], hfin[8];
#pragma unroll
  for (int i = 0; i < 8; i++) { st[i] = c_H0[i]; hfin[i] = 0; }
  for (uint32_t b0 = 0; b0 < total; b0 += TW_PASS) {
    const uint32_t nb = min((uint32_t)TW_PASS, total - b0);
    // (1) padded message words of the pass (lib.rs:98-117)
    for (uint32_t idx = lane; idx < nb * 16; idx += 32) sW[(idx >> 4) * TW_WSTRIDE + (idx & 15)] = padded_word(msg, len, num_round, b0 + (idx >> 4), (int)(idx & 15));
    __syncwarp();
    // (2) message schedules, lane = block (compression.rs:57-96 computes the same words in-circuit)
    if ((uint32_t)lane < nb) {
      uint32_t* w = sW + lane * TW_WSTRIDE;
      for (int t = 16; t < 64; t++) {
        const uint32_t w15 = w[t - 15], w2 = w[t - 2];
        const uint32_t s0 = rotr32(w15, 7) ^ rotr32(w15, 18) ^ (w15 >> 3);
        const uint32_t s1 = rotr32(w2, 17) ^ rotr32(w2, 19) ^ (w2 >> 10);
        w[t] = w[t - 16] + s0 + w[t - 7] + s1;
      }
    }
    __syncwarp();
    // (3) the chain: one lane, rounds only
    if (lane == 0) {
      for (uint32_t lb = 0; lb < nb; lb++) {
        const uint32_t* w = sW + lb * TW_WSTRIDE;
        uint32_t* pa = sA + lb * 68;
        uint32_t* pe = sE + lb * 68;
#pragma unroll
        for (int i = 0; i < 8; i++) sS[lb * 8 + i] = st[i];
        uint32_t a = st[0], b = st[1], c = st[2], dd_ = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
        pa[3] = a; pa[2] = b; pa[1] = c; pa[0] = dd_; pe[3] = e; pe[2] = f; pe[1] = g; pe[0] = h;
#pragma unroll 8
        for (int t = 0; t < 64; t++) {
          const uint32_t t1 = h + (rotr32(e, 6) ^ rotr32(e, 11) ^ rotr32(e, 25)) + ((e & f) ^ (~e & g)) + c_K[t] + w[t];
          const uint32_t t2 = (rotr32(a, 2) ^ rotr32(a, 13) ^ rotr32(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
          h = g; g = f; f = e; e = dd_ + t1; dd_ = c; c = b; b = a; a = t1 + t2;
          pa[4 + t] = a; pe[4 + t] = e;
        }
        st[0] += a; st[1] += b; st[2] += c; st[3] += dd_; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
        if (b0 + lb + 1 == num_round) {
#pragma unroll
          for (int i = 0; i < 8; i++) hfin[i] = st[i];
        }
      }
#pragma unroll
      for (int i = 0; i < 8; i++) sS[nb * 8 + i] = st[i];
    }
    __syncwarp();
    // (4) traces of the constrained blocks of the pass (blocks below pre_round are the unconstrained prefix, lib.rs:153-160)
    for (uint32_t lb = 0; lb < nb; lb++) {
      const uint32_t blk = b0 + lb;
      if (blk < pre_round) continue;
      const uint32_t j = blk - pre_round;
      uint32_t* tw = bt + (uint64_t)j * n_inst;   // word k at tw + k * bstride
      for (uint32_t k = lane; k < TR_BLOCK_WORDS; k += 32) {
        const uint32_t v = k < TR_A ? sW[lb * TW_WSTRIDE + k] : (k < TR_E ? sA[lb * 68 + (k - TR_A)] : sE[lb * 68 + (k - TR_E)]);
        tw[(uint64_t)k * bstride] = v;
      }
      if (lane < 8) dt[(uint64_t)(TD_STATES + 8 * j + lane) * n_inst] = sS[lb * 8 + lane];
      else if (lane < 24) dt[(uint64_t)(words_base + 16 * j + (lane - 8)) * n_inst] = sW[lb * TW_WSTRIDE + (lane - 8)];
    }
    if (b0 + nb == total && lane < 8) dt[(uint64_t)(TD_STATES + 8 * R + lane) * n_inst] = sS[nb * 8 + lane];
    __syncwarp();
  }
  if (lane == 0) {
    dt[(uint64_t)(TD_LEN) * n_inst] = len; dt[(uint64_t)(TD_NUM_ROUND) * n_inst] = num_round; dt[(uint64_t)(TD_PRE_ROUND) * n_inst] = pre_round;
    dt[(uint64_t)(TD_TARGET) * n_inst] = num_round - pre_round;
#pragma unroll
    for (int i = 0; i < 8; i++) dt[(uint64_t)(TD_H + i) * n_inst] = hfin[i];
    if (A.digests) {
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const uint32_t x = hfin[i];
        A.digests[m * 32 + 4 * i + 0] = (uint8_t)(x >> 24); A.digests[m * 32 + 4 * i + 1] = (uint8_t)(x >> 16);
        A.digests[m * 32 + 4 * i + 2] = (uint8_t)(x >> 8);  A.digests[m * 32 + 4 * i + 3] = (uint8_t)x;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// k_expand
// ---------------------------------------------------------------------------------------------------
// per-consumer-warp scratch of phase 2: Montgomery values of the chunk's distinct non-constant cells (low / high
// 16 bytes in separate arrays so that random 128-bit reads spread over all bank groups) + their checksum hashes
struct WarpScratch {   // runtime-sized: lo[max_fill] | hi[max_fill] (| raw[max_fill] in MODE 1); slots [0, n_resident) hold the resident constants
  uint4* lo;
  uint4* hi;
  uint32_t* raw;         // MODE 1: raw value of the looked-up distinct values of the chunk
};
// job descriptor a producer warp leaves in its stage
struct StageDesc {
  unsigned long long inst;      // first circuit instance of the job
  uint32_t cls, gate0, lk0, limb0;
  uint32_t valid;               // 0: the producer has run out of jobs
  uint32_t n_inst;              // circuit instances the job covers (digest jobs are batched)
  uint32_t dict0;               // dictionary index of the job's first distinct value inside its instance (compact hand-off)
};

// ---- mbarrier helpers (shared::cta) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// the producers' wait: polls with a 256 ns __nanosleep back-off between tries (longer sleeps, suspend-time hints and a
// back-off for the consumers' wait measured no better in time or power: DESIGN.md section 10)
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  for (;;) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(256);
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

__device__ __forceinline__ uint64_t vm_operand(uint32_t o, const uint64_t* slots, const uint64_t* raw) {
  if (o & 1u) return raw[o >> 1];
  return extract(slots[(o >> 1) & 0xfffu], (o >> 13) & 63u, (o >> 19) & 127u);
}

// phase 1: run the slot program of group `g` for unit instance `u` (one lane); `trace` is the trace of the circuit
// instance the unit belongs to and `uu` the unit's index inside that instance
__device__ __forceinline__ void run_unit_program(const UnitGroup& g, const UnitType& ut, uint32_t uu, const VmIns* prog, const uint64_t* raw,
                                                 const uint32_t* trace, uint64_t* slots) {
  for (uint32_t k = 0; k < ut.n_in; k++) {
    int32_t base = g.in[k].base;
    slots[k] = (base < 0) ? (uint64_t)(g.in[k].stride + (int32_t)uu) : (uint64_t)trace[base + g.in[k].stride * (int32_t)uu];
  }
  // (Round 2: fetching the next instruction word early and reading all three operands before the opcode dispatch changed neither the
  // 11.5 us a 49-instruction program takes nor the sustained launch time -- the chain through the result slots dominates.)
  const VmIns* ins = prog + ut.prog_off;
  for (uint32_t pc = 0; pc < ut.prog_len; pc++) {
    const VmIns I = ins[pc];
    const uint32_t op = I.op_dst & 0xffu, dst = (I.op_dst >> 8) & 0xffu;
    uint64_t a = vm_operand(I.a, slots, raw);
    uint64_t r;
    switch (op) {
      case OP_ADD: r = a + vm_operand(I.b, slots, raw); break;
      case OP_SUB: r = a - vm_operand(I.b, slots, raw); break;
      case OP_MULADD: r = a * vm_operand(I.b, slots, raw) + vm_operand(I.c, slots, raw); break;
      case OP_SPREAD: r = spread32(a); break;
      case OP_COMPRESS2: {
        uint32_t x = (uint32_t)a, y = (uint32_t)vm_operand(I.b, slots, raw);
        r = (uint64_t)even16(x) | ((uint64_t)even16(y) << 16) | ((uint64_t)even16(x >> 1) << 32) | ((uint64_t)even16(y >> 1) << 48);
        break;
      }
      case OP_EQ: r = (a == vm_operand(I.b, slots, raw)) ? 1 : 0; break;
      case OP_GT: r = (a > vm_operand(I.b, slots, raw)) ? 1 : 0; break;
      case OP_SEL: r = a ? vm_operand(I.b, slots, raw) : vm_operand(I.c, slots, raw); break;
      default: r = a; break;  // OP_MOV
    }
    slots[dst] = r;
  }
}

// one 256-bit store per Fr cell (STG.E.256, sm_100+); p must be 32-byte aligned
__device__ __forceinline__ void store_cell2(uint32_t* p, const uint4& lo, const uint4& hi) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w), "r"(hi.x),
               "r"(hi.y), "r"(hi.z), "r"(hi.w)
               : "memory");
}

// fill phase: the chunk's distinct values -> warp scratch.  Each function returns the checksum hash of the value.
__device__ __forceinline__ uint32_t hash8(const uint4& lo, const uint4& hi) {
  return lo.x * c_CKM[0] + lo.y * c_CKM[1] + lo.z * c_CKM[2] + lo.w * c_CKM[3] + hi.x * c_CKM[4] + hi.y * c_CKM[5] + hi.z * c_CKM[6] +
         hi.w * c_CKM[7];
}
// value of a table-copy entry (constants, 8-bit limbs, spread limbs, inverses): static Montgomery table[tbl + extract]
__device__ __forceinline__ void value_table(const FillEntry& e, const uint64_t* slots, const uint4* table_lo, const uint4* table_hi, uint32_t* raw,
                                            uint4* lo, uint4* hi) {
  const uint64_t s = slots[H2SHA_TE_SLOT(e)];
  *raw = (uint32_t)extract(s, H2SHA_TE_SH(e), H2SHA_TE_W(e));
  const uint32_t idx = H2SHA_TE_TBL(e) + *raw;
  *lo = table_lo[idx]; *hi = table_hi[idx];
}
// value of a Barrett entry: the 32-bit path when every lane of the warp iteration holds a value < 2^32, else the 64-bit path
__device__ __forceinline__ void value_generic(const FillEntry& e, const uint64_t* slots, bool active, uint64_t* raw, uint4* lo, uint4* hi) {
  bool neg = false;
  uint64_t v = 0;
  if (active) {
    const uint64_t s = slots[H2SHA_TE_SLOT(e)];
    neg = H2SHA_TE_NEG(e);
    if (H2SHA_TE_KIND(e) == KIND_SIGNED) {
      int64_t sv = (int64_t)s;
      neg = sv < 0;
      v = neg ? (uint64_t)(-sv) : (uint64_t)sv;
    } else {
      v = extract(s, H2SHA_TE_SH(e), H2SHA_TE_W(e)) << H2SHA_TE_SHL(e);
    }
  }
  *raw = v;
  uint32_t x[8];
  if (__any_sync(0xffffffffu, (v >> 32) != 0)) {
    uint64_t r[4];
    mont_from_u64(v, r);
    if (neg) fr_negate(r);
    x[0] = (uint32_t)r[0]; x[1] = (uint32_t)(r[0] >> 32); x[2] = (uint32_t)r[1]; x[3] = (uint32_t)(r[1] >> 32);
    x[4] = (uint32_t)r[2]; x[5] = (uint32_t)(r[2] >> 32); x[6] = (uint32_t)r[3]; x[7] = (uint32_t)(r[3] >> 32);
  } else {
    mont_from_u32((uint32_t)v, x);
    if (neg) fr_negate32(x);
  }
  *lo = make_uint4(x[0], x[1], x[2], x[3]); *hi = make_uint4(x[4], x[5], x[6], x[7]);
}
__device__ __forceinline__ uint32_t fill_table(const FillEntry& e, const uint64_t* slots, const uint4* table_lo, const uint4* table_hi,
                                               const WarpScratch& ws, uint32_t* raw, uint32_t* dict_out) {
  const uint32_t i = H2SHA_TE_DST(e);
  uint4 lo, hi;
  value_table(e, slots, table_lo, table_hi, raw, &lo, &hi);
  ws.lo[i] = lo; ws.hi[i] = hi;
  if (dict_out) store_cell2(dict_out, lo, hi);
  return hash8(lo, hi);
}
__device__ __forceinline__ uint32_t fill_generic(const FillEntry& e, const uint64_t* slots, const WarpScratch& ws, bool active, uint64_t* raw, uint32_t* dict_out) {
  const uint32_t i = H2SHA_TE_DST(e);
  uint4 lo, hi;
  value_generic(e, slots, active, raw, &lo, &hi);
  if (active) {
    ws.lo[i] = lo; ws.hi[i] = hi;
    if (dict_out) store_cell2(dict_out, lo, hi);
  }
  return hash8(lo, hi);
}

// the copy loops' read of a cell's value from the warp scratch
#define H2SHA_SCRATCH_READ(src) const uint4 lo = ws.lo[src], hi = ws.hi[src];
// warp-reduce the three checksum accumulators and add them to the instance's totals (gate, lookup, spread, all)
__device__ __forceinline__ void flush_checksums(unsigned long long* cks, uint64_t inst, unsigned long long ck_g, unsigned long long ck_l,
                                                unsigned long long ck_s, int lane) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ck_g += __shfl_xor_sync(0xffffffffu, ck_g, o);
    ck_l += __shfl_xor_sync(0xffffffffu, ck_l, o);
    ck_s += __shfl_xor_sync(0xffffffffu, ck_s, o);
  }
  if (lane == 0) {
    if (ck_g) atomicAdd(&cks[inst * 4 + 0], ck_g);
    if (ck_l) atomicAdd(&cks[inst * 4 + 1], ck_l);
    if (ck_s) atomicAdd(&cks[inst * 4 + 2], ck_s);
    atomicAdd(&cks[inst * 4 + 3], ck_g + ck_l + ck_s);
  }
}

// MODE 0: cells (+ checksums); 1: also write the raw values of the looked-up cells (A.lookup_raw / A.dense_raw: the input of the
// multiplicity kernel); 2: also write the dictionary of distinct values
// (A.dict).  Separate instantiations: the extra code costs registers the plain path (80 per thread at 768 threads) does not have.
template <int NCONS, int NPROD, int MODE>
__global__ void __launch_bounds__((NCONS + NPROD) * 32, 1) k_expand(const DevPlan P, const JobArgs A) {
  constexpr bool MULT = MODE == 1, DICT = MODE == 2;
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int NT = (NCONS + NPROD) * 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // ---- static plan -> shared memory (once per persistent CTA) ----
  {
    const uint4* src = reinterpret_cast<const uint4*>(P.blob);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (uint32_t i = tid; i < P.blob_bytes / 16; i += NT) dst[i] = src[i];
  }
  const FillEntry* s_fill = reinterpret_cast<const FillEntry*>(smem + P.off_fill);
  const CellEntry* s_cells = reinterpret_cast<const CellEntry*>(smem + P.off_cells);
  const Chunk* s_chunks = reinterpret_cast<const Chunk*>(smem + P.off_chunks);
  const ItemDesc* s_items = reinterpret_cast<const ItemDesc*>(smem + P.off_items);
  const uint4* s_table_lo = reinterpret_cast<const uint4*>(smem + P.off_table_lo);
  const uint4* s_table_hi = reinterpret_cast<const uint4*>(smem + P.off_table_hi);
  const uint32_t* s_resident = reinterpret_cast<const uint32_t*>(smem + P.off_resident);
  const VmIns* s_prog = reinterpret_cast<const VmIns*>(smem + P.off_prog);
  const UnitGroup* s_groups = reinterpret_cast<const UnitGroup*>(smem + P.off_groups);
  const WarpTask* s_tasks = reinterpret_cast<const WarpTask*>(smem + P.off_tasks);
  const UnitType* s_types = reinterpret_cast<const UnitType*>(smem + P.off_types);
  const JobClass* s_classes = reinterpret_cast<const JobClass*>(smem + P.off_classes);
  const uint64_t* s_raw = reinterpret_cast<const uint64_t*>(smem + P.off_raw);
  const uint32_t* s_breaks = reinterpret_cast<const uint32_t*>(smem + P.off_breaks);
  const DevDigest* s_digests = reinterpret_cast<const DevDigest*>(smem + P.off_digests);
  [[maybe_unused]] const uint32_t* s_item_dict = reinterpret_cast<const uint32_t*>(smem + P.off_item_dict);
  uint64_t* s_full = reinterpret_cast<uint64_t*>(smem + P.off_misc);   // [NPROD]
  uint64_t* s_empty = s_full + NPROD;                                  // [NPROD]
  if (tid == 0) {
    for (int i = 0; i < NPROD; i++) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], NCONS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();  // blob + barriers visible; the only CTA-wide barrier
#ifdef H2SHA_DEBUG_TIMING
  unsigned long long dbg_t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t1));
#endif
  // everything above is independent of the trace kernel; from here on its outputs are read
  asm volatile("griddepcontrol.wait;" ::: "memory");
#ifdef H2SHA_DEBUG_TIMING
  unsigned long long dbg_t2; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t2));
#endif

  // jobs: all block-job parts first, then per digest the batched prologue/epilogue jobs
  const uint64_t n_block_jobs = A.n_inst * P.blocks_per_inst * P.n_block_parts;
  uint64_t n_jobs = n_block_jobs;
  for (uint32_t c = P.n_block_parts; c < P.n_classes; c++) {
    const uint32_t batch = s_classes[c].batch;
    n_jobs += (A.n_inst + batch - 1) / batch;
  }

  if (warp >= NCONS) {
    // =========================== producer warp: owns stage `st` ===========================
    const int st = warp - NCONS;
    uint8_t* stage = smem + P.off_trace + (size_t)st * P.stage_bytes;
    uint32_t* s_trace = reinterpret_cast<uint32_t*>(stage);
    uint64_t* s_slots = reinterpret_cast<uint64_t*>(stage + P.stage_off_slots);
    StageDesc* desc = reinterpret_cast<StageDesc*>(stage + P.stage_off_desc);
    for (int i = lane; i < 64; i += 32) s_trace[TR_K + i] = c_K[i];
    for (uint32_t k = 0;; k++) {
      mbar_wait_relaxed(&s_empty[st], (k & 1u) ^ 1u);   // consumers are done with this stage's previous job
#ifdef H2SHA_DEBUG_TIMING
      unsigned long long dbg_p0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_p0));
#endif
      // the first job of every producer is assigned statically (job = producer * grid + CTA), the later ones come from the global
      // counter: with fewer jobs than producers (a single digest: latency, not throughput) every CTA gets at most one job instead
      // of the quickest CTA grabbing four
      unsigned long long job = 0;
      bool static_job = (k == 0);
    next_job:
      if (static_job) {
        job = (unsigned long long)st * gridDim.x + blockIdx.x;
        static_job = false;
      } else {
        if (lane == 0) job = (unsigned long long)gridDim.x * NPROD + atomicAdd(A.job_counter, 1ULL);
        job = __shfl_sync(0xffffffffu, job, 0);
      }
#ifdef H2SHA_DEBUG_TIMING
      unsigned long long dbg_p1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_p1));
#endif
      if (job >= n_jobs) {
        if (lane == 0) { desc->valid = 0; }
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_full[st]);
        break;
      }
      // ---- decode job ----
      uint64_t inst; uint32_t cls, gate0, lk0, limb0, n_valid = 1, tr_words, dict0;
      if (job < n_block_jobs) {
        const uint64_t blk = job / P.n_block_parts;          // global block index = inst * blocks_per_inst + r
        cls = (uint32_t)(job - blk * P.n_block_parts);        // part of the block job
        inst = blk / P.blocks_per_inst;
        uint32_t r = (uint32_t)(blk - inst * P.blocks_per_inst);
        uint32_t d = 0;
        while (d + 1 < P.n_digests && r >= s_digests[d + 1].blk_prefix) d++;
        if (A.only_digest && d + 1 != A.only_digest) goto next_job;
        const DevDigest& dd = s_digests[d];
        uint32_t jb = r - dd.blk_prefix;
        gate0 = dd.dp.blk_gate_base + jb * dd.dp.blk_gate_stride;
        lk0 = dd.dp.blk_lk_base + jb * dd.dp.blk_lk_stride;
        limb0 = dd.dp.blk_limb_base + jb * dd.dp.blk_limb_stride;
        dict0 = dd.dp.dict_base + dd.dp.dict_dig_len + jb * dd.dp.dict_blk_len;
        const uint32_t* tr_src = A.btrace + (uint64_t)r * A.n_inst + inst;
        const uint64_t tr_stride = (uint64_t)P.blocks_per_inst * A.n_inst;
        tr_words = TR_BLOCK_WORDS;
        for (uint32_t i = lane; i < tr_words; i += 32) s_trace[i] = tr_src[(uint64_t)i * tr_stride];
      } else {
        // digest-job classes follow the block-job parts, digest by digest (a long digest owns several consecutive classes)
        uint64_t kk = job - n_block_jobs;
        cls = P.n_block_parts;
        uint32_t batch = s_classes[cls].batch;
        for (;;) {
          const uint64_t nb = (A.n_inst + batch - 1) / batch;
          if (kk < nb) break;
          kk -= nb; cls++;
          batch = s_classes[cls].batch;
        }
        if (A.only_digest && s_classes[cls].digest + 1 != A.only_digest) goto next_job;
        const DevDigest& dd = s_digests[s_classes[cls].digest];
        inst = kk * batch;
        n_valid = (uint32_t)min((uint64_t)batch, A.n_inst - inst);
        gate0 = 0; lk0 = 0; limb0 = 0;
        dict0 = dd.dp.dict_base;
        tr_words = dd.dp.trace_words;
        // word-major global layout: consecutive instances are adjacent, so lanes run over the instances of the batch
        const uint32_t* tr_src = A.dtrace + (uint64_t)dd.dtrace_off * A.n_inst + inst;
        for (uint32_t idx = lane; idx < tr_words * n_valid; idx += 32) {
          const uint32_t k2 = idx / n_valid, i2 = idx - k2 * n_valid;
          s_trace[i2 * tr_words + k2] = tr_src[(uint64_t)k2 * A.n_inst + i2];
        }
      }
      const JobClass jc = s_classes[cls];
      if (lane == 0) { desc->inst = inst; desc->cls = cls; desc->gate0 = gate0; desc->lk0 = lk0; desc->limb0 = limb0; desc->valid = 1; desc->n_inst = n_valid; desc->dict0 = dict0; }
      __syncwarp();
#ifdef H2SHA_DEBUG_TIMING
      unsigned long long dbg_p2; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_p2));
#endif
      // ---- phase 1: slot programs, lanes = unit instances ----
      for (uint32_t t = 0; t < jc.n_tasks; t++) {
        const WarpTask wt = s_tasks[jc.task_off + t];
        const UnitGroup& g = s_groups[jc.group_off + wt.group];
        const UnitType& ut = s_types[g.type];
        const uint32_t u = wt.first + lane;
        const uint32_t ii = u / g.per_inst, uu = u - ii * g.per_inst;   // circuit instance inside the job, unit inside the instance
        if (u < g.count && ii < n_valid)
          run_unit_program(g, ut, uu, s_prog, s_raw, s_trace + ii * tr_words, s_slots + g.slot_base + u * (ut.n_slots | 1u));
      }
      if (tr_words * n_valid > TR_K) {  // a digest trace overwrote the round constants kept at TR_K for block jobs: restore them
        __syncwarp();
        for (int i = lane; i < 64; i += 32) s_trace[TR_K + i] = c_K[i];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_full[st]);
#ifdef H2SHA_DEBUG_TIMING
      if (H2SHA_DEBUG_TIMING == 1 && lane == 0 && k < 3 && (blockIdx.x % 37) == 0) {
        unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        printf("P cta %3d prod %d job# %u cls %u: wait_trace %llu | empty-wait done +%llu, job fetched +%llu, trace loaded +%llu, full +%llu ns\n", blockIdx.x, st, k, cls,
               dbg_t2 - dbg_t1, dbg_p0 - dbg_t2, dbg_p1 - dbg_t2, dbg_p2 - dbg_t2, t - dbg_t2);
      }
#endif
    }
    return;
  }

  // =========================== consumer warp ===========================
  WarpScratch ws;
  {
    uint8_t* base = smem + P.off_scratch + (size_t)warp * P.scratch_bytes;
    ws.lo = reinterpret_cast<uint4*>(base);
    ws.hi = ws.lo + P.max_fill;
    ws.raw = reinterpret_cast<uint32_t*>(ws.hi + P.max_fill);   // only inside the scratch of a MODE 1 launch (larger scratch_bytes)
    for (uint32_t i = lane; i < P.n_resident; i += 32) { ws.lo[i] = s_table_lo[s_resident[i]]; ws.hi[i] = s_table_hi[s_resident[i]]; }
    __syncwarp();
  }
  uint32_t finished = 0;   // bit st: producer st has run out of jobs
#ifdef H2SHA_DEBUG_TIMING
  unsigned long long dbg_wait = 0; uint32_t dbg_nwait = 0;
#endif
  for (uint32_t k = 0; finished != (1u << NPROD) - 1u; k++) {
    const int st = k % NPROD;
    const uint32_t round = k / NPROD;
    if (finished & (1u << st)) continue;
#ifdef H2SHA_DEBUG_TIMING
    unsigned long long dbg_w0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_w0));
#endif
    mbar_wait(&s_full[st], round & 1u);
#ifdef H2SHA_DEBUG_TIMING
    {
      unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      dbg_wait += t - dbg_w0; dbg_nwait++;
      if (H2SHA_DEBUG_TIMING == 1 && lane == 0 && (blockIdx.x % 37) == 0 && (warp % 7) == 0 && (k < 6 || t - dbg_w0 > 3000))
        printf("C cta %3d warp %2d k %3u: waited %llu ns at +%llu ns\n", blockIdx.x, warp, k, t - dbg_w0, t - dbg_t2);
    }
#endif
    const uint8_t* stage = smem + P.off_trace + (size_t)st * P.stage_bytes;
    const uint64_t* s_slots = reinterpret_cast<const uint64_t*>(stage + P.stage_off_slots);
    const StageDesc* desc = reinterpret_cast<const StageDesc*>(stage + P.stage_off_desc);
    if (!desc->valid) { finished |= 1u << st; continue; }   // this producer has run out of jobs and exited
    const uint64_t inst0 = desc->inst;
    const uint32_t gate0 = desc->gate0, lk0 = desc->lk0, limb0 = desc->limb0, n_valid = desc->n_inst;
    const JobClass jc = s_classes[desc->cls];
    unsigned long long ck_g = 0, ck_l = 0, ck_s = 0;
    // static item -> warp assignment, rotated per job so that the heavier leading items do not always hit the same warps
    for (uint32_t it = (uint32_t)(warp + k) % NCONS; it < jc.n_items; it += NCONS) {
      const ItemDesc item = s_items[jc.item_off + it];
      const uint32_t inst_off = H2SHA_ITEM_INST(item.slot_chunk);
      if (inst_off >= n_valid) continue;   // partial last batch of digest jobs (warp-uniform)
      const uint64_t inst = inst0 + inst_off;
      uint32_t* gate_out = A.gate ? A.gate + inst * P.gate_inst_cells * 8 : nullptr;
      uint32_t* lk_out = A.lookup ? A.lookup + inst * P.lookup_inst_cells * 8 : nullptr;
      uint32_t* sp_out = A.spread ? A.spread + inst * P.spread_inst_cells * 8 : nullptr;
      const Chunk ch = s_chunks[H2SHA_ITEM_CHUNK(item.slot_chunk)];
      const uint64_t* slots = s_slots + H2SHA_ITEM_SLOT(item.slot_chunk);
      // ---- positions of the chunk's gate cells; a column break inside the chunk (rare) takes the per-cell path ----
      const uint32_t g_lo = gate0 + item.gate_rel;   // instance-relative gate-stream index of the unit's first cell
      uint32_t c0 = 0;
      if (P.n_breaks > 1) {
        // a column holds at most max_rows cells, so column c starts at or before c * max_rows: start the search at the quotient
        // (a linear search from column 0 cost ~0.7 % of the launch per gate column: config 5 has 18)
        c0 = min((g_lo + ch.gate_dst_min) / P.max_rows, P.n_breaks - 1u);
        while (c0 + 1 < P.n_breaks && s_breaks[c0 + 1] <= g_lo + ch.gate_dst_min) c0++;
      }
      const uint32_t next_brk = (c0 + 1 < P.n_breaks) ? s_breaks[c0 + 1] : 0xffffffffu;
      const uint32_t off0 = c0 * P.gate_col_rows - s_breaks[c0];          // pos = gidx + off0 before the break,
      const uint32_t off1 = (c0 + 1) * P.gate_col_rows - next_brk;        //       gidx + off1 from the break on
      const bool straddle = g_lo + ch.gate_dst_max >= next_brk;
      // checksum weight of a value carried by cnt cells whose offsets sum to sumdst: sum (2*pos+1) = cnt*w0 + 2*sumdst
      const unsigned long long w0 = straddle ? 0ull : (unsigned long long)(2u * (g_lo + off0) + 1u);
      const unsigned long long w1 = straddle ? 0ull : 2ull;
      // ---- compact hand-off: the chunk's distinct values also go to the instance's dictionary, fill entry i -> entry dict_chunk + i ----
      [[maybe_unused]] uint32_t* dict_chunk = nullptr;
      if constexpr (DICT) dict_chunk = A.dict + (inst * A.dict_inst_cells + desc->dict0 + s_item_dict[jc.item_off + it]) * 8;
      // ---- fill: table copies, then Barrett conversions ----
      {
        const FillEntry* fl = s_fill + ch.fill_off;
        const uint32_t n_tab = ch.n_fill_table, n_all = ch.n_fill;
        for (uint32_t i = lane; i < n_tab; i += 32) {
          const FillEntry e = fl[i];
          uint32_t raw;
          const uint32_t h = fill_table(e, slots, s_table_lo, s_table_hi, ws, &raw, DICT ? dict_chunk + (uint64_t)i * 8 : nullptr);
          ck_g += (unsigned long long)h * (H2SHA_FE_GATE_CNT(e) * w0 + e.sumdst * w1);
          if constexpr (MULT) { if (H2SHA_FE_LK_CNT(e)) ws.raw[H2SHA_TE_DST(e)] = raw; }
        }
        for (uint32_t i0 = n_tab; i0 < n_all; i0 += 32) {
          const uint32_t i = i0 + lane;
          const bool active = i < n_all;
          FillEntry e = fl[active ? i : n_tab];
          uint64_t raw;
          const uint32_t h = fill_generic(e, slots, ws, active, &raw, DICT ? dict_chunk + (uint64_t)i * 8 : nullptr);
          if (active) {
            ck_g += (unsigned long long)h * (H2SHA_FE_GATE_CNT(e) * w0 + e.sumdst * w1);
            if constexpr (MULT) { if (H2SHA_FE_LK_CNT(e)) ws.raw[H2SHA_TE_DST(e)] = (raw >> 32) ? 0xffffffffu : (uint32_t)raw; }
          }
        }
        if (lane == 0 && !straddle) ck_g += ch.res_a + ch.res_b * w0;
      }
      __syncwarp();
      // ---- copy: gate cells ----
      if (ch.gate_len && (gate_out || (straddle && A.cks))) {   // nothing to do when only the dictionary / checksums of a non-straddling chunk are wanted
        const CellEntry* cells = s_cells + ch.gate_off;
        if (!straddle) {
          // warp stores are aligned to 256-byte groups of the output: iteration k covers the 32 cells starting at
          // (pos0 - shift) + 32 k, shift = pos0 mod 8 cells, so only the first iteration has idle lanes and the
          // quarter-warp grouping is the one the planner coloured the scratch slots for
          const uint32_t pos0 = g_lo + off0 + ch.gate_dst_min;          // position of cells[0]
          const int shift = (int)(pos0 & 7u);
          uint32_t* out0 = gate_out + (uint64_t)(g_lo + off0) * 8;
          const int n = (int)ch.gate_len;
#pragma unroll 4
          for (int i = (int)lane - shift; i < n; i += 32) {
            if (i >= 0) {
              const CellEntry ce = cells[i];
              const uint32_t src = H2SHA_CE_SRC(ce);
              H2SHA_SCRATCH_READ(src)
              if (gate_out) store_cell2(out0 + (uint64_t)H2SHA_CE_DST(ce) * 8, lo, hi);
            }
          }
        } else {
          for (uint32_t i = lane; i < ch.gate_len; i += 32) {
            const CellEntry ce = cells[i];
            const uint32_t src = H2SHA_CE_SRC(ce);
            H2SHA_SCRATCH_READ(src)
            const uint32_t gidx = g_lo + H2SHA_CE_DST(ce);
            const uint32_t pos = gidx + ((gidx >= next_brk) ? off1 : off0);
            if (gate_out) store_cell2(gate_out + (uint64_t)pos * 8, lo, hi);
            ck_g += (unsigned long long)hash8(lo, hi) * (unsigned long long)(2u * pos + 1u);
          }
        }
      }
      // ---- lookup-column cells (range.finalize copies cells_to_lookup in push order, wrapping at max_rows) ----
      if (ch.lk_len && (lk_out || A.cks)) {
        const uint32_t l_lo = lk0 + item.lk_rel;
        // pos = li + loff0 before the column wrap at `wrap`, li + loff1 after it (no division in the loop)
        uint32_t loff0 = 0, loff1 = 0, wrap = 0xffffffffu;
        if (P.n_lookup_cols > 1) {
          const uint32_t col0 = l_lo / P.max_rows;
          wrap = (col0 + 1) * P.max_rows;
          loff0 = col0 * (P.lookup_col_rows - P.max_rows);
          loff1 = (col0 + 1) * (P.lookup_col_rows - P.max_rows);
        }
        // lanes aligned to the 256-byte groups of the output, like the gate loop (a misaligned warp store costs ~1.7x the
        // LSU wavefronts: tools/stg_wave_probe.cu)
        const uint32_t lpos0 = l_lo + ((l_lo >= wrap) ? loff1 : loff0);
        const int lshift = (int)(lpos0 & 7u);
        const int ln = (int)ch.lk_len;
        for (int i = (int)lane - lshift; i < ln; i += 32) {
          if (i < 0) continue;
          const CellEntry ce = s_cells[ch.lk_off + i];
          const uint32_t src = H2SHA_CE_SRC(ce);
          H2SHA_SCRATCH_READ(src)
          const uint32_t li = l_lo + H2SHA_CE_DST(ce);
          const uint32_t pos = li + ((li >= wrap) ? loff1 : loff0);
          if (lk_out) store_cell2(lk_out + (uint64_t)pos * 8, lo, hi);
          if constexpr (MULT) A.lookup_raw[inst * A.n_lookup_total + li] = ws.raw[src];
          ck_l += (unsigned long long)hash8(lo, hi) * (unsigned long long)(2u * pos + 1u);
        }
      }
      // ---- spread-table columns: limb n -> column n % cols, row n / cols (spread.rs:202,228-231); dense then spread ----
      if (ch.limb_len && (sp_out || A.cks || MULT)) {
        const uint32_t m_lo = limb0 + item.limb_rel;
        for (uint32_t i = lane; i < ch.limb_len; i += 32) {
          const CellEntry ce = s_cells[ch.limb_off + i];
          const uint32_t src = H2SHA_LE_SRC(ce);
          H2SHA_SCRATCH_READ(src)
          const uint32_t n = m_lo + (H2SHA_LE_DST(ce) >> 1), which = H2SHA_LE_DST(ce) & 1u;
          uint32_t row, col;
          if (P.spread_cols_shift >= 0) { row = n >> P.spread_cols_shift; col = n & (P.spread_cols - 1u); }
          else { row = n / P.spread_cols; col = n - row * P.spread_cols; }
          // the (dense, spread) pair of limb n is row `dense` of the spread table: its raw dense value goes to the multiplicity kernel
          if (MULT && which == 0) A.dense_raw[inst * A.n_limb_total + n] = (uint8_t)extract(slots[H2SHA_LE_SLOT(ce)], H2SHA_LE_SH(ce), A.limb_bits);
          const uint32_t pos = (which * P.spread_cols + col) * P.spread_rows + row;
          if (sp_out) store_cell2(sp_out + (uint64_t)pos * 8, lo, hi);
          ck_s += (unsigned long long)hash8(lo, hi) * (unsigned long long)(2u * pos + 1u);
        }
      }
      if (A.cks && jc.batch > 1) {   // batched digest jobs: the items of a warp belong to different instances
        flush_checksums(A.cks, inst, ck_g, ck_l, ck_s, lane);
        ck_g = 0; ck_l = 0; ck_s = 0;
      }
      __syncwarp();  // scratch is overwritten by the next item's fill
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[st]);   // this warp no longer reads the stage
    // ---- checksums: warp reduce, one global atomic per kind and warp (block jobs: one instance per job) ----
    if (A.cks && jc.batch == 1) flush_checksums(A.cks, inst0, ck_g, ck_l, ck_s, lane);
  }
#ifdef H2SHA_DEBUG_TIMING
  if (lane == 0 && (H2SHA_DEBUG_TIMING == 2 ? (warp == 0 || warp == NCONS - 1) : ((blockIdx.x % 37) == 0 && (warp % 7) == 0))) {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    printf("E cta %3d warp %2d: done at +%llu ns, waited %llu ns in %u waits\n", blockIdx.x, warp, t - dbg_t2, dbg_wait, dbg_nwait);
  }
#endif
}

// Table-row multiplicities of one instance from the raw values k_expand<.., 1> left next to the cells: one CTA zeroes the
// instance's bins (258 KB for a 16-bit range table: coalesced, and L2-resident for the atomics that follow), then bins the
// 3.4 k looked-up values and 2 k dense limbs per block.  Never-assigned rows of every lookup input column hold 0 = table row 0.
struct MultArgs {
  const uint32_t* lookup_raw;
  const uint8_t* dense_raw;
  uint32_t* mult;
  uint32_t* bad;
  LookupGeom G;
};
enum { MULT_SMALL_BINS = 4096 };   // looked-up values below this (bytes, zeros: the hot bins) are binned in shared memory
__global__ void __launch_bounds__(512) k_mult_from_raw(const MultArgs A) {
  extern __shared__ uint32_t s_bins[];   // [MULT_SMALL_BINS] range bins of lookup column 0 | [spread_cols << limb_bits] spread bins
  const LookupGeom& G = A.G;
  const uint64_t inst = blockIdx.x;
  const uint64_t mult_words = G.mult_words();
  uint32_t* bins = A.mult + inst * mult_words;
  const uint32_t n_small = min((uint32_t)MULT_SMALL_BINS, 1u << G.lookup_bits), n_sp = G.spread_cols << G.limb_bits;
  uint32_t* s_sp = s_bins + MULT_SMALL_BINS;
  for (uint32_t i = threadIdx.x; i < MULT_SMALL_BINS + n_sp; i += blockDim.x) s_bins[i] = 0;
  __syncthreads();
  // pass A: the hot bins in shared memory (same-address atomics on the zeros and small bytes would serialise in L2)
  uint32_t n_bad = 0;
  const uint32_t* lr = A.lookup_raw + inst * G.n_lookup;
  const uint32_t n0 = G.range_used(0);   // cells of lookup column 0
  for (uint32_t k = threadIdx.x; k < n0; k += blockDim.x) {
    const uint32_t v = lr[k];
    if (v < n_small) atomicAdd(&s_bins[v], 1u);
  }
  const uint8_t* dr = A.dense_raw + inst * G.n_limb;
  for (uint32_t n = threadIdx.x; n < G.n_limb; n += blockDim.x) atomicAdd(&s_sp[(G.spread_cell(n).col << G.limb_bits) + dr[n]], 1u);
  if (threadIdx.x < G.n_lookup_cols + G.spread_cols) {   // never-assigned rows of every lookup input column hold 0 = table row 0
    const uint32_t c = threadIdx.x;
    if (c == 0) { if (G.usable_rows > n0) atomicAdd(&s_bins[0], G.usable_rows - n0); }
    else if (c >= G.n_lookup_cols) {
      const uint32_t cc = c - G.n_lookup_cols, used = G.spread_used(cc);
      if (G.usable_rows > used) atomicAdd(&s_sp[cc << G.limb_bits], G.usable_rows - used);
    }
  }
  __syncthreads();
  // pass B: every bin of the instance written once, coalesced: the shared-memory counts where they exist, zero elsewhere
  {
    uint4* b4 = reinterpret_cast<uint4*>(bins);   // mult_words is a multiple of 4 and the buffer 16-byte aligned: checked on the host
    const uint64_t sp0 = G.range_words();
    for (uint64_t i = threadIdx.x; i < mult_words / 4; i += blockDim.x) {
      uint4 v = make_uint4(0, 0, 0, 0);
      const uint64_t w = i * 4;
      if (w < n_small) v = *reinterpret_cast<const uint4*>(s_bins + w);
      else if (w >= sp0) v = *reinterpret_cast<const uint4*>(s_sp + (w - sp0));
      b4[i] = v;
    }
  }
  __syncthreads();
  // pass C: the (spread-out) large values and the further lookup columns, with global atomics on bins that are now L2-resident
  for (uint32_t k = threadIdx.x; k < G.n_lookup; k += blockDim.x) {
    const uint32_t v = lr[k], col = G.range_cell(k).col;
    if ((v >> G.lookup_bits) != 0) { n_bad++; continue; }
    if (col == 0 && v < n_small) continue;
    atomicAdd(&bins[((uint64_t)col << G.lookup_bits) + v], 1u);
  }
  if (threadIdx.x >= 1 && threadIdx.x < G.n_lookup_cols) {
    const uint32_t c = threadIdx.x, used = G.range_used(c);
    if (G.usable_rows > used) atomicAdd(&bins[(uint64_t)c << G.lookup_bits], G.usable_rows - used);
  }
  if (n_bad && A.bad) atomicAdd(A.bad, n_bad);
}

__global__ void k_mont_debug(const uint64_t* vals, uint64_t* out, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t r[4];
  mont_from_u64(vals[i], r);
  out[4 * i] = r[0]; out[4 * i + 1] = r[1]; out[4 * i + 2] = r[2]; out[4 * i + 3] = r[3];
}

__global__ void k_mont_debug32(const uint64_t* vals, uint64_t* out, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t x[8];
  mont_from_u32((uint32_t)vals[i], x);
  for (int k = 0; k < 4; k++) out[4 * i + k] = (uint64_t)x[2 * k] | ((uint64_t)x[2 * k + 1] << 32);
}

// reference point for the roofline: the plainest possible writer of incompressible 32-byte cells (one 256-bit store per lane,
// consecutive lanes -> consecutive cells), no shared memory, no arithmetic
__global__ void k_store_probe(uint32_t* out, uint64_t n_cells, uint32_t salt) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cells; i += stride) {
    const uint32_t v = (uint32_t)i * 2654435761u + salt;
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(out + i * 8), "r"(v), "r"(v ^ 0x9E3779B1u), "r"(v + 0x85EBCA77u),
                 "r"(v ^ 0xC2B2AE3Du), "r"(v + 0x27D4EB2Fu), "r"(v ^ 0x165667B1u), "r"(v + 0xD3A2646Du), "r"(v ^ 0xFD7046C5u)
                 : "memory");
  }
}

// second reference point (the north star names two rooflines): integer ALU throughput of this GPU for the instruction mix the
// expansion kernel is made of -- 32-bit multiply-adds (IMAD: Barrett / Montgomery limbs, checksum hashes) and 3-input logic ops
// (LOP3: extracts, spreads) -- from 8 independent dependency chains per thread, no memory traffic
__global__ void __launch_bounds__(256) k_int_probe(uint32_t* out, uint32_t iters, uint32_t seed) {
  uint32_t a[8];
#pragma unroll
  for (int i = 0; i < 8; i++) a[i] = seed + threadIdx.x * 8u + i + blockIdx.x;
  const uint32_t m = seed | 1u, x = seed * 2654435761u;
  for (uint32_t it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++) {
      a[i] = a[i] * m + x;                                   // IMAD
      a[i] = (a[i] ^ (a[(i + 1) & 7] & x));                  // LOP3
    }
  }
  uint32_t r = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) r ^= a[i];
  if (r == 0x12345678u) out[blockIdx.x * blockDim.x + threadIdx.x] = r;   // keeps the chains alive, (almost) never stores
}

__global__ void k_zero_ranges(uint4* buf, uint64_t inst_cells, uint64_t n_inst, const uint32_t* ranges /*pos,count pairs*/, uint32_t n_ranges) {
  // grid.y = instance, grid.x strides over the cells of all ranges
  uint64_t inst = blockIdx.y;
  if (inst >= n_inst) return;
  for (uint32_t r = 0; r < n_ranges; r++) {
    uint64_t pos = ranges[2 * r], cnt = ranges[2 * r + 1];
    uint4* p = buf + (inst * inst_cells + pos) * 2;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt * 2; i += (uint64_t)gridDim.x * blockDim.x) p[i] = make_uint4(0, 0, 0, 0);
  }
}

// launch variants (consumer warps, producer warps); selected at engine creation (H2SHA_TUNE "cons=..,prod=..")
struct ExpandVariant {
  int ncons, nprod;
  const void* fn[3];        // by MODE: plain | + lookup multiplicities | + dictionary of distinct values
};
template <int NC, int NP>
ExpandVariant make_variant() {
  return ExpandVariant{NC, NP, {(const void*)k_expand<NC, NP, 0>, (const void*)k_expand<NC, NP, 1>, (const void*)k_expand<NC, NP, 2>}};
}
const ExpandVariant* expand_variants(int* n) {
  // the tuned default and the fallback chain for plans that need more shared memory (fewer consumer warps = less scratch)
  static const ExpandVariant v[] = {make_variant<20, 4>(), make_variant<16, 4>(), make_variant<12, 4>(), make_variant<8, 4>(), make_variant<8, 2>()};
  *n = (int)(sizeof v / sizeof v[0]);
  return v;
}
int tune_value(const char* key, int dflt) {
  const char* t = getenv("H2SHA_TUNE");
  if (!t) return dflt;
  std::string s(t), k = std::string(key) + "=";
  size_t p = s.find(k);
  if (p == std::string::npos) return dflt;
  return atoi(s.c_str() + p + k.size());
}
uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

}  // namespace

// ---------------------------------------------------------------------------------------------------
// host engine
// ---------------------------------------------------------------------------------------------------
// One of the two device-side input / trace workspaces.  Calls alternate between them, so the H2D copy and the trace kernel
// of batch i+1 (on the engine's copy stream) can run while the expansion kernel of batch i still reads its traces.
struct InputSet {
  uint64_t cap_msgs = 0, cap_inst = 0, cap_in = 0;
  uint8_t* d_in = nullptr;            // offsets [n] u64 | lens [n] u32 | precomputed_lens [n] u32 | message bytes: one H2D copy
  uint32_t* d_btrace = nullptr;
  uint32_t* d_dtrace = nullptr;
  uint8_t* d_digests_out = nullptr;
  unsigned long long* d_cks = nullptr;
  unsigned long long* d_counter = nullptr;
  cudaEvent_t trace_done = nullptr;   // recorded on the copy stream after k_trace
  cudaEvent_t expand_done = nullptr;  // recorded on the caller's stream after the last reader of this set (k_expand, D2H copies)
  bool used = false;
  cudaStream_t last_stream = nullptr;
  // inputs resident in this set (reuse_inputs)
  uint64_t n_instances = 0;
  bool has_pre = false;
  const uint8_t* msgs = nullptr;
};
// One slot of the pinned staging ring: the caller's host arrays are copied here before the call returns, so the call itself
// never waits for the device.
struct HostSlot {
  uint8_t* p = nullptr;               // inside the engine's pinned arena (one allocation for the whole ring: cudaHostAlloc costs ~1 ms a call)
  cudaEvent_t copied = nullptr;       // recorded after the H2D copy out of this slot
  bool used = false;
};
enum { H2SHA_N_SETS = 2, H2SHA_N_SLOTS = 8 };

struct h2sha_compact_state;   // export.cuh
struct h2sha_perm_state;      // permutation_product.cuh
struct h2sha_check_items;     // batch_check.cuh

struct h2sha_engine {
  Plan plan;
  int device = 0;
  int n_sms = 0;
  DevPlan dplan{};
  uint8_t* d_blob = nullptr;
  DevDigest* d_digests = nullptr;
  uint32_t* d_zero_ranges[3] = {nullptr, nullptr, nullptr};
  uint32_t n_zero_ranges[3] = {0, 0, 0};
  // input / trace workspaces (grown on demand), pinned staging ring, copy stream
  InputSet sets[H2SHA_N_SETS];
  HostSlot slots[H2SHA_N_SLOTS];
  uint8_t* pinned_arena = nullptr;
  uint64_t slot_cap = 0;             // bytes per ring slot
  cudaStream_t copy_stream = nullptr;
  uint64_t seq = 0;                  // calls that uploaded inputs
  int resident_set = -1;             // set holding the inputs of the last such call
  bool overlap_enabled = true;       // H2SHA_TUNE overlap=0: everything on the caller's stream
  uint64_t trace_warp_below = 2048;  // batches of at most this many messages take k_trace_warp (measured crossover: 1024 x 1 block 13.6 vs 17.8 us, 4096 x 1 block 35 vs 21 us, 512 x 33 blocks 95 vs 373 us)
  uint32_t blocks_per_inst = 0, dtrace_words_per_inst = 0;
  int last_launches = 0;
  int expand_ctas = 0;
  ExpandVariant variant{};
  DevPlan dplan_mult{};              // the plan as a MODE 1 launch sees it: the warps' scratch also holds the raw looked-up values
  bool mult_fits = false;            // ... when that still fits in shared memory
  uint32_t* d_lookup_raw = nullptr;  // [cap][n_lookup] raw looked-up values of the last MODE 1 batch
  uint8_t* d_dense_raw = nullptr;    // [cap][n_limb]
  uint64_t raw_cap = 0;
  uint64_t raw_n = 0;                // instances of the last batch that left raw lists (0: none valid)
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // trace start/stop, expand start/stop
  bool timed = false, timed_expand = false;
  // lookup-argument pre-work (lookup_prework.cuh)
  uint32_t* d_lk_ws = nullptr;    // scans of the permutation kernels
  uint64_t lk_ws_bytes = 0;
  uint32_t* d_lk_tab = nullptr;   // compressed spread table in sorted order
  uint32_t* d_range_tab = nullptr;   // Montgomery form of the range table's values
  uint64_t* d_lp_ws = nullptr;   // lookup product (lookup_product.cuh): spread table, tile products and tile constants
  uint64_t lp_ws_bytes = 0;
  uint64_t* d_chal = nullptr;    // per-instance challenges of the last *_per_instance call: [n][3][4] theta, beta, gamma (Montgomery)
  uint64_t chal_bytes = 0;
  // device-side batch check (batch_check.cuh)
  uint32_t *d_chk_gate_on = nullptr, *d_chk_pairs = nullptr, *d_chk_out_bytes = nullptr;
  uint64_t *d_chk_fixed = nullptr, *d_chk_bytes = nullptr;
  unsigned long long* d_chk_viol = nullptr;
  uint32_t n_chk_gate_on = 0, n_chk_pairs = 0;
  uint32_t* d_chk_counts = nullptr;   // per-instance counts of one chunk (h2sha_check_batch)
  uint64_t chk_counts_cap = 0;       // instances d_chk_counts holds
  h2sha_check_items* chk_items = nullptr;   // every check item's cells (host), built on first use
  // compact hand-off (export.cuh): the cell -> dictionary-entry map, planned on first use
  h2sha_compact_state* compact = nullptr;
  // permutation product (permutation_product.cuh): the moved cells of the last column list, planned on first use
  h2sha_perm_state* perm = nullptr;
};

namespace {

// frees *p (nulling it, so that a later failure leaves no dangling pointer behind) and allocates `bytes`
template <class T>
int dev_realloc(T*& p, size_t bytes) {
  if (p) { cudaFree(p); p = nullptr; }
  CUDA_TRY(cudaMalloc(&p, bytes ? bytes : 16));
  return H2SHA_OK;
}

int ensure_set(h2sha_engine* e, InputSet* S, uint64_t n_inst, uint64_t in_bytes) {
  const uint64_t n_msgs = n_inst * e->plan.digests.size();
  int rc;
  if (n_msgs > S->cap_msgs || n_inst > S->cap_inst) {
    S->cap_msgs = 0; S->cap_inst = 0;
    if ((rc = dev_realloc(S->d_btrace, n_inst * e->blocks_per_inst * (uint64_t)TR_BLOCK_WORDS * 4))) return rc;
    if ((rc = dev_realloc(S->d_dtrace, n_inst * (uint64_t)e->dtrace_words_per_inst * 4))) return rc;
    if ((rc = dev_realloc(S->d_digests_out, n_msgs * 32))) return rc;
    if ((rc = dev_realloc(S->d_cks, n_inst * 32))) return rc;
    S->cap_msgs = n_msgs; S->cap_inst = n_inst;
  }
  if (in_bytes + 16 > S->cap_in) {
    S->cap_in = 0;
    if ((rc = dev_realloc(S->d_in, in_bytes + 16))) return rc;
    S->cap_in = in_bytes + 16;
  }
  return H2SHA_OK;
}

int ensure_slot(h2sha_engine* e, HostSlot* H, uint64_t bytes) {
  if (bytes > e->slot_cap) {
    // grow the whole ring: every slot has to be idle first
    for (HostSlot& X : e->slots)
      if (X.used) { CUDA_TRY(cudaEventSynchronize(X.copied)); X.used = false; }
    if (e->pinned_arena) { cudaFreeHost(e->pinned_arena); e->pinned_arena = nullptr; }
    e->slot_cap = 0;
    const uint64_t cap = (std::max<uint64_t>(bytes + bytes / 4, 1 << 16) + 4095) / 4096 * 4096;
    CUDA_TRY(cudaHostAlloc((void**)&e->pinned_arena, cap * H2SHA_N_SLOTS, cudaHostAllocDefault));
    e->slot_cap = cap;
    for (int i = 0; i < H2SHA_N_SLOTS; i++) e->slots[i].p = e->pinned_arena + (uint64_t)i * cap;
  }
  if (H->used) { CUDA_TRY(cudaEventSynchronize(H->copied)); H->used = false; }   // the copy that last read this slot (8 calls ago): back-pressure on a host that runs far ahead
  return H2SHA_OK;
}

struct EngineGuard {   // error paths of h2sha_create: releases whatever has been allocated so far
  h2sha_engine* e;
  ~EngineGuard() { if (e) h2sha_destroy(e); }
};

}  // namespace

extern "C" {

const char* h2sha_last_error(void) { return g_err.c_str(); }

#ifndef H2SHA_BUILD_ID_STR
#define H2SHA_BUILD_ID_STR "unstamped"
#endif
const char* h2sha_build_id(void) {
  static const char id[] = "H2SHA_BUILD_ID=" H2SHA_BUILD_ID_STR;   // build.py finds this marker in the file
  return id + 15;
}

int h2sha_create(const h2sha_config_t* cfg, h2sha_engine_t** out) {
  if (!cfg || !out) return set_err(H2SHA_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->n_digests == 0 || !cfg->max_variable_byte_sizes) return set_err(H2SHA_EINVAL, "max_variable_byte_sizes is empty");
  // device == -1: plan-only engine (layout / shape / handle queries on the host); it can never generate a witness
  const bool plan_only = cfg->device == -1;
  cudaDeviceProp prop{};
  if (!plan_only) {
    int n_dev = 0;
    cudaError_t ce = cudaGetDeviceCount(&n_dev);
    if (ce != cudaSuccess || n_dev == 0)
      return set_err(H2SHA_ECUDA, std::string("no usable CUDA device (this engine has no CPU path): ") + cudaGetErrorString(ce));
    if (cfg->device < 0 || cfg->device >= n_dev) return set_err(H2SHA_EINVAL, "bad device ordinal");
    CUDA_TRY(cudaSetDevice(cfg->device));
    CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10) return set_err(H2SHA_ECUDA, "this engine is built for sm_100a (B200) only");
  }

  Config pc;
  pc.max_variable_byte_sizes.assign(cfg->max_variable_byte_sizes, cfg->max_variable_byte_sizes + cfg->n_digests);
  if (cfg->max_rows) pc.max_rows = cfg->max_rows;
  if (cfg->lookup_bits) pc.lookup_bits = cfg->lookup_bits;
  if (cfg->num_bits_lookup) pc.limb_bits = cfg->num_bits_lookup;
  if (cfg->num_advice_columns) pc.spread_cols = cfg->num_advice_columns;
  pc.is_input_range_check = cfg->is_input_range_check ? 1 : 0;
  pc.record_shape = cfg->build_shape ? 1 : 0;
  if (cfg->block_parts) pc.block_parts = cfg->block_parts;
  pc.block_parts = (uint32_t)tune_value("parts", (int)pc.block_parts);
  pc.max_fill = (uint32_t)tune_value("fill", (int)pc.max_fill);
  pc.resident_consts = (uint32_t)tune_value("res", (int)pc.resident_consts);
  pc.digest_batch = (uint32_t)tune_value("dbatch", (int)pc.digest_batch);
  h2sha_engine* e = new h2sha_engine();
  e->device = cfg->device;
  EngineGuard guard{e};   // every early return below destroys the half-built engine (h2sha_destroy frees what exists)
  std::string err;
  if (!build_plan(pc, &e->plan, &err)) return set_err(H2SHA_EINVAL, err);
  Plan& P = e->plan;
  if (cfg->gate_col_rows) { if (cfg->gate_col_rows < P.gate_col_rows) return set_err(H2SHA_EINVAL, "gate_col_rows too small"); P.gate_col_rows = cfg->gate_col_rows; }
  if (cfg->lookup_col_rows) { if (cfg->lookup_col_rows < P.lookup_col_rows) return set_err(H2SHA_EINVAL, "lookup_col_rows too small"); P.lookup_col_rows = cfg->lookup_col_rows; }
  if (cfg->spread_rows) { if (cfg->spread_rows < P.spread_rows) return set_err(H2SHA_EINVAL, "spread_rows too small"); P.spread_rows = cfg->spread_rows; }
  if ((P.gate_col_rows | P.lookup_col_rows | P.spread_rows) & 1u) return set_err(H2SHA_EINVAL, "column row strides must be even");
  if (cfg->num_lookup_advice) {   // RangeConfig's NUM_LOOKUP_ADVICE: a configure-time input of halo2-base, not something the cells decide
    if (cfg->num_lookup_advice < P.n_lookup_cols)
      return set_err(H2SHA_EINVAL, "num_lookup_advice: the looked-up cells need " + std::to_string(P.n_lookup_cols) + " lookup advice column(s)");
    P.n_lookup_cols = cfg->num_lookup_advice;
  }
  e->n_sms = prop.multiProcessorCount;
  {
    uint32_t bp0 = 0, dw0 = 0;
    for (auto& dgp : P.digests) { bp0 += dgp.n_blocks; dw0 += dgp.trace_words; }
    e->blocks_per_inst = bp0; e->dtrace_words_per_inst = dw0;
  }
  compute_zero_ranges(&P);  // against the final (possibly widened) strides
  if (plan_only) { guard.e = nullptr; *out = e; return H2SHA_OK; }

  // ---- field constants ----
  FrConsts fc;
  memcpy(fc.p, fr::P, 32);
  U256 r1 = fr::mont_r();
  memcpy(fc.r1, r1.l, 32);
  fc.mu = fr::floor_pow2_div_p(317);
  fc.mu32 = (uint32_t)fr::floor_pow2_div_p(285);
  fc.pad = 0;
  fc.ninv = fr::neg_p_inv64();
  CUDA_TRY(cudaMemcpyToSymbol(c_fr, &fc, sizeof fc));

  // ---- per-digest device info ----
  std::vector<DevDigest> dds(P.digests.size());
  uint32_t bp = 0, dw = 0;
  for (size_t d = 0; d < P.digests.size(); d++) {
    dds[d].dp = P.digests[d];
    dds[d].blk_prefix = bp; dds[d].dtrace_off = dw;
    bp += P.digests[d].n_blocks; dw += P.digests[d].trace_words;
  }
  e->blocks_per_inst = bp; e->dtrace_words_per_inst = dw;

  // ---- blob ----
  DevPlan& D = e->dplan;
  std::vector<uint8_t> blob;
  auto put = [&](const void* p, size_t bytes) {
    uint32_t off = (uint32_t)blob.size();
    blob.resize(align_up((uint32_t)(off + bytes), 16), 0);
    if (bytes) memcpy(blob.data() + off, p, bytes);
    return off;
  };
  D.off_fill = put(P.fill.data(), P.fill.size() * sizeof(FillEntry));
  D.off_cells = put(P.cells.data(), P.cells.size() * sizeof(CellEntry));
  D.off_chunks = put(P.chunks.data(), P.chunks.size() * sizeof(Chunk));
  D.off_items = put(P.items.data(), P.items.size() * sizeof(ItemDesc));
  {
    std::vector<uint64_t> lo(2 * P.mont_table.size()), hi(2 * P.mont_table.size());
    for (size_t i = 0; i < P.mont_table.size(); i++) {
      lo[2 * i] = P.mont_table[i].l[0]; lo[2 * i + 1] = P.mont_table[i].l[1];
      hi[2 * i] = P.mont_table[i].l[2]; hi[2 * i + 1] = P.mont_table[i].l[3];
    }
    D.off_table_lo = put(lo.data(), lo.size() * 8);
    D.off_table_hi = put(hi.data(), hi.size() * 8);
  }
  D.off_resident = put(P.resident.data(), P.resident.size() * 4);
  D.n_resident = (uint32_t)P.resident.size();
  D.off_prog = put(P.prog.data(), P.prog.size() * sizeof(VmIns));
  D.off_groups = put(P.groups.data(), P.groups.size() * sizeof(UnitGroup));
  D.off_tasks = put(P.tasks.data(), P.tasks.size() * sizeof(WarpTask));
  D.off_types = put(P.types.data(), P.types.size() * sizeof(UnitType));
  D.off_classes = put(P.classes.data(), P.classes.size() * sizeof(JobClass));
  D.off_raw = put(P.raw_consts.data(), P.raw_consts.size() * 8);
  D.off_breaks = put(P.breaks.data(), P.breaks.size() * 4);
  D.off_digests = put(dds.data(), dds.size() * sizeof(DevDigest));
  D.off_item_dict = put(P.item_dict.data(), P.item_dict.size() * 4);
  D.blob_bytes = (uint32_t)blob.size();
  D.n_breaks = (uint32_t)P.breaks.size();
  D.n_digests = (uint32_t)P.digests.size();
  D.n_block_parts = P.n_block_parts;
  D.n_classes = (uint32_t)P.classes.size();
  D.off_trace = D.blob_bytes;
  D.stage_off_slots = align_up(4 * std::max<uint32_t>(P.max_trace_words, TR_BLOCK_WORDS_WITH_K), 16);
  D.stage_off_desc = align_up(D.stage_off_slots + 8 * (P.max_slots + 1), 16);
  D.stage_bytes = align_up(D.stage_off_desc + (uint32_t)sizeof(StageDesc), 16);
  {
    // launch variant: the tuned default (or H2SHA_TUNE cons=/prod=); when the plan of an unusual configuration does not
    // fit in shared memory with it, fall back to variants with fewer consumer warps
    int nv = 0;
    const ExpandVariant* vs = expand_variants(&nv);
    const bool forced = getenv("H2SHA_TUNE") && (strstr(getenv("H2SHA_TUNE"), "cons=") || strstr(getenv("H2SHA_TUNE"), "prod="));
    const int pref[][2] = {{tune_value("cons", 20), tune_value("prod", 4)}, {16, 4}, {12, 4}, {8, 4}, {8, 2}};
    bool ok = false;
    for (int pi = 0; pi < (forced ? 1 : 5) && !ok; pi++) {
      for (int i = 0; i < nv && !ok; i++) {
        if (vs[i].ncons != pref[pi][0] || vs[i].nprod != pref[pi][1]) continue;
        e->variant = vs[i];
        D.max_fill = pc.max_fill;
        D.scratch_bytes = pc.max_fill * 32;   // per consumer warp: the scratch table
        D.off_scratch = align_up(D.off_trace + e->variant.nprod * D.stage_bytes, 128);
        D.off_misc = align_up(D.off_scratch + e->variant.ncons * D.scratch_bytes, 16);
        D.smem_bytes = D.off_misc + 2 * e->variant.nprod * 8;
        ok = D.smem_bytes <= 227 * 1024;
      }
    }
    if (!ok) return set_err(H2SHA_EINVAL, "configuration needs more than 227 KB of shared memory (or H2SHA_TUNE names no launch variant)");
  }
  D.max_rows = pc.max_rows; D.spread_cols = pc.spread_cols;
  const uint32_t mult_scratch = pc.max_fill * 36, mult_misc = align_up(D.off_scratch + e->variant.ncons * mult_scratch, 16);
  e->mult_fits = mult_misc + 2 * e->variant.nprod * 8 <= 227 * 1024;
  D.spread_cols_shift = -1;
  for (int sh = 0; sh < 16; sh++) if ((1u << sh) == pc.spread_cols) D.spread_cols_shift = sh;
  D.n_gate_cols = P.n_gate_cols; D.gate_col_rows = P.gate_col_rows;
  D.n_lookup_cols = P.n_lookup_cols; D.lookup_col_rows = P.lookup_col_rows; D.spread_rows = P.spread_rows;
  D.blocks_per_inst = bp; D.dtrace_words_per_inst = dw;
  D.gate_inst_cells = (uint64_t)P.n_gate_cols * P.gate_col_rows;
  D.lookup_inst_cells = lookup_geom(P).lookup_inst_cells;
  D.spread_inst_cells = lookup_geom(P).spread_inst_cells;
  CUDA_TRY(cudaMalloc(&e->d_blob, blob.size()));
  CUDA_TRY(cudaMemcpy(e->d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice));
  D.blob = e->d_blob;
  CUDA_TRY(cudaMalloc(&e->d_digests, dds.size() * sizeof(DevDigest)));
  CUDA_TRY(cudaMemcpy(e->d_digests, dds.data(), dds.size() * sizeof(DevDigest), cudaMemcpyHostToDevice));
  for (int b = 0; b < 3; b++) {
    std::vector<uint32_t> rr;
    for (auto& z : P.zero_ranges) if ((int)z.buf == b) { rr.push_back(z.pos); rr.push_back(z.count); }
    e->n_zero_ranges[b] = (uint32_t)rr.size() / 2;
    if (!rr.empty()) {
      CUDA_TRY(cudaMalloc(&e->d_zero_ranges[b], rr.size() * 4));
      CUDA_TRY(cudaMemcpy(e->d_zero_ranges[b], rr.data(), rr.size() * 4, cudaMemcpyHostToDevice));
    }
  }
  const int expand_threads = (e->variant.ncons + e->variant.nprod) * 32;
  // the attribute belongs to the kernel function, not to this engine: always raise it to the 227 KB cap, so that engines of
  // different configurations that share a launch variant never lower each other's limit
  for (const void* fn : e->variant.fn) CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  int occ = 0;
  for (const void* fn : e->variant.fn) {
    int o = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, fn, expand_threads, D.smem_bytes));
    occ = (fn == e->variant.fn[0]) ? o : std::min(occ, o);
  }
  if (occ < 1) return set_err(H2SHA_ECUDA, "expand kernel does not fit on an SM");
  if (getenv("H2SHA_VERBOSE"))
    fprintf(stderr, "[h2sha] k_expand<%d,%d>: blob %u B, stage %u B x %d, scratch %u B x %d, shared memory %u B, %d CTAs\n", e->variant.ncons, e->variant.nprod,
            D.blob_bytes, D.stage_bytes, e->variant.nprod, D.scratch_bytes, e->variant.ncons, D.smem_bytes, occ * e->n_sms);
  e->expand_ctas = occ * e->n_sms;
  e->dplan_mult = e->dplan;
  if (e->mult_fits) { e->dplan_mult.scratch_bytes = mult_scratch; e->dplan_mult.off_misc = mult_misc; e->dplan_mult.smem_bytes = mult_misc + 2 * e->variant.nprod * 8; }
  // ---- copy stream, events, job counters ----
  // the latency setting keeps everything on the caller's stream (trace kernel -> expansion with programmatic dependent launch): handing
  // the copy and the trace kernel to the second stream costs two event hops, 6 us of a 64 us digest
  e->overlap_enabled = tune_value("overlap", pc.block_parts >= 12 ? 0 : 1) != 0;
  e->trace_warp_below = (uint64_t)tune_value("tracewarp", 2048);
  CUDA_TRY(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
  for (InputSet& S : e->sets) {
    CUDA_TRY(cudaEventCreateWithFlags(&S.trace_done, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&S.expand_done, cudaEventDisableTiming));
    CUDA_TRY(cudaMalloc(&S.d_counter, 8));
  }
  for (HostSlot& H : e->slots) CUDA_TRY(cudaEventCreateWithFlags(&H.copied, cudaEventDisableTiming));
  guard.e = nullptr;
  *out = e;
  return H2SHA_OK;
}

void h2sha_free_compact_state(h2sha_compact_state* s);   // defined after export.cuh (complete type)
void h2sha_free_perm_state(h2sha_perm_state* s);         // permutation_product.cuh
void h2sha_free_check_items(h2sha_check_items* c);      // batch_check.cuh

void h2sha_destroy(h2sha_engine_t* e) {
  if (!e) return;
  h2sha_free_compact_state(e->compact); e->compact = nullptr;
  h2sha_free_check_items(e->chk_items); e->chk_items = nullptr;
  if (e->device < 0) { delete e; return; }
  cudaSetDevice(e->device);
  if (e->copy_stream) { cudaStreamSynchronize(e->copy_stream); cudaStreamDestroy(e->copy_stream); }
  cudaFree(e->d_blob); cudaFree(e->d_digests);
  for (int b = 0; b < 3; b++) cudaFree(e->d_zero_ranges[b]);
  for (InputSet& S : e->sets) {
    if (S.expand_done && S.used) cudaEventSynchronize(S.expand_done);   // no kernel of ours may still read the workspace
    cudaFree(S.d_in); cudaFree(S.d_btrace); cudaFree(S.d_dtrace); cudaFree(S.d_digests_out); cudaFree(S.d_cks); cudaFree(S.d_counter);
    if (S.trace_done) cudaEventDestroy(S.trace_done);
    if (S.expand_done) cudaEventDestroy(S.expand_done);
  }
  for (HostSlot& H : e->slots)
    if (H.copied) cudaEventDestroy(H.copied);
  if (e->pinned_arena) cudaFreeHost(e->pinned_arena);
  for (int i = 0; i < 4; i++) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
  cudaFree(e->d_lk_ws); cudaFree(e->d_lk_tab); cudaFree(e->d_range_tab); cudaFree(e->d_lp_ws); cudaFree(e->d_chal); cudaFree(e->d_lookup_raw); cudaFree(e->d_dense_raw);
  h2sha_free_perm_state(e->perm); e->perm = nullptr;
  cudaFree(e->d_chk_gate_on); cudaFree(e->d_chk_pairs); cudaFree(e->d_chk_out_bytes); cudaFree(e->d_chk_fixed); cudaFree(e->d_chk_bytes); cudaFree(e->d_chk_viol); cudaFree(e->d_chk_counts);
  delete e;
}

int h2sha_get_layout(const h2sha_engine_t* e, h2sha_layout_t* L) {
  if (!e || !L) return set_err(H2SHA_EINVAL, "null argument");
  const Plan& P = e->plan;
  memset(L, 0, sizeof *L);
  L->n_digests = (uint32_t)P.digests.size();
  L->n_gate_cells = P.n_gate; L->n_lookup_cells = P.n_lookup; L->n_spread_limbs = P.n_limb;
  L->n_gate_cols = P.n_gate_cols; L->gate_col_rows = P.gate_col_rows;
  L->n_lookup_cols = P.n_lookup_cols; L->lookup_col_rows = P.lookup_col_rows;
  L->n_spread_cols = 2 * P.cfg.spread_cols; L->spread_rows = P.spread_rows;
  L->n_blocks = e->blocks_per_inst;
  L->n_fixed = (uint32_t)P.fixed_consts.size(); L->n_copies = (uint32_t)P.copies.size();
  uint32_t on = 0; for (uint8_t s : P.selectors) on += s;
  L->n_selectors_on = on;
  L->cells_per_instance = P.cells_per_instance();
  L->gate_bytes = (uint64_t)P.n_gate_cols * P.gate_col_rows * 32;
  L->lookup_bytes = (uint64_t)P.n_lookup_cols * P.lookup_col_rows * 32;
  L->spread_bytes = (uint64_t)2 * P.cfg.spread_cols * P.spread_rows * 32;
  return H2SHA_OK;
}

int h2sha_get_breaks(const h2sha_engine_t* e, uint32_t* breaks) {
  if (!e || !breaks) return set_err(H2SHA_EINVAL, "null argument");
  memcpy(breaks, e->plan.breaks.data(), e->plan.breaks.size() * 4);
  return H2SHA_OK;
}

int h2sha_get_handles(const h2sha_engine_t* e, uint32_t d, uint32_t* input_len_idx, uint32_t* input_bytes_idx, uint32_t* output_bytes_idx) {
  if (!e || d >= e->plan.handles.size()) return set_err(H2SHA_EINVAL, "bad digest index");
  const DigestHandles& h = e->plan.handles[d];
  if (input_len_idx) *input_len_idx = h.input_len_idx;
  if (input_bytes_idx) memcpy(input_bytes_idx, h.input_bytes_idx.data(), h.input_bytes_idx.size() * 4);
  if (output_bytes_idx) memcpy(output_bytes_idx, h.output_bytes_idx, 32 * 4);
  return H2SHA_OK;
}

int h2sha_get_digest_ranges(const h2sha_engine_t* e, uint32_t* ranges) {
  if (!e || !ranges) return set_err(H2SHA_EINVAL, "null argument");
  const Plan& P = e->plan;
  for (size_t d = 0; d < P.digests.size(); d++) {
    const bool last = d + 1 == P.digests.size();
    uint32_t* r = ranges + 6 * d;
    r[0] = P.digests[d].gate_base; r[1] = last ? P.n_gate : P.digests[d + 1].gate_base;
    r[2] = P.digests[d].lk_base; r[3] = last ? P.n_lookup : P.digests[d + 1].lk_base;
    r[4] = P.digests[d].limb_base; r[5] = last ? P.n_limb : P.digests[d + 1].limb_base;
  }
  return H2SHA_OK;
}

int h2sha_get_shape(const h2sha_engine_t* e, uint8_t* selectors, uint32_t* copies, uint64_t* fixed, uint32_t* lookup_src,
                    uint32_t* limb_dense_src, uint32_t* limb_spread_src) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  const Plan& P = e->plan;
  if (!P.cfg.record_shape) return set_err(H2SHA_EINVAL, "engine was created without build_shape");
  if (selectors) memcpy(selectors, P.selectors.data(), P.selectors.size());
  if (copies) memcpy(copies, P.copies.data(), P.copies.size() * sizeof(CopyPair));
  if (fixed) memcpy(fixed, P.fixed_consts.data(), P.fixed_consts.size() * 32);
  if (lookup_src) memcpy(lookup_src, P.lookup_cells.data(), P.lookup_cells.size() * 4);
  if (limb_dense_src) memcpy(limb_dense_src, P.limb_gate_dense.data(), P.limb_gate_dense.size() * 4);
  if (limb_spread_src) memcpy(limb_spread_src, P.limb_gate_spread.data(), P.limb_gate_spread.size() * 4);
  return H2SHA_OK;
}

int h2sha_get_lookup_tables(const h2sha_engine_t* e, uint64_t* table_dense, uint64_t* table_spread, uint32_t* n_spread_rows, uint32_t* n_range_rows) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  const uint32_t bits = e->plan.cfg.limb_bits, n = 1u << bits;
  for (uint32_t i = 0; i < n; i++) {
    uint64_t sp = 0;
    for (uint32_t b = 0; b < bits; b++) sp |= (uint64_t)((i >> b) & 1u) << (2 * b);   // spread.rs:171-180
    if (table_dense) table_dense[i] = i;
    if (table_spread) table_spread[i] = sp;
  }
  if (n_spread_rows) *n_spread_rows = n;
  if (n_range_rows) *n_range_rows = 1u << e->plan.cfg.lookup_bits;
  return H2SHA_OK;
}

int h2sha_digest_batch(h2sha_engine_t* e, const h2sha_batch_t* b) {
  if (!e || !b) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): witness generation needs a CUDA device; there is no CPU path");
  if (b->n_instances == 0) return H2SHA_OK;
  const Plan& P = e->plan;
  const uint32_t D = (uint32_t)P.digests.size();
  const uint64_t n_msgs = b->n_instances * D;
  if (n_msgs > 0xffffffffull) return set_err(H2SHA_EINVAL, "batch too large");
  if (b->only_digest > D) return set_err(H2SHA_EINVAL, "only_digest names a digest() call the configuration does not have");
  const bool want_raw = b->lookup_mult_dev || b->keep_lookup_raw;
  if (b->compact_dict && (want_raw || b->only_digest))
    return set_err(H2SHA_EINVAL, "compact_dict cannot be combined with lookup_mult_dev or only_digest (separate kernel instantiations): issue two calls");
  if (want_raw) {
    if (b->only_digest) return set_err(H2SHA_EINVAL, "lookup multiplicities need every digest() call of the region (only_digest must be 0)");
    if (!b->gate || !b->lookup || !b->spread) return set_err(H2SHA_EINVAL, "lookup multiplicities are counted while the cells are written: gate, lookup and spread must be given");
    if (!e->mult_fits) return set_err(H2SHA_EINVAL, "this configuration leaves no shared memory for the fused multiplicity count: use h2sha_lookup_multiplicities");
    if (P.cfg.limb_bits > 8) return set_err(H2SHA_EINVAL, "the fused multiplicity count keeps the spread-table bins in shared memory: num_bits_lookup <= 8");
  }
  if (b->lookup_mult_dev) {
    if (b->mult_usable_rows < lookup_geom(P).min_usable_rows()) return set_err(H2SHA_EINVAL, "mult_usable_rows is smaller than an assigned column or a lookup table");
    if (P.cfg.lookup_bits < 2 || P.cfg.limb_bits < 2 || ((uintptr_t)b->lookup_mult_dev & 15u)) return set_err(H2SHA_EINVAL, "lookup_mult_dev must be 16-byte aligned (tables of >= 4 rows)");
  }
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)b->stream;
  const bool timed = b->time_kernels != 0;
  InputSet* S = nullptr;
  cudaStream_t ts = st;        // stream of the H2D copy and the trace kernel
  bool overlap = false;
  if (b->reuse_inputs) {
    if (e->resident_set < 0 || b->n_instances > e->sets[e->resident_set].n_instances)
      return set_err(H2SHA_EINVAL, "reuse_inputs: no resident inputs for that many instances");
    S = &e->sets[e->resident_set];
    if (S->used && S->last_stream != st) CUDA_TRY(cudaStreamWaitEvent(st, S->expand_done, 0));   // ordered after the call that left them there
  } else {
    if (!b->msgs && b->msgs_bytes) return set_err(H2SHA_EINVAL, "msgs is null");
    if (!b->offsets || !b->lens) return set_err(H2SHA_EINVAL, "offsets / lens are null");
    // every host array is staged in the engine's pinned ring before the call returns: the call only enqueues
    const uint64_t hdr = n_msgs * 16;
    const uint64_t in_bytes = hdr + (b->msgs_on_device ? 0 : b->msgs_bytes);
    HostSlot* H = &e->slots[e->seq % H2SHA_N_SLOTS];
    int rc = ensure_slot(e, H, in_bytes);
    if (rc) return rc;
    uint64_t* h_off = reinterpret_cast<uint64_t*>(H->p);
    uint32_t* h_len = reinterpret_cast<uint32_t*>(H->p + n_msgs * 8);
    uint32_t* h_pre = reinterpret_cast<uint32_t*>(H->p + n_msgs * 12);
    // the reference's panics (lib.rs:89-90) become error returns; lengths are checked in 64 bits (no wrap on the device)
    for (uint64_t m = 0; m < n_msgs; m++) {
      const uint32_t maxb = P.digests[m % D].max_bytes;
      const uint64_t len = b->lens[m], pre = b->precomputed_lens ? b->precomputed_lens[m] : 0, off = b->offsets[m];
      if (pre % 64 != 0) return set_err(H2SHA_EPANIC, "precomputed_input_len is not a multiple of 64 (lib.rs:89), message " + std::to_string(m));
      const uint64_t padded = (len + 9 + 63) / 64 * 64;
      if (padded < pre || padded - pre > maxb)
        return set_err(H2SHA_EPANIC, "padded input does not fit max_variable_byte_size (lib.rs:90), message " + std::to_string(m));
      if (off > b->msgs_bytes || len > b->msgs_bytes - off) return set_err(H2SHA_EINVAL, "message " + std::to_string(m) + " exceeds msgs_bytes");
      h_off[m] = off; h_len[m] = (uint32_t)len; h_pre[m] = (uint32_t)pre;
    }
    if (!b->msgs_on_device && b->msgs_bytes) memcpy(H->p + hdr, b->msgs, b->msgs_bytes);
    S = &e->sets[e->seq % H2SHA_N_SETS];
    e->resident_set = -1;
    if ((rc = ensure_set(e, S, b->n_instances, in_bytes))) return rc;
    // host in, host out (no caller-owned device result buffer the trace kernel would have to touch early): the copy and
    // the trace kernel go to the engine's copy stream and overlap the previous batch's expansion on the caller's stream
    overlap = e->overlap_enabled && !b->msgs_on_device && !b->digests_dev && !b->checksums_dev && !timed;
    ts = overlap ? e->copy_stream : st;
    if (S->used && !(ts == st && S->last_stream == st)) CUDA_TRY(cudaStreamWaitEvent(ts, S->expand_done, 0));
    CUDA_TRY(cudaMemcpyAsync(S->d_in, H->p, in_bytes, cudaMemcpyHostToDevice, ts));
    CUDA_TRY(cudaEventRecord(H->copied, ts));
    H->used = true;
    S->n_instances = b->n_instances; S->has_pre = b->precomputed_lens != nullptr;
    S->msgs = b->msgs_on_device ? b->msgs : S->d_in + hdr;
    e->resident_set = (int)(e->seq % H2SHA_N_SETS);
    e->seq++;
  }
  e->timed = timed; e->timed_expand = false;
  if (timed && !e->ev[0])
    for (int i = 0; i < 4; i++) CUDA_TRY(cudaEventCreate(&e->ev[i]));

  // caller-owned device result buffers are written on the caller's stream only; the overlap path (never taken when they
  // are given) uses the set's own buffers
  uint8_t* dig_dev = b->digests_dev ? b->digests_dev : (b->digests_host ? S->d_digests_out : nullptr);
  unsigned long long* cks_dev = b->checksums_dev ? (unsigned long long*)b->checksums_dev : (b->checksums_host ? S->d_cks : nullptr);
  int launches = 0;
  const uint64_t cap_n = S->n_instances * D;   // the header layout follows the uploaded batch, not this (possibly smaller) one
  TraceArgs ta{};
  ta.n_msgs = n_msgs; ta.n_digests = D; ta.msgs = S->msgs;
  ta.offsets = reinterpret_cast<const uint64_t*>(S->d_in);
  ta.lens = reinterpret_cast<const uint32_t*>(S->d_in + cap_n * 8);
  ta.pre_lens = S->has_pre ? reinterpret_cast<const uint32_t*>(S->d_in + cap_n * 12) : nullptr;
  ta.btrace = S->d_btrace; ta.dtrace = S->d_dtrace; ta.digests = dig_dev; ta.digests_plan = e->d_digests;
  ta.blocks_per_inst = e->blocks_per_inst; ta.dtrace_words_per_inst = e->dtrace_words_per_inst;
  const bool expand = b->gate || b->lookup || b->spread || cks_dev || b->compact_dict;
  ta.job_counter = expand ? S->d_counter : nullptr;
  ta.cks = cks_dev;
  if (want_raw) {
    e->raw_n = 0;
    if (b->n_instances > e->raw_cap) {
      e->raw_cap = 0;
      int rc2;
      if ((rc2 = dev_realloc(e->d_lookup_raw, b->n_instances * (uint64_t)P.n_lookup * 4))) return rc2;
      if ((rc2 = dev_realloc(e->d_dense_raw, b->n_instances * (uint64_t)P.n_limb))) return rc2;
      e->raw_cap = b->n_instances;
    }
    if (b->lookup_mult_dev && b->mult_not_in_table_dev) CUDA_TRY(cudaMemsetAsync(b->mult_not_in_table_dev, 0, 4, st));
  }
  if (timed) CUDA_TRY(cudaEventRecord(e->ev[0], ts));
  // few messages: the warp-per-message kernel (latency); many: one thread per message (throughput).  H2SHA_TUNE "tracewarp=N" moves the switch.
  if (n_msgs <= e->trace_warp_below) k_trace_warp<<<(unsigned)n_msgs, 32, 0, ts>>>(ta);
  else k_trace<<<(unsigned)((n_msgs + 63) / 64), 64, 0, ts>>>(ta);
  launches++;
  CUDA_TRY(cudaGetLastError());
  if (timed) CUDA_TRY(cudaEventRecord(e->ev[1], ts));
  if (overlap) {
    CUDA_TRY(cudaEventRecord(S->trace_done, ts));
    CUDA_TRY(cudaStreamWaitEvent(st, S->trace_done, 0));
  }
  if (expand) {
    JobArgs ja{};
    ja.n_inst = b->n_instances; ja.btrace = S->d_btrace; ja.dtrace = S->d_dtrace;
    ja.gate = (uint32_t*)b->gate; ja.lookup = (uint32_t*)b->lookup; ja.spread = (uint32_t*)b->spread;
    ja.cks = cks_dev; ja.job_counter = S->d_counter; ja.only_digest = b->only_digest;
    if (b->compact_dict) { ja.dict = (uint32_t*)b->compact_dict; ja.dict_inst_cells = P.dict_cells; }
    if (want_raw) {
      ja.lookup_raw = e->d_lookup_raw; ja.dense_raw = e->d_dense_raw;
      ja.limb_bits = P.cfg.limb_bits; ja.n_lookup_total = P.n_lookup; ja.n_limb_total = P.n_limb;
    }
    uint64_t n_jobs = b->n_instances * (uint64_t)e->blocks_per_inst * P.n_block_parts;
    for (size_t c = P.n_block_parts; c < P.classes.size(); c++) n_jobs += (b->n_instances + P.classes[c].batch - 1) / P.classes[c].batch;
    unsigned grid = (unsigned)std::min<uint64_t>(n_jobs, (uint64_t)e->expand_ctas);
    if (timed) CUDA_TRY(cudaEventRecord(e->ev[2], st));
    {
      // programmatic dependent launch: prologue (plan -> shared memory) overlaps the trace kernel when both are on one stream
      const DevPlan& dp = want_raw ? e->dplan_mult : e->dplan;
      void* args[2] = {(void*)&dp, (void*)&ja};
      cudaLaunchConfig_t lc{};
      lc.gridDim = dim3(grid); lc.blockDim = dim3((e->variant.ncons + e->variant.nprod) * 32);
      lc.dynamicSmemBytes = dp.smem_bytes; lc.stream = st;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[0].val.programmaticStreamSerializationAllowed = (timed || overlap) ? 0 : 1;   // plain serialisation when kernels are timed individually
      lc.attrs = at; lc.numAttrs = 1;
      CUDA_TRY(cudaLaunchKernelExC(&lc, e->variant.fn[want_raw ? 1 : (b->compact_dict ? 2 : 0)], args));
    }
    launches++;
    CUDA_TRY(cudaGetLastError());
    if (want_raw) e->raw_n = b->n_instances;
    if (b->lookup_mult_dev) {
      MultArgs ma{};
      ma.lookup_raw = e->d_lookup_raw; ma.dense_raw = e->d_dense_raw; ma.mult = b->lookup_mult_dev; ma.bad = b->mult_not_in_table_dev;
      ma.G = lookup_geom(P, b->mult_usable_rows);
      const size_t mult_smem = ((size_t)MULT_SMALL_BINS + ((size_t)P.cfg.spread_cols << P.cfg.limb_bits)) * 4;
      if (mult_smem > 48 * 1024) return set_err(H2SHA_EINVAL, "spread tables too large for the multiplicity kernel's shared memory");
      k_mult_from_raw<<<(unsigned)b->n_instances, 512, mult_smem, st>>>(ma);
      launches++;
      CUDA_TRY(cudaGetLastError());
    }
    if (timed) { CUDA_TRY(cudaEventRecord(e->ev[3], st)); e->timed_expand = true; }
  }
  if (b->digests_host) CUDA_TRY(cudaMemcpyAsync(b->digests_host, dig_dev, n_msgs * 32, cudaMemcpyDeviceToHost, st));
  if (b->checksums_host) CUDA_TRY(cudaMemcpyAsync(b->checksums_host, cks_dev, b->n_instances * 32, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaEventRecord(S->expand_done, st));
  S->used = true; S->last_stream = st;
  e->last_launches = launches;
  return H2SHA_OK;
}

int h2sha_export_instance(h2sha_engine_t* e, uint64_t instance, const void* gate, const void* lookup, const void* spread,
                          uint64_t* const* host_columns, uint32_t rows_per_column, void* stream) {
  if (!e || !host_columns) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  const Plan& P = e->plan;
  const LookupGeom G = lookup_geom(P);
  const uint32_t col_rows[3] = {P.gate_col_rows, P.lookup_col_rows, P.spread_rows};
  const uint32_t n_cols[3] = {P.n_gate_cols, P.n_lookup_cols, 2 * P.cfg.spread_cols};
  const void* bufs[3] = {gate, lookup, spread};
  const uint64_t inst_cells[3] = {e->dplan.gate_inst_cells, e->dplan.lookup_inst_cells, e->dplan.spread_inst_cells};
  for (int b = 0; b < 3; b++)
    if (col_rows[b] > rows_per_column && bufs[b]) {
      // only the assigned prefix of a column has to fit: the stride may exceed rows_per_column through alignment padding
      uint32_t used = (b == 0) ? 0 : (b == 1 ? G.max_range_used() : G.max_spread_used());
      if (b == 0)
        for (size_t c = 0; c < P.breaks.size(); c++) used = std::max(used, ((c + 1 < P.breaks.size()) ? P.breaks[c + 1] : P.n_gate) - P.breaks[c]);
      if (used > rows_per_column) return set_err(H2SHA_EINVAL, "rows_per_column is smaller than the assigned rows of a column");
    }
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t k = 0;
  for (int b = 0; b < 3; b++)
    for (uint32_t c = 0; c < n_cols[b]; c++, k++) {
      if (!bufs[b]) continue;
      uint64_t* dst = host_columns[k];
      if (!dst) return set_err(H2SHA_EINVAL, "null host column");
      const uint32_t rows = std::min(col_rows[b], rows_per_column);
      const uint8_t* src = (const uint8_t*)bufs[b] + ((instance * inst_cells[b] + (uint64_t)c * col_rows[b]) * 32);
      CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)rows * 32, cudaMemcpyDeviceToHost, st));
      if (rows < rows_per_column) memset(dst + (size_t)rows * 4, 0, (size_t)(rows_per_column - rows) * 32);
    }
  return H2SHA_OK;
}

int h2sha_zero_outputs(h2sha_engine_t* e, uint64_t n_inst, void* gate, void* lookup, void* spread, int only_unassigned, void* stream) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  void* bufs[3] = {gate, lookup, spread};
  uint64_t cells[3] = {e->dplan.gate_inst_cells, e->dplan.lookup_inst_cells, e->dplan.spread_inst_cells};
  for (int b = 0; b < 3; b++) {
    if (!bufs[b]) continue;
    if (!only_unassigned) { CUDA_TRY(cudaMemsetAsync(bufs[b], 0, n_inst * cells[b] * 32, st)); continue; }
    if (e->n_zero_ranges[b] == 0) continue;
    for (uint64_t i0 = 0; i0 < n_inst; i0 += 65535) {   // grid.y = instance: at most 65535 per launch
      const uint64_t ni = std::min<uint64_t>(65535, n_inst - i0);
      k_zero_ranges<<<dim3(64, (unsigned)ni), 256, 0, st>>>((uint4*)bufs[b] + i0 * cells[b] * 2, cells[b], ni, e->d_zero_ranges[b], e->n_zero_ranges[b]);
      CUDA_TRY(cudaGetLastError());
    }
  }
  return H2SHA_OK;
}

int h2sha_debug_mont_from_u64(h2sha_engine_t* e, const uint64_t* vals_dev, uint64_t* out_dev, uint64_t n, void* stream) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  CUDA_TRY(cudaSetDevice(e->device));
  if (n == 0) return H2SHA_OK;
  k_mont_debug<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vals_dev, out_dev, n);
  CUDA_TRY(cudaGetLastError());
  return H2SHA_OK;
}

int h2sha_debug_mont_from_u32(h2sha_engine_t* e, const uint64_t* vals_dev, uint64_t* out_dev, uint64_t n, void* stream) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  CUDA_TRY(cudaSetDevice(e->device));
  if (n == 0) return H2SHA_OK;
  k_mont_debug32<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vals_dev, out_dev, n);
  CUDA_TRY(cudaGetLastError());
  return H2SHA_OK;
}

int h2sha_debug_store_probe(h2sha_engine_t* e, void* buf_dev, uint64_t bytes, void* stream) {
  if (!e || !buf_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  CUDA_TRY(cudaSetDevice(e->device));
  if (bytes < 32) return H2SHA_OK;
  k_store_probe<<<(unsigned)(e->n_sms * 8), 256, 0, (cudaStream_t)stream>>>((uint32_t*)buf_dev, bytes / 32, (uint32_t)bytes);
  CUDA_TRY(cudaGetLastError());
  return H2SHA_OK;
}

int h2sha_debug_int_probe(h2sha_engine_t* e, uint32_t* scratch_dev, uint32_t iters, uint64_t* thread_instructions, void* stream) {
  if (!e || !scratch_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine");
  CUDA_TRY(cudaSetDevice(e->device));
  const unsigned ctas = (unsigned)e->n_sms * 8u;
  k_int_probe<<<ctas, 256, 0, (cudaStream_t)stream>>>(scratch_dev, iters, 0x9E3779B9u);
  CUDA_TRY(cudaGetLastError());
  if (thread_instructions) *thread_instructions = (uint64_t)ctas * 256u * iters * 16u;
  return H2SHA_OK;
}

int h2sha_last_launch_count(const h2sha_engine_t* e) { return e ? e->last_launches : 0; }

int h2sha_last_kernel_ms(h2sha_engine_t* e, float* trace_ms, float* expand_ms) {
  if (!e || !e->timed || !e->ev[0]) return set_err(H2SHA_EINVAL, "last batch was not run with time_kernels");
  CUDA_TRY(cudaEventSynchronize(e->timed_expand ? e->ev[3] : e->ev[1]));
  if (trace_ms) CUDA_TRY(cudaEventElapsedTime(trace_ms, e->ev[0], e->ev[1]));
  if (expand_ms) {
    *expand_ms = 0.f;   // a digests-only batch has no expansion step
    if (e->timed_expand) CUDA_TRY(cudaEventElapsedTime(expand_ms, e->ev[2], e->ev[3]));
  }
  return H2SHA_OK;
}

}  // extern "C"

#include "lookup_prework.cuh"
#include "batch_check.cuh"
#include "grand_product.cuh"
#include "lookup_product.cuh"
#include "permutation_product.cuh"
#include "export.cuh"

void h2sha_free_compact_state(h2sha_compact_state* s) { delete s; }
