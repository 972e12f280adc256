// permutation_product.cuh -- the permutation argument's product columns on the device (PSE halo2_proofs
// plonk/permutation/prover.rs `Argument::commit`, without the blinding rows) for the chip's copy constraints, for every instance
// of a batch.  Included at the end of engine.cu after grand_product.cuh.
//
// Chunk h of the C listed columns covers [h*m, min(C, (h+1)*m)); chunks chain (z_h[0] = z_{h-1}[U]), so the columns of all chunks
// form ONE sequence of fractions over (chunk, row).  A cell whose sigma is the identity contributes exactly 1 to its row's
// fraction; only *moved* cells (sigma != id) matter, and they are static per (configuration, column list, usable_rows):
// 81 862 of ~0.9 M usable cells for config 2, 326 255 for the TestCircuit with its instance column.  So:
//   plan (host, once per desc)  permutation.cc replays the copies; the moved cells, sorted by (chunk, row), with their source
//                               (buffer and Fr offset in an instance, fixed constant, digest byte), identity delta^j w^r and sigma;
//                               per chunk a row index ptr[h][0 .. U+1] into that list
//   k_perm_prep                 per call: a = beta id + gamma, b = beta sigma + gamma per moved cell (shared by all instances);
//                               with per-instance challenges (h2sha_permutation_product_per_instance) a and b are formed in the row
//                               source instead, from the resident identity and sigma and the CTA's beta_i, gamma_i
//   grand_product.cuh           with the row source PermRows: u_i = prod (p + a), v_i = prod (p + b) over the moved cells of a row;
//                               rows run 0 .. U in every chunk (row U has no moved cell), so the fill writes z[0 .. U] of every
//                               chunk, and the closing value the fold checks against 1 is the last chunk's z[U]
// Bound: the integer arithmetic of the rows that hold moved cells, not HBM (z leaves at 0.02-0.04 of the store probe; DESIGN.md §4e).
// Zero terms: a zero denominator at a moved cell gives the row the fraction 0 (u, v) := (0, 1), like ff's batch_invert.  The
// one departure from halo2: a zero term p + beta delta^j w^i + gamma at an UNMOVED cell (probability ~2^-230 over beta, gamma) is
// taken as 1; halo2 would zero that row's fraction.
#pragma once

namespace {

enum : uint64_t { PS_GATE = 0, PS_LOOKUP = 1, PS_SPREAD = 2, PS_FIXED = 3, PS_BYTE = 4, PS_ZERO = 5 };   // source kind (bits 60..63)
constexpr uint64_t PS_OFF_MASK = (1ull << 60) - 1;

// the moved cells of a batch as a row source of grand_product.cuh; PI: beta and gamma per instance, from s_chal
template <bool PI>
struct PermRows {
  const uint64_t* gate;         // batch buffers at instance 0 of the launch
  const uint64_t* lookup;
  const uint64_t* spread;
  uint64_t gate_inst, lookup_inst, spread_inst;   // Fr per instance in each buffer
  const uint8_t* digests;       // [n][digest_bytes] at instance 0 of the launch
  uint32_t digest_bytes;        // 32 * n_digests
  const uint64_t* fixed;        // [n_fixed][4] Montgomery
  const uint64_t* bytes;        // [256][4] Montgomery of 0 .. 255
  const uint64_t* src;          // [n_moved] (kind << 60) | offset
  const uint64_t* ab;           // [n_moved][2][4]: beta id + gamma, beta sigma + gamma; PI: id, sigma
  const uint32_t* ptr;          // [n_chunks][U + 2]: first moved cell of each row
  uint32_t usable_rows;
  const uint64_t* chal;         // PI: [n][3][4] at instance 0 of the launch

  __device__ __forceinline__ void setup(uint64_t inst) const {
    if constexpr (PI) load_chal(chal, inst);
  }
  __device__ __forceinline__ bool any(uint32_t h, uint32_t i0, uint32_t i1) const;
  __device__ bool terms(uint64_t inst, uint32_t h, uint32_t i, uint64_t u[4], uint64_t v[4]) const;
};

struct PermChallenges {
  uint64_t beta[4], gamma[4];   // Montgomery
};

__global__ void k_perm_prep(const uint64_t* __restrict__ idsig, uint64_t* __restrict__ ab, uint32_t n, const PermChallenges ch) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  uint64_t x[4], t[4];
  for (int q = 0; q < 2; q++) {
    load_cell(idsig + ((uint64_t)k * 2 + q) * 4, x);
    mont_mul_dev(ch.beta, x, t);
    fr_add_dev(t, ch.gamma, x);
    store_fr(ab + ((uint64_t)k * 2 + q) * 4, x);
  }
}

template <class Rows>
__device__ __forceinline__ void perm_value(const Rows& A, uint64_t inst, uint64_t s, uint64_t p[4]) {
  const uint64_t off = s & PS_OFF_MASK;
  switch (s >> 60) {
    case PS_GATE: load_cell(A.gate + (inst * A.gate_inst + off) * 4, p); break;
    case PS_LOOKUP: load_cell(A.lookup + (inst * A.lookup_inst + off) * 4, p); break;
    case PS_SPREAD: load_cell(A.spread + (inst * A.spread_inst + off) * 4, p); break;
    case PS_FIXED: load_cell(A.fixed + off * 4, p); break;
    case PS_BYTE: load_cell(A.bytes + (uint64_t)A.digests[inst * A.digest_bytes + off] * 4, p); break;
    default: p[0] = p[1] = p[2] = p[3] = 0;
  }
}

// a moved cell in rows [i0, i1) of chunk h (ptr ends at index U + 1)
template <bool PI>
__device__ __forceinline__ bool PermRows<PI>::any(uint32_t h, uint32_t i0, uint32_t i1) const {
  const uint32_t* pr = ptr + (uint64_t)h * (usable_rows + 2);
  return pr[min(i0, usable_rows + 1)] != pr[min(i1, usable_rows + 1)];
}

// u, v of a row from its moved cells [k0, k1); false for a row without any
template <bool PI>
__device__ bool PermRows<PI>::terms(uint64_t inst, uint32_t h, uint32_t i, uint64_t u[4], uint64_t v[4]) const {
  const uint32_t* pr = ptr + (uint64_t)h * (usable_rows + 2);
  const uint32_t k0 = pr[i], k1 = pr[i + 1];
  if (k0 == k1) return false;
  uint64_t p[4], t[4];
  for (uint32_t k = k0; k < k1; k++) {
    perm_value(*this, inst, src[k], p);
    if constexpr (PI) {   // p + beta x + gamma for x = id, sigma: two more products per moved cell than the shared path
      uint64_t x[4], a[4];
#pragma unroll
      for (int q = 0; q < 2; q++) {
        load_cell(ab + (uint64_t)k * 8 + 4 * q, x);
        mont_mul_dev(s_chal[1], x, t);
        fr_add_dev(t, s_chal[2], a);
        fr_add_dev(p, a, x);
        uint64_t* acc = q ? v : u;
        if (k == k0) fr_copy(x, acc);
        else fr_mul_into(acc, x);
      }
    } else if (k == k0) {
      fr_add_dev(p, ab + (uint64_t)k * 8, u);
      fr_add_dev(p, ab + (uint64_t)k * 8 + 4, v);
    } else {
      fr_add_dev(p, ab + (uint64_t)k * 8, t);
      fr_mul_into(u, t);
      fr_add_dev(p, ab + (uint64_t)k * 8 + 4, t);
      fr_mul_into(v, t);
    }
  }
  return true;
}

}  // namespace

// The moved cells of one (desc, usable_rows), resident on the device
struct h2sha_perm_state {
  std::vector<uint32_t> key;    // desc fields + column list + usable_rows the state was planned for
  uint32_t n_moved = 0, n_chunks = 0, usable_rows = 0;
  uint64_t* d_src = nullptr;    // [n_moved]
  uint64_t* d_idsig = nullptr;  // [n_moved][2][4] Montgomery identity, sigma
  uint64_t* d_ab = nullptr;     // [n_moved][2][4] per call
  uint32_t* d_ptr = nullptr;    // [n_chunks][U + 2]
  uint64_t* d_fixed = nullptr;  // [n_fixed][4] Montgomery
  uint64_t* d_bytes = nullptr;  // [256][4] Montgomery
  uint64_t* d_ws = nullptr;     // tile products and tile constants
  uint64_t ws_bytes = 0;
  ~h2sha_perm_state() {
    cudaFree(d_src); cudaFree(d_idsig); cudaFree(d_ab); cudaFree(d_ptr); cudaFree(d_fixed); cudaFree(d_bytes); cudaFree(d_ws);
  }
};

namespace {

std::vector<uint32_t> perm_key(const h2sha_perm_desc_t& d, const PermColumns& C) {
  std::vector<uint32_t> k = {C.n_cols, C.num_fixed, C.m, C.bind, C.k, C.usable_rows};
  k.insert(k.end(), d.columns, d.columns + 2 * (size_t)d.n_columns);
  return k;
}

// plans the moved cells of `C` and uploads them (synchronous: once per desc)
int ensure_perm_state(h2sha_engine* e, const h2sha_perm_desc_t& d, const PermColumns& C) {
  std::vector<uint32_t> key = perm_key(d, C);
  if (e->perm && e->perm->key == key) return H2SHA_OK;
  if (e->perm) {   // kernels of an earlier call may still read the resident cells
    CUDA_TRY(cudaDeviceSynchronize());
    delete e->perm; e->perm = nullptr;
  }
  const Plan& P = e->plan;
  std::vector<uint32_t> mapping;
  std::string err;
  if (!replay_permutation(P, C, &mapping, &err)) return set_err(H2SHA_EINVAL, err);
  const uint32_t U = C.usable_rows, nc = P.cfg.spread_cols;
  // identity and sigma values: delta^c w^r
  std::vector<U256> dpow(C.n_cols), wpow(U);
  const U256 one = fr::to_mont(fr::from_u64(1)), delta = perm_delta_mont(), omega = perm_omega_mont(C.k);
  dpow[0] = one; wpow[0] = one;
  for (uint32_t c = 1; c < C.n_cols; c++) dpow[c] = fr::mont_mul(dpow[c - 1], delta);
  for (uint32_t r = 1; r < U; r++) wpow[r] = fr::mont_mul(wpow[r - 1], omega);
  std::vector<uint64_t> src;
  std::vector<U256> idsig;
  std::vector<uint32_t> ptr((size_t)C.n_chunks * (U + 2));
  for (uint32_t h = 0; h < C.n_chunks; h++) {
    const uint32_t c0 = h * C.m, c1 = std::min(C.n_cols, c0 + C.m);
    uint32_t* pr = &ptr[(size_t)h * (U + 2)];
    for (uint32_t r = 0; r < U; r++) {
      pr[r] = (uint32_t)src.size();
      for (uint32_t c = c0; c < c1; c++) {
        const uint32_t id = c * U + r, to = mapping[id];
        if (to == id) continue;
        const uint32_t kind = C.kind[c], idx = C.index[c];
        uint64_t s = PS_ZERO << 60;
        if (kind == H2SHA_COL_GATE) s = (PS_GATE << 60) | ((uint64_t)idx * P.gate_col_rows + r);
        else if (kind == H2SHA_COL_LOOKUP) s = (PS_LOOKUP << 60) | ((uint64_t)idx * P.lookup_col_rows + r);
        else if (kind == H2SHA_COL_DENSE) s = (PS_SPREAD << 60) | ((uint64_t)idx * P.spread_rows + r);
        else if (kind == H2SHA_COL_SPREAD) s = (PS_SPREAD << 60) | ((uint64_t)(nc + idx) * P.spread_rows + r);
        else if (kind == H2SHA_COL_FIXED) {
          const uint64_t k = (uint64_t)r * C.num_fixed + idx;   // Context::assign_fixed: round-robin
          if (k < P.fixed_consts.size()) s = (PS_FIXED << 60) | k;
        } else if (kind == H2SHA_COL_INSTANCE) {
          if (r < 32 * P.digests.size()) s = (PS_BYTE << 60) | r;
        }
        src.push_back(s);
        idsig.push_back(fr::mont_mul(dpow[c], wpow[r]));
        idsig.push_back(fr::mont_mul(dpow[to / U], wpow[to % U]));
      }
    }
    pr[U] = pr[U + 1] = (uint32_t)src.size();
  }
  std::vector<U256> fixed_m(std::max<size_t>(P.fixed_consts.size(), 1), U256{{0, 0, 0, 0}}), bytes_m(256);
  for (size_t k = 0; k < P.fixed_consts.size(); k++) fixed_m[k] = fr::to_mont(P.fixed_consts[k]);
  bytes_m[0] = U256{{0, 0, 0, 0}};
  for (uint32_t b = 1; b < 256; b++) bytes_m[b] = fr::add(bytes_m[b - 1], one);
  h2sha_perm_state* S = new h2sha_perm_state();
  e->perm = S;   // freed with the engine (or replaced) also when an upload below fails
  S->n_moved = (uint32_t)src.size(); S->n_chunks = C.n_chunks; S->usable_rows = U;
  const size_t nm = std::max<size_t>(src.size(), 1);
  CUDA_TRY(cudaMalloc(&S->d_src, nm * 8));
  CUDA_TRY(cudaMalloc(&S->d_idsig, nm * 64));
  CUDA_TRY(cudaMalloc(&S->d_ab, nm * 64));
  CUDA_TRY(cudaMalloc(&S->d_ptr, ptr.size() * 4));
  CUDA_TRY(cudaMalloc(&S->d_fixed, fixed_m.size() * 32));
  CUDA_TRY(cudaMalloc(&S->d_bytes, 256 * 32));
  if (!src.empty()) {
    CUDA_TRY(cudaMemcpy(S->d_src, src.data(), src.size() * 8, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(S->d_idsig, idsig.data(), idsig.size() * 32, cudaMemcpyHostToDevice));
  }
  CUDA_TRY(cudaMemcpy(S->d_ptr, ptr.data(), ptr.size() * 4, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(S->d_fixed, fixed_m.data(), fixed_m.size() * 32, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(S->d_bytes, bytes_m.data(), 256 * 32, cudaMemcpyHostToDevice));
  S->key = std::move(key);   // valid only once everything is resident
  return H2SHA_OK;
}

}  // namespace

void h2sha_free_perm_state(h2sha_perm_state* s) { delete s; }

extern "C" {

int h2sha_get_permutation(h2sha_engine_t* e, const h2sha_perm_desc_t* desc, uint32_t usable_rows, uint32_t* mapping) {
  if (!e || !desc) return set_err(H2SHA_EINVAL, "null argument");
  PermColumns C;
  std::string err;
  if (!perm_columns(e->plan, *desc, usable_rows, &C, &err)) return set_err(H2SHA_EINVAL, err);
  std::vector<uint32_t> m;
  if (!replay_permutation(e->plan, C, &m, &err)) return set_err(H2SHA_EINVAL, err);
  if (mapping)
    for (size_t i = 0; i < m.size(); i++) { mapping[2 * i] = m[i] / usable_rows; mapping[2 * i + 1] = m[i] % usable_rows; }
  return H2SHA_OK;
}

}  // extern "C"

namespace {

// per_inst: beta_mont and gamma_mont are [n_instances][4] with rows checked by the caller, errors_dev is [n_instances]
int permutation_product_impl(h2sha_engine_t* e, uint64_t n_instances, const h2sha_perm_desc_t* desc, uint32_t usable_rows,
                             const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                             const uint64_t* beta_mont, const uint64_t* gamma_mont, bool per_inst, void* z_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !desc || !beta_mont || !gamma_mont || !z_dev) return set_err(H2SHA_EINVAL, "null argument");
  const Plan& P = e->plan;
  PermColumns C;
  std::string err;
  if (!perm_columns(P, *desc, usable_rows, &C, &err)) return set_err(H2SHA_EINVAL, err);
  if (!per_inst && (fr::geq_p(beta_mont) || fr::geq_p(gamma_mont))) return set_err(H2SHA_EINVAL, "beta and gamma must be reduced field elements");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  bool reads[3] = {false, false, false};
  for (uint32_t k : C.kind) {
    if (k == H2SHA_COL_GATE) reads[0] = true;
    if (k == H2SHA_COL_LOOKUP) reads[1] = true;
    if (k == H2SHA_COL_DENSE || k == H2SHA_COL_SPREAD) reads[2] = true;
  }
  const void* bufs[3] = {gate, lookup, spread};
  for (int b = 0; b < 3; b++)
    if (reads[b] && !bufs[b]) return set_err(H2SHA_EINVAL, "null argument: a witness buffer a listed column reads");
  if (C.bind && !digests_dev) return set_err(H2SHA_EINVAL, "bind_output_bytes: digests_dev is needed for the instance column");
  for (const void* b : {gate, lookup, spread, (const void*)z_dev})
    if ((uintptr_t)b & 31u) return set_err(H2SHA_EINVAL, "Fr buffers must be 32-byte aligned");
  if (n_instances == 0) return H2SHA_OK;
  CUDA_TRY(cudaSetDevice(e->device));
  int rc = ensure_perm_state(e, *desc, C);
  if (rc) return rc;
  h2sha_perm_state* S = e->perm;
  cudaStream_t st = (cudaStream_t)stream;
  GrandProduct Z{};
  Z.rows = usable_rows + 1; Z.n_chunks = C.n_chunks; Z.z_stride = usable_rows + 1;
  Z.tiles_per_chunk = (uint32_t)((usable_rows + 1ull + GP_TILE - 1) / GP_TILE);
  const uint32_t n_tiles = Z.n_chunks * Z.tiles_per_chunk;
  if (per_inst) {
    if ((rc = stage_challenges(e, n_instances, nullptr, beta_mont, gamma_mont, st))) return rc;
  } else if (S->n_moved) {   // per call: a, b of every moved cell
    PermChallenges ch;
    memcpy(ch.beta, beta_mont, 32); memcpy(ch.gamma, gamma_mont, 32);
    k_perm_prep<<<(S->n_moved + 255) / 256, 256, 0, st>>>(S->d_idsig, S->d_ab, S->n_moved, ch);
    CUDA_TRY(cudaGetLastError());
  }
  // workspace: [tile products of a chunk of instances] [tile constants]
  const uint64_t chunk = std::min<uint64_t>(std::min<uint64_t>(n_instances, 65535), (uint64_t)std::max(1, tune_value("pmchunk", 256)));
  const uint64_t need = chunk * n_tiles * 12ull * 8;
  if (need > S->ws_bytes) {
    cudaFree(S->d_ws); S->d_ws = nullptr; S->ws_bytes = 0;
    CUDA_TRY(cudaMalloc(&S->d_ws, need));
    S->ws_bytes = need;
  }
  Z.tiles = S->d_ws;
  Z.consts = S->d_ws + chunk * n_tiles * 8;
  Z.err_stride = per_inst ? 1u : 0u;
  auto run = [&](auto& A) {
    A.usable_rows = usable_rows;
    A.gate_inst = e->dplan.gate_inst_cells; A.lookup_inst = e->dplan.lookup_inst_cells; A.spread_inst = e->dplan.spread_inst_cells;
    A.digest_bytes = 32u * (uint32_t)P.digests.size();
    A.fixed = S->d_fixed; A.bytes = S->d_bytes; A.src = S->d_src; A.ptr = S->d_ptr;
    A.ab = per_inst ? S->d_idsig : S->d_ab;
    for (uint64_t i0 = 0; i0 < n_instances; i0 += chunk) {
      const unsigned ni = (unsigned)std::min<uint64_t>(chunk, n_instances - i0);
      A.gate = gate ? (const uint64_t*)gate + i0 * A.gate_inst * 4 : nullptr;
      A.lookup = lookup ? (const uint64_t*)lookup + i0 * A.lookup_inst * 4 : nullptr;
      A.spread = spread ? (const uint64_t*)spread + i0 * A.spread_inst * 4 : nullptr;
      A.digests = digests_dev ? digests_dev + i0 * A.digest_bytes : nullptr;
      if (per_inst) A.chal = e->d_chal + i0 * 12;
      Z.z = (uint64_t*)z_dev + i0 * Z.n_chunks * (usable_rows + 1ull) * 4;
      Z.errors = errors_dev ? errors_dev + (per_inst ? i0 : 0) : nullptr;
      if (int r = launch_product(Z, A, ni, st)) return r;
    }
    return (int)H2SHA_OK;
  };
  if (per_inst) {
    PermRows<true> A{};
    return run(A);
  }
  PermRows<false> A{};
  return run(A);
}

}  // namespace

extern "C" {

int h2sha_permutation_product(h2sha_engine_t* e, uint64_t n_instances, const h2sha_perm_desc_t* desc, uint32_t usable_rows,
                              const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                              const uint64_t* beta_mont, const uint64_t* gamma_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
  return permutation_product_impl(e, n_instances, desc, usable_rows, gate, lookup, spread, digests_dev, beta_mont, gamma_mont, false, z_dev,
                                  errors_dev, stream);
}

int h2sha_permutation_product_per_instance(h2sha_engine_t* e, uint64_t n_instances, const h2sha_perm_desc_t* desc, uint32_t usable_rows,
                                           const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                                           const uint64_t* betas_mont, const uint64_t* gammas_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !betas_mont || !gammas_mont) return set_err(H2SHA_EINVAL, "null argument");
  int rc;
  if ((rc = check_challenge_rows(betas_mont, n_instances, "betas_mont")) || (rc = check_challenge_rows(gammas_mont, n_instances, "gammas_mont"))) return rc;
  return permutation_product_impl(e, n_instances, desc, usable_rows, gate, lookup, spread, digests_dev, betas_mont, gammas_mont, true, z_dev,
                                  errors_dev, stream);
}

}  // extern "C"

