// lookup_product.cuh -- the lookup argument's grand-product column z on the device (SURVEY.md §8f #4), the step after
// the permutation: PSE halo2_proofs plonk/lookup/prover.rs `Permuted::commit_product`, for one lookup of every instance.
// Included at the end of engine.cu, after lookup_prework.cuh (ensure_range_tab) and grand_product.cuh.  Which column a lookup
// reads and how many of its rows are assigned: select_lookup (lookup_geom.h).
//
//   u_i = (A[i] + beta)(S[i] + gamma),  v_i = (A'[i] + beta)(S'[i] + gamma),  i < U = usable_rows
//   z[0] = 1,  z[j+1] = z[j] * u_j / v_j                                      (U + 1 values)
// One chunk of U rows, every row a fraction: the kernels of grand_product.cuh with the row source below; the fill writes
// z[0 .. U-1], the fold z[U].
// Bound: integer multiply-adds (about 12 Montgomery products per row, 14 for a spread lookup; DESIGN.md §4b), not HBM: 224 B of traffic per row.
#pragma once

namespace {

// PI: theta, beta and gamma per instance (h2sha_lookup_product_per_instance), from s_chal; the table expression of a spread lookup
// is formed on the fly for rows below n_vals
template <bool PI>
struct LookupRows {
  const uint64_t* cells;        // the lookup's witness buffer (lookup or spread) at instance 0 of the launch
  uint64_t inst_cells;          // Fr per instance in that buffer
  uint64_t col_off;             // Fr offset of the looked-up column (range) / the dense column (spread) inside an instance
  uint64_t spread_off;          // spread lookups: Fr distance from a dense cell to its spread cell
  uint32_t used;                // assigned rows of that column; the rows above hold 0
  uint32_t is_spread;
  const uint64_t* a_p;          // [n][usable_rows] Fr: A', S'
  const uint64_t* s_p;
  const uint64_t* tab;          // [n_vals] Fr: the table expression in table-row order (padded rows hold 0)
  uint32_t n_vals, usable_rows;
  uint64_t theta[4], beta[4], gamma[4];   // Montgomery (shared challenges)
  const uint64_t* chal;         // PI: [n][3][4] at instance 0 of the launch

  __device__ __forceinline__ void setup(uint64_t inst) const {
    if constexpr (PI) load_chal(chal, inst);
  }
  __device__ __forceinline__ bool any(uint32_t, uint32_t, uint32_t) const { return true; }
  __device__ __forceinline__ bool terms(uint64_t inst, uint32_t, uint32_t i, uint64_t u[4], uint64_t v[4]) const {
    const uint64_t* theta = PI ? s_chal[0] : this->theta;
    const uint64_t* beta = PI ? s_chal[1] : this->beta;
    const uint64_t* gamma = PI ? s_chal[2] : this->gamma;
    uint64_t x[4] = {0, 0, 0, 0}, y[4] = {0, 0, 0, 0}, t[4];
    if (i < used) {
      const uint64_t* c = cells + (inst * inst_cells + col_off + i) * 4;
      load_cell(c, x);
      if (is_spread) {   // dense * theta + spread (halo2 `compress_expressions`)
        mont_mul_dev(theta, x, t);
        load_cell(c + spread_off * 4, y);
        fr_add_dev(t, y, x);
      }
    }
    fr_add_dev(x, beta, t);
    if (i < n_vals) {
      if (PI && is_spread) compressed_spread_row(theta, i, y);
      else load_cell(tab + (uint64_t)i * 4, y);
    } else {
      y[0] = y[1] = y[2] = y[3] = 0;
    }
    fr_add_dev(y, gamma, x);
    mont_mul_dev(t, x, u);
    const uint64_t row = inst * usable_rows + i;
    load_cell(a_p + row * 4, x);
    fr_add_dev(x, beta, t);
    load_cell(s_p + row * 4, y);
    fr_add_dev(y, gamma, x);
    mont_mul_dev(t, x, v);
    return true;
  }
};

}  // namespace

namespace {

// per_inst: theta_mont (may be null for a range lookup), beta_mont and gamma_mont are [n_instances][4] with rows checked by the
// caller, errors_dev is [n_instances]
int lookup_product_impl(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                        const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows, const uint64_t* theta_mont,
                        const uint64_t* beta_mont, const uint64_t* gamma_mont, bool per_inst, void* z_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !permuted_input_dev || !permuted_table_dev || !beta_mont || !gamma_mont || !z_dev) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  const LookupGeom G = lookup_geom(e->plan, usable_rows);
  const LookupSel L = select_lookup(G, lookup_idx);
  if (!L.valid) return set_err(H2SHA_EINVAL, "bad lookup index");
  const bool is_range = L.is_range;
  const void* cells = L.buffer(lookup, spread);
  if (!cells) return set_err(H2SHA_EINVAL, "null argument: the witness buffer this lookup reads");
  if (!is_range && !theta_mont) return set_err(H2SHA_EINVAL, "a spread lookup has two expressions: theta is needed to compress them");
  if (usable_rows < G.min_usable_rows()) return set_err(H2SHA_EINVAL, "usable_rows is smaller than an assigned column or a lookup table");
  if (!per_inst && (fr::geq_p(beta_mont) || fr::geq_p(gamma_mont) || (theta_mont && !is_range && fr::geq_p(theta_mont))))
    return set_err(H2SHA_EINVAL, "beta, gamma and theta must be reduced field elements");
  const void* bufs[] = {cells, permuted_input_dev, permuted_table_dev, z_dev};
  for (const void* b : bufs)
    if ((uintptr_t)b & 31u) return set_err(H2SHA_EINVAL, "Fr buffers must be 32-byte aligned");
  if (n_instances == 0) return H2SHA_OK;
  CUDA_TRY(cudaSetDevice(e->device));
  int rc;
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t n_vals = L.n_vals;
  GrandProduct Z{};
  Z.rows = usable_rows; Z.n_chunks = 1; Z.z_stride = usable_rows + 1;
  Z.tiles_per_chunk = (uint32_t)((usable_rows + (uint64_t)GP_TILE - 1) / GP_TILE);
  // workspace: [spread table (shared challenges)] [tile products of a chunk] [tile constants of a chunk]
  const uint64_t chunk = std::min<uint64_t>(std::min<uint64_t>(n_instances, 65535), (uint64_t)std::max(1, tune_value("lkchunk", 256)));
  const uint64_t tab_words = is_range || per_inst ? 0 : (uint64_t)n_vals * 4;
  const uint64_t need = (tab_words + chunk * Z.tiles_per_chunk * 12ull) * 8;
  if (need > e->lp_ws_bytes) {
    cudaFree(e->d_lp_ws); e->d_lp_ws = nullptr; e->lp_ws_bytes = 0;
    CUDA_TRY(cudaMalloc(&e->d_lp_ws, need));
    e->lp_ws_bytes = need;
  }
  Z.tiles = e->d_lp_ws + tab_words;
  Z.consts = Z.tiles + chunk * Z.tiles_per_chunk * 8;
  Z.err_stride = per_inst ? 1u : 0u;
  const uint64_t* tab = nullptr;
  if (is_range) {
    if ((rc = ensure_range_tab(e, st))) return rc;
    tab = reinterpret_cast<const uint64_t*>(e->d_range_tab);
  } else if (!per_inst) {
    U256 th_m; memcpy(th_m.l, theta_mont, 32);
    const std::vector<U256> t = compressed_spread_table(th_m, G.limb_bits);
    CUDA_TRY(cudaMemcpyAsync(e->d_lp_ws, t.data(), t.size() * 32, cudaMemcpyHostToDevice, st));   // pageable: staged before return
    tab = e->d_lp_ws;
  }
  if (per_inst && (rc = stage_challenges(e, n_instances, is_range ? nullptr : theta_mont, beta_mont, gamma_mont, st))) return rc;
  auto run = [&](auto& A) {
    A.n_vals = n_vals; A.usable_rows = usable_rows; A.tab = tab;
    A.inst_cells = L.inst_cells; A.col_off = L.col_off; A.spread_off = L.spread_off; A.used = L.used;
    A.is_spread = is_range ? 0u : 1u;
    const uint64_t* cells0 = (const uint64_t*)cells;
    for (uint64_t i0 = 0; i0 < n_instances; i0 += chunk) {
      const unsigned ni = (unsigned)std::min<uint64_t>(chunk, n_instances - i0);
      A.cells = cells0 + i0 * A.inst_cells * 4;
      A.a_p = (const uint64_t*)permuted_input_dev + i0 * usable_rows * 4;
      A.s_p = (const uint64_t*)permuted_table_dev + i0 * usable_rows * 4;
      if (per_inst) A.chal = e->d_chal + i0 * 12;
      Z.z = (uint64_t*)z_dev + i0 * (usable_rows + 1ull) * 4;
      Z.errors = errors_dev ? errors_dev + (per_inst ? i0 : 0) : nullptr;
      if (int r = launch_product(Z, A, ni, st)) return r;
    }
    return (int)H2SHA_OK;
  };
  if (per_inst) {
    LookupRows<true> A{};
    return run(A);
  }
  LookupRows<false> A{};
  memcpy(A.beta, beta_mont, 32); memcpy(A.gamma, gamma_mont, 32);
  if (!is_range) memcpy(A.theta, theta_mont, 32);
  return run(A);
}

}  // namespace

extern "C" {

int h2sha_lookup_product(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                         const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows, const uint64_t* theta_mont,
                         const uint64_t* beta_mont, const uint64_t* gamma_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
  return lookup_product_impl(e, n_instances, lookup_idx, lookup, spread, permuted_input_dev, permuted_table_dev, usable_rows, theta_mont, beta_mont,
                             gamma_mont, false, z_dev, errors_dev, stream);
}

int h2sha_lookup_product_per_instance(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                                      const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows,
                                      const uint64_t* thetas_mont, const uint64_t* betas_mont, const uint64_t* gammas_mont,
                                      void* z_dev, uint32_t* errors_dev, void* stream) {
  if (!e || !betas_mont || !gammas_mont) return set_err(H2SHA_EINVAL, "null argument");
  const LookupSel L = select_lookup(lookup_geom(e->plan), lookup_idx);
  const bool is_spread = L.valid && !L.is_range;
  if (is_spread && !thetas_mont) return set_err(H2SHA_EINVAL, "a spread lookup has two expressions: thetas_mont is needed to compress them");
  int rc;
  if ((rc = check_challenge_rows(betas_mont, n_instances, "betas_mont")) || (rc = check_challenge_rows(gammas_mont, n_instances, "gammas_mont")) ||
      (is_spread && (rc = check_challenge_rows(thetas_mont, n_instances, "thetas_mont"))))
    return rc;
  return lookup_product_impl(e, n_instances, lookup_idx, lookup, spread, permuted_input_dev, permuted_table_dev, usable_rows,
                             is_spread ? thetas_mont : nullptr, betas_mont, gammas_mont, true, z_dev, errors_dev, stream);
}

}  // extern "C"
