// host_api.hpp -- header-only C++ mirror of the reference's chip API (halo2-dynamic-sha256 src/lib.rs:38-369) over the
// C-ABI (include/h2sha_b200.h).  Same names, argument meaning and error behaviour: a panic of the reference
// (lib.rs:89-90) surfaces as h2sha::ReferencePanic, every other failure as h2sha::EngineError.
#pragma once
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/h2sha_b200.h"

namespace h2sha {

struct EngineError : std::runtime_error {
  int code;
  EngineError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
struct ReferencePanic : EngineError {
  using EngineError::EngineError;
};

struct AssignedHashResult {  // lib.rs:31-36, as gate-stream indices
  uint32_t input_len;
  std::vector<uint32_t> input_bytes, output_bytes;
};

class Sha256DynamicConfig {
 public:
  std::vector<uint32_t> max_variable_byte_sizes;  // lib.rs:40
  size_t cur_hash_idx = 0;                        // lib.rs:43

  // lib.rs:49-56 (+ max_rows / lookup_bits of the RangeConfig, lib.rs:409-418)
  static Sha256DynamicConfig configure(std::vector<uint32_t> sizes, uint32_t max_rows, uint32_t lookup_bits, uint32_t num_bits_lookup,
                                       uint32_t num_advice_columns, bool is_input_range_check, int device = 0, bool build_shape = false) {
    Sha256DynamicConfig c;
    c.max_variable_byte_sizes = std::move(sizes);
    h2sha_config_t cfg{};
    cfg.n_digests = (uint32_t)c.max_variable_byte_sizes.size();
    cfg.max_variable_byte_sizes = c.max_variable_byte_sizes.data();
    cfg.max_rows = max_rows; cfg.lookup_bits = lookup_bits; cfg.num_bits_lookup = num_bits_lookup;
    cfg.num_advice_columns = num_advice_columns; cfg.is_input_range_check = is_input_range_check;
    cfg.device = device; cfg.build_shape = build_shape;
    check(h2sha_create(&cfg, &c.engine_));
    check(h2sha_get_layout(c.engine_, &c.layout_));
    return c;
  }
  Sha256DynamicConfig(Sha256DynamicConfig&& o) noexcept { *this = std::move(o); }
  Sha256DynamicConfig& operator=(Sha256DynamicConfig&& o) noexcept {
    std::swap(engine_, o.engine_); std::swap(layout_, o.layout_);
    max_variable_byte_sizes = std::move(o.max_variable_byte_sizes); cur_hash_idx = o.cur_hash_idx;
    return *this;
  }
  ~Sha256DynamicConfig() { if (engine_) h2sha_destroy(engine_); }

  const h2sha_layout_t& layout() const { return layout_; }

  // digest (lib.rs:71-76) for a batch; see h2sha_batch_t for the buffers
  void digest_batch(const h2sha_batch_t& batch) { check(h2sha_digest_batch(engine_, &batch)); }

  // AssignedHashResult of the next digest call; advances cur_hash_idx like lib.rs:347
  AssignedHashResult handles() {
    AssignedHashResult r;
    r.input_bytes.resize(max_variable_byte_sizes.at(cur_hash_idx));
    r.output_bytes.resize(32);
    check(h2sha_get_handles(engine_, (uint32_t)cur_hash_idx, &r.input_len, r.input_bytes.data(), r.output_bytes.data()));
    cur_hash_idx++;
    return r;
  }
  std::vector<uint32_t> breaks() const {
    std::vector<uint32_t> b(layout_.n_gate_cols);
    check(h2sha_get_breaks(engine_, b.data()));
    return b;
  }
  // ---- lookup-argument pre-work on the witness in HBM (halo2 lookup prover `permute_expression_pair`) ----
  h2sha_lookup_info_t lookup_info() const {
    h2sha_lookup_info_t li{};
    check(h2sha_get_lookup_info(engine_, &li));
    return li;
  }
  // table-row multiplicities of every lookup (spread.rs:53-62; range lookup of lib.rs:409-418,469); all pointers are device memory
  void lookup_multiplicities(uint64_t n_instances, const void* lookup, const void* spread, uint32_t usable_rows, uint32_t* mult_dev,
                             uint32_t* not_in_table_dev, void* stream) {
    check(h2sha_lookup_multiplicities(engine_, n_instances, lookup, spread, usable_rows, mult_dev, not_in_table_dev, stream));
  }
  // permuted (A', S') columns of one lookup for every instance; theta_mont only for spread lookups
  void permute_lookup(uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows, const uint64_t* theta_mont,
                      void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
    check(h2sha_permute_lookup(engine_, n_instances, lookup_idx, mult_dev, usable_rows, theta_mont, permuted_input_dev, permuted_table_dev,
                               errors_dev, stream));
  }
  // grand-product column z [n_instances][usable_rows + 1] of one lookup (halo2 `commit_product`); beta / gamma / theta on the host
  void lookup_product(uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread, const void* permuted_input_dev,
                      const void* permuted_table_dev, uint32_t usable_rows, const uint64_t* theta_mont, const uint64_t* beta_mont,
                      const uint64_t* gamma_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
    check(h2sha_lookup_product(engine_, n_instances, lookup_idx, lookup, spread, permuted_input_dev, permuted_table_dev, usable_rows, theta_mont,
                               beta_mont, gamma_mont, z_dev, errors_dev, stream));
  }
  // ---- permutation argument (copy constraints; halo2 plonk/permutation) ----
  // keygen Assembly mapping [desc.n_columns][usable_rows][2] (column position, row); works on a plan-only engine with build_shape
  std::vector<uint32_t> permutation_mapping(const h2sha_perm_desc_t& desc, uint32_t usable_rows) const {
    std::vector<uint32_t> m((size_t)desc.n_columns * usable_rows * 2);
    check(h2sha_get_permutation(engine_, &desc, usable_rows, m.data()));
    return m;
  }
  // product columns z [n_instances][n_chunks][usable_rows + 1] (halo2 `permutation::prover` commit); beta / gamma on the host
  void permutation_product(uint64_t n_instances, const h2sha_perm_desc_t& desc, uint32_t usable_rows, const void* gate, const void* lookup,
                           const void* spread, const uint8_t* digests_dev, const uint64_t* beta_mont, const uint64_t* gamma_mont, void* z_dev,
                           uint32_t* errors_dev, void* stream) {
    check(h2sha_permutation_product(engine_, n_instances, &desc, usable_rows, gate, lookup, spread, digests_dev, beta_mont, gamma_mont, z_dev,
                                    errors_dev, stream));
  }
  // ---- per-instance challenges (independent proofs): challenge arrays [n_instances][4] on the host, errors_dev [n_instances] ----
  void permute_lookup_per_instance(uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows,
                                   const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream) {
    check(h2sha_permute_lookup_per_instance(engine_, n_instances, lookup_idx, mult_dev, usable_rows, thetas_mont, permuted_input_dev,
                                            permuted_table_dev, errors_dev, stream));
  }
  void permute_lookup_from_raw_per_instance(uint64_t first_instance, uint64_t n_instances, uint32_t lookup_idx, uint32_t usable_rows,
                                            const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev,
                                            void* stream) {
    check(h2sha_permute_lookup_from_raw_per_instance(engine_, first_instance, n_instances, lookup_idx, usable_rows, thetas_mont, permuted_input_dev,
                                                     permuted_table_dev, errors_dev, stream));
  }
  void lookup_product_per_instance(uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread, const void* permuted_input_dev,
                                   const void* permuted_table_dev, uint32_t usable_rows, const uint64_t* thetas_mont, const uint64_t* betas_mont,
                                   const uint64_t* gammas_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
    check(h2sha_lookup_product_per_instance(engine_, n_instances, lookup_idx, lookup, spread, permuted_input_dev, permuted_table_dev, usable_rows,
                                            thetas_mont, betas_mont, gammas_mont, z_dev, errors_dev, stream));
  }
  void permutation_product_per_instance(uint64_t n_instances, const h2sha_perm_desc_t& desc, uint32_t usable_rows, const void* gate,
                                        const void* lookup, const void* spread, const uint8_t* digests_dev, const uint64_t* betas_mont,
                                        const uint64_t* gammas_mont, void* z_dev, uint32_t* errors_dev, void* stream) {
    check(h2sha_permutation_product_per_instance(engine_, n_instances, &desc, usable_rows, gate, lookup, spread, digests_dev, betas_mont, gammas_mont,
                                                 z_dev, errors_dev, stream));
  }
  // MockProver-style check of every instance of a batch on the device (lib.rs:525-526): violations[5] = gates, copies,
  // range lookups, spread lookups, digest bytes
  void check_batch(uint64_t n_instances, const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                   uint64_t violations[5], void* stream) {
    check(h2sha_check_batch(engine_, n_instances, gate, lookup, spread, digests_dev, violations, stream));
  }
  // the same check per instance, asynchronous: counts_dev / first_dev [n_instances][5] u32 (first_dev may be null); see the header
  void check_batch_per_instance(uint64_t n_instances, const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                                uint32_t* counts_dev, uint32_t* first_dev, void* stream) {
    check(h2sha_check_batch_per_instance(engine_, n_instances, gate, lookup, spread, digests_dev, counts_dev, first_dev, stream));
  }
  // the cells a check item reads (host only)
  h2sha_check_site_t check_site(uint32_t check_class, uint32_t item) {
    h2sha_check_site_t s{};
    check(h2sha_check_site(engine_, check_class, item, &s));
    return s;
  }
  h2sha_engine_t* raw() const { return engine_; }

 private:
  Sha256DynamicConfig() = default;
  static void check(int rc) {
    if (rc == H2SHA_OK) return;
    if (rc == H2SHA_EPANIC) throw ReferencePanic(rc, h2sha_last_error());
    throw EngineError(rc, h2sha_last_error());
  }
  h2sha_engine_t* engine_ = nullptr;
  h2sha_layout_t layout_{};
};

}  // namespace h2sha
