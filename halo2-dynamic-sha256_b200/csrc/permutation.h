// permutation.h -- keygen half of the permutation argument (copy constraints): the chip's copies replayed through halo2's
// `permutation::keygen::Assembly` (permutation.cc).  Used by h2sha_get_permutation and by the device product
// (permutation_product.cuh), which needs the cells whose sigma is not the identity.
#pragma once
#include <string>
#include <vector>

#include "../../include/h2sha_b200.h"
#include "planner.h"

namespace h2sha {

// The validated column list of an h2sha_perm_desc_t.
struct PermColumns {
  uint32_t n_cols = 0, usable_rows = 0, m = 0, n_chunks = 0, k = 0, num_fixed = 1, bind = 0;
  std::vector<uint32_t> kind, index;   // per column position
  std::vector<int32_t> pos[7];         // [kind][index] -> column position, -1 when not listed
};

// Checks `d` against the plan (H2SHA_EINVAL rules of h2sha_get_permutation); false and *err on a refusal.
bool perm_columns(const Plan& P, const h2sha_perm_desc_t& d, uint32_t usable_rows, PermColumns* out, std::string* err);

// Assembly::new + one Assembly::copy per constrain_equal / constrain_instance of the chip API, in its order.  mapping[c * U + r]
// = c' * U + r' (U = usable_rows).  False and *err when a copied cell is in no listed column or at a row >= usable_rows.
bool replay_permutation(const Plan& P, const PermColumns& cols, std::vector<uint32_t>* mapping, std::string* err);

// Canonical DELTA = 7^(2^28) and the 2^k-th root of unity ROOT_OF_UNITY^(2^(28 - k)), ROOT_OF_UNITY = 7^((p - 1) / 2^28)
// (halo2curves bn256::Fr), both in Montgomery form.
U256 perm_delta_mont();
U256 perm_omega_mont(uint32_t k);

}  // namespace h2sha
