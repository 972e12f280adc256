// batch_check.cuh -- MockProver-style constraint check of a WHOLE batch on the device.  Included at the end of engine.cu.
//
// The reference's tests accept a witness when `MockProver::run(..).verify() == Ok(())` (src/lib.rs:525-526): every gate,
// every copy constraint, every range / spread lookup, and the digest bytes against the instance column.  oracle/mock_prover.py
// does that on the host for sampled instances; this does it for every instance of a batch where the witness lies, in HBM:
//   (i)   gates:   q * (a + b*c - d) = 0 on the 4 consecutive rows of every enabled gate (halo2-base FlexGate, Vertical);
//   (ii)  copies:  every copy constraint the chip emits while `digest` runs (gate cell <-> gate cell / fixed constant), the
//                  lookup-column cells against the cells range.finalize copies (lib.rs:469) and the spread-column cells
//                  against their gate cells (spread.rs:209-227);
//   (iii) lookups: lookup-column cells < 2^lookup_bits; (dense, spread) pairs are rows of the spread table (spread.rs:53-62);
//   (iv)  digest:  the 32 output-byte cells of every digest() call (lib.rs:311-341) against the engine's digest bytes.
// The static shape (selectors, copies, fixed cells) is the planner's (record_shape); it is built on first use.
// Result per instance and class: the violation count and the smallest failing item number (the numbering of
// h2sha_check_batch_per_instance; check_items() below is its one definition).  Every warp reduces its lanes and issues one
// atomicAdd / atomicMin pair per class, and only when it holds a failure: a clean batch issues no atomics.
// Not on the timed path; reads every cell a few times (L2-resident per instance).
#pragma once

// Every check item, in the numbering of h2sha_check_site (include/h2sha_b200.h).  The device tables are derived from these lists
// and the resolver reads them, so the kernels and the resolver cannot number an item differently.  Classes 2 and 3 need no list:
// item k / n is lookup cell k / spread limb n (LookupGeom).
struct h2sha_check_items {
  struct Cell {
    uint32_t kind, index, row;   // H2SHA_COL_*, column index, row
  };
  std::vector<Cell> gate;       // class 0: the first of the gate's four rows
  std::vector<Cell> copy;       // class 1: [n][2]
  std::vector<Cell> out_byte;   // class 4: [n_digests][32]
  std::vector<U256> fixed;      // canonical fixed constants (fixed column rows)
  LookupGeom G;
};

void h2sha_free_check_items(h2sha_check_items* c) { delete c; }

namespace {

enum { N_CHECK_CLASSES = 5 };

// the item lists, from a shape-recording plan of the engine's configuration (the engine's own plan when it records the shape)
int ensure_check_items(h2sha_engine* e) {
  if (e->chk_items) return H2SHA_OK;
  Plan shape_local;
  const Plan* S = &e->plan;
  if (!e->plan.cfg.record_shape) {
    Config c = e->plan.cfg;
    c.record_shape = 1;
    std::string err;
    if (!build_plan(c, &shape_local, &err)) return set_err(H2SHA_EINVAL, "shape plan: " + err);
    S = &shape_local;
  }
  const Plan& P = e->plan;   // strides of the engine (possibly widened)
  if (S->n_gate != P.n_gate || S->breaks != P.breaks) return set_err(H2SHA_EINVAL, "shape plan does not match the engine's plan");
  using Cell = h2sha_check_items::Cell;
  auto gate_cell = [&](uint32_t idx) {
    const uint32_t c = (uint32_t)(std::upper_bound(P.breaks.begin(), P.breaks.end(), idx) - P.breaks.begin()) - 1;
    return Cell{H2SHA_COL_GATE, c, idx - P.breaks[c]};
  };
  h2sha_check_items* I = new h2sha_check_items();
  I->G = lookup_geom(P);
  for (uint32_t i = 0; i < S->selectors.size(); i++)
    if (S->selectors[i]) {
      const Cell c = gate_cell(i);
      if (i + 3 >= P.n_gate || gate_cell(i + 3).index != c.index) { delete I; return set_err(H2SHA_EINVAL, "a gate straddles a column"); }
      I->gate.push_back(c);
    }
  I->copy.reserve(2 * S->copies.size() + 2 * S->lookup_cells.size() + 4 * S->limb_gate_dense.size());
  auto shape_cell = [&](uint32_t kind, uint32_t idx) { return kind == CP_GATE ? gate_cell(idx) : Cell{H2SHA_COL_FIXED, 0, idx}; };
  for (const CopyPair& cp : S->copies) { I->copy.push_back(shape_cell(cp.a_kind, cp.a_idx)); I->copy.push_back(shape_cell(cp.b_kind, cp.b_idx)); }
  for (uint32_t k = 0; k < S->lookup_cells.size(); k++) {   // range.finalize
    const LookupCell c = I->G.range_cell(k);
    I->copy.push_back(Cell{H2SHA_COL_LOOKUP, c.col, c.row});
    I->copy.push_back(gate_cell(S->lookup_cells[k]));
  }
  for (uint32_t n = 0; n < S->limb_gate_dense.size(); n++) {   // the dense and the spread cell of limb n
    const LookupCell c = I->G.spread_cell(n);
    I->copy.push_back(Cell{H2SHA_COL_DENSE, c.col, c.row});
    I->copy.push_back(gate_cell(S->limb_gate_dense[n]));
    I->copy.push_back(Cell{H2SHA_COL_SPREAD, c.col, c.row});
    I->copy.push_back(gate_cell(S->limb_gate_spread[n]));
  }
  for (const DigestHandles& h : S->handles) for (int j = 0; j < 32; j++) I->out_byte.push_back(gate_cell(h.output_bytes_idx[j]));
  I->fixed = S->fixed_consts;
  e->chk_items = I;
  return H2SHA_OK;
}

// items of a class per instance
uint64_t check_class_items(const h2sha_check_items& I, uint32_t cls) {
  switch (cls) {
    case 0: return I.gate.size();
    case 1: return I.copy.size() / 2;
    case 2: return I.G.n_lookup;
    case 3: return I.G.n_limb;
    default: return I.out_byte.size();
  }
}

struct CheckArgs {
  uint64_t gate_inst_cells, lookup_inst_cells, spread_inst_cells;
  const uint64_t* gate;
  const uint64_t* lookup;
  const uint64_t* spread;
  const uint8_t* digests;        // [n_inst][n_digests][32] or null
  const uint32_t* gate_on;       // positions (inside the instance's gate buffer) of the first row of every enabled gate
  uint32_t n_gate_on;
  const uint32_t* pairs;         // [n_pairs][2]: buffer-tagged positions that must hold equal values (tag in the top 2 bits:
  uint32_t n_pairs;              //   0 gate, 1 lookup, 2 spread, 3 fixed-constant index)
  const uint64_t* fixed;         // Montgomery form of the fixed-column constants
  const uint32_t* out_bytes;     // [n_digests][32] positions of the output-byte cells
  uint32_t n_digests;
  const uint32_t* byte_tab;      // Montgomery form of 0..255 (prefix of the range table)
  LookupGeom G;
  uint32_t* counts;              // [n_inst][5] violations per class
  uint32_t* first;               // [n_inst][5] smallest failing item per class, or null
};

__device__ __forceinline__ const uint64_t* tagged_cell(const CheckArgs& A, uint64_t inst, uint32_t t) {
  const uint32_t tag = t >> 30, pos = t & 0x3fffffffu;
  if (tag == 0) return A.gate + (inst * A.gate_inst_cells + pos) * 4;
  if (tag == 1) return A.lookup + (inst * A.lookup_inst_cells + pos) * 4;
  if (tag == 2) return A.spread + (inst * A.spread_inst_cells + pos) * 4;
  return A.fixed + (uint64_t)pos * 4;
}

__device__ __forceinline__ bool cells_differ(const uint64_t x[4], const uint64_t y[4]) {
  return ((x[0] ^ y[0]) | (x[1] ^ y[1]) | (x[2] ^ y[2]) | (x[3] ^ y[3])) != 0;
}

// The 32 lanes' failures of class `cls` in instance `inst` (all lanes of the warp call it, for the same instance): `bad` failures
// per lane, the smallest of them `first_item` (0xFFFFFFFF when none).
__device__ __forceinline__ void report_warp(const CheckArgs& A, uint64_t inst, uint32_t cls, uint32_t bad, uint32_t first_item) {
  bad = __reduce_add_sync(0xffffffffu, bad);
  if (bad == 0) return;
  first_item = __reduce_min_sync(0xffffffffu, first_item);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&A.counts[inst * N_CHECK_CLASSES + cls], bad);
    if (A.first) atomicMin(&A.first[inst * N_CHECK_CLASSES + cls], first_item);
  }
}

// grid = (tiles, instances)
__global__ void __launch_bounds__(256) k_check_gates(const CheckArgs A) {
  const uint64_t inst = blockIdx.y;
  const uint64_t* g = A.gate + inst * A.gate_inst_cells * 4;
  uint32_t bad = 0, first = 0xffffffffu;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_gate_on; i += gridDim.x * blockDim.x) {
    const uint64_t* p = g + (uint64_t)A.gate_on[i] * 4;
    uint64_t a[4], b[4], c[4], d[4], bc[4], s[4];
    load_cell(p, a); load_cell(p + 4, b); load_cell(p + 8, c); load_cell(p + 12, d);
    mont_mul_dev(b, c, bc);
    fr_add_dev(a, bc, s);
    if (cells_differ(s, d)) { first = min(first, i); bad++; }
  }
  report_warp(A, inst, 0, bad, first);
}

__global__ void __launch_bounds__(256) k_check_pairs(const CheckArgs A) {
  const uint64_t inst = blockIdx.y;
  uint32_t bad = 0, first = 0xffffffffu;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_pairs; i += gridDim.x * blockDim.x) {
    const uint2 pr = reinterpret_cast<const uint2*>(A.pairs)[i];
    uint64_t x[4], y[4];
    load_cell(tagged_cell(A, inst, pr.x), x);
    load_cell(tagged_cell(A, inst, pr.y), y);
    if (cells_differ(x, y)) { first = min(first, i); bad++; }
  }
  report_warp(A, inst, 1, bad, first);
}

// lookup-column cells outside the range table.  grid = (tiles, instances)
__global__ void __launch_bounds__(256) k_check_range(const CheckArgs A) {
  const LookupGeom& G = A.G;
  const uint64_t inst = blockIdx.y;
  const uint64_t* base = A.lookup + inst * G.lookup_inst_cells * 4;
  const uint32_t n_vals = 1u << G.lookup_bits;
  uint32_t bad = 0, first = 0xffffffffu;
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < G.n_lookup; k += gridDim.x * blockDim.x) {
    const LookupCell c = G.range_cell(k);
    uint32_t v;
    if (!range_table_row(base + ((uint64_t)c.col * G.lookup_col_rows + c.row) * 4, n_vals, &v)) { first = min(first, k); bad++; }
  }
  report_warp(A, inst, 2, bad, first);
}

// (dense, spread) pairs that are no spread-table row; no shared memory, so 16-bit limbs work too.  grid = (tiles, instances)
__global__ void __launch_bounds__(256) k_check_spread(const CheckArgs A) {
  const LookupGeom& G = A.G;
  const uint64_t inst = blockIdx.y;
  const uint64_t* base = A.spread + inst * G.spread_inst_cells * 4;
  const uint32_t n_vals = 1u << G.limb_bits;
  uint32_t bad = 0, first = 0xffffffffu;
  for (uint32_t n = blockIdx.x * blockDim.x + threadIdx.x; n < G.n_limb; n += gridDim.x * blockDim.x) {
    const LookupCell c = G.spread_cell(n);
    uint32_t d;
    if (!spread_table_row(base + ((uint64_t)c.col * G.spread_rows + c.row) * 4, base + ((uint64_t)(G.spread_cols + c.col) * G.spread_rows + c.row) * 4,
                          n_vals, &d)) {
      first = min(first, n);
      bad++;
    }
  }
  report_warp(A, inst, 3, bad, first);
}

// one thread per output byte: grid = n_inst * n_digests * 32 / 256 rounded up.  An instance has n_digests * 32 bytes, a multiple of
// the warp: the lanes of a warp are the 32 bytes of one digest of one instance.
__global__ void __launch_bounds__(256) k_check_digest_bytes(const CheckArgs A, uint64_t n_inst) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t per_inst = A.n_digests * 32u;
  if (i - (threadIdx.x & 31) >= n_inst * per_inst) return;   // a whole warp past the batch
  const uint64_t inst = i / per_inst;
  const uint32_t r = (uint32_t)(i - inst * per_inst);   // d * 32 + byte
  const uint64_t* cell = A.gate + (inst * A.gate_inst_cells + A.out_bytes[r]) * 4;
  const uint64_t* want = reinterpret_cast<const uint64_t*>(A.byte_tab) + (uint64_t)A.digests[i] * 4;
  uint64_t x[4], y[4];
  load_cell(cell, x); load_cell(want, y);
  const bool bad = cells_differ(x, y);
  report_warp(A, inst, 4, bad ? 1u : 0u, bad ? r : 0xffffffffu);
}

// counts [n_inst][5] -> viol[5] (added)
__global__ void __launch_bounds__(256) k_check_sum(const uint32_t* counts, uint32_t n_inst, unsigned long long* viol) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
  for (int c = 0; c < N_CHECK_CLASSES; c++) {
    const uint32_t s = __reduce_add_sync(0xffffffffu, i < n_inst ? counts[(uint64_t)i * N_CHECK_CLASSES + c] : 0u);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(&viol[c], (unsigned long long)s);
  }
}

// the device tables of the check, from the item lists: uploaded once
int ensure_check_tables(h2sha_engine* e) {
  if (e->d_chk_gate_on) return H2SHA_OK;
  int rc = ensure_check_items(e);
  if (rc) return rc;
  const h2sha_check_items& I = *e->chk_items;
  const Plan& P = e->plan;
  if ((uint64_t)P.n_gate_cols * P.gate_col_rows >= (1u << 30)) return set_err(H2SHA_EINVAL, "instance too large for the checker's position tags");
  // buffer-tagged position of a cell (CheckArgs::pairs)
  auto tag = [&](const h2sha_check_items::Cell& c) -> uint32_t {
    switch (c.kind) {
      case H2SHA_COL_GATE: return c.index * P.gate_col_rows + c.row;
      case H2SHA_COL_LOOKUP: return (1u << 30) | (c.index * P.lookup_col_rows + c.row);
      case H2SHA_COL_DENSE: return (2u << 30) | (c.index * P.spread_rows + c.row);
      case H2SHA_COL_SPREAD: return (2u << 30) | ((I.G.spread_cols + c.index) * P.spread_rows + c.row);
      default: return (3u << 30) | c.row;   // fixed constant
    }
  };
  std::vector<uint32_t> gate_on, pairs, out_bytes;
  gate_on.reserve(I.gate.size()); pairs.reserve(I.copy.size()); out_bytes.reserve(I.out_byte.size());
  for (const auto& c : I.gate) gate_on.push_back(tag(c));
  for (const auto& c : I.copy) pairs.push_back(tag(c));
  for (const auto& c : I.out_byte) out_bytes.push_back(tag(c));
  std::vector<uint64_t> fixed(I.fixed.size() * 4 + 4, 0);
  for (size_t i = 0; i < I.fixed.size(); i++) { const U256 m = fr::to_mont(I.fixed[i]); memcpy(&fixed[4 * i], m.l, 32); }
  std::vector<uint64_t> bytes(256 * 4);
  for (uint32_t v = 0; v < 256; v++) { const U256 m = fr::to_mont(fr::from_u64(v)); memcpy(&bytes[4 * v], m.l, 32); }
  auto up = [&](const void* src, size_t bytes_n, void** dst) -> int {
    CUDA_TRY(cudaMalloc(dst, std::max<size_t>(bytes_n, 16)));
    CUDA_TRY(cudaMemcpy(*dst, src, bytes_n, cudaMemcpyHostToDevice));
    return H2SHA_OK;
  };
  if ((rc = up(pairs.data(), pairs.size() * 4, (void**)&e->d_chk_pairs))) return rc;
  if ((rc = up(fixed.data(), fixed.size() * 8, (void**)&e->d_chk_fixed))) return rc;
  if ((rc = up(out_bytes.data(), out_bytes.size() * 4, (void**)&e->d_chk_out_bytes))) return rc;
  if ((rc = up(bytes.data(), bytes.size() * 8, (void**)&e->d_chk_bytes))) return rc;
  CUDA_TRY(cudaMalloc(&e->d_chk_viol, 5 * 8));
  e->n_chk_gate_on = (uint32_t)gate_on.size(); e->n_chk_pairs = (uint32_t)(pairs.size() / 2);
  if ((rc = up(gate_on.data(), gate_on.size() * 4, (void**)&e->d_chk_gate_on))) return rc;   // last: marks the tables as ready
  return H2SHA_OK;
}

// the common part of both calls: argument checks, tables, and the arguments every chunk shares
int check_setup(h2sha_engine_t* e, const void* gate, const void* lookup, const void* spread, CheckArgs* A) {
  if (!e || !gate || !lookup || !spread) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  CUDA_TRY(cudaSetDevice(e->device));
  const int rc = ensure_check_tables(e);
  if (rc) return rc;
  *A = CheckArgs{};
  A->gate_inst_cells = e->dplan.gate_inst_cells; A->lookup_inst_cells = e->dplan.lookup_inst_cells; A->spread_inst_cells = e->dplan.spread_inst_cells;
  A->gate_on = e->d_chk_gate_on; A->n_gate_on = e->n_chk_gate_on;
  A->pairs = e->d_chk_pairs; A->n_pairs = e->n_chk_pairs; A->fixed = e->d_chk_fixed;
  A->out_bytes = e->d_chk_out_bytes; A->n_digests = (uint32_t)e->plan.digests.size(); A->byte_tab = (const uint32_t*)e->d_chk_bytes;
  A->G = e->chk_items->G;
  return H2SHA_OK;
}

// Every check of instances [i0, i0 + ni) (ni <= 65535: grid.y), into counts / first [ni][5], which are overwritten.
int check_chunk(CheckArgs A, uint64_t i0, unsigned ni, const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                uint32_t* counts, uint32_t* first, cudaStream_t st) {
  A.gate = (const uint64_t*)gate + i0 * A.gate_inst_cells * 4;
  A.lookup = (const uint64_t*)lookup + i0 * A.lookup_inst_cells * 4;
  A.spread = (const uint64_t*)spread + i0 * A.spread_inst_cells * 4;
  A.digests = digests_dev ? digests_dev + i0 * A.n_digests * 32 : nullptr;
  A.counts = counts; A.first = first;
  CUDA_TRY(cudaMemsetAsync(counts, 0, (size_t)ni * N_CHECK_CLASSES * 4, st));
  if (first) CUDA_TRY(cudaMemsetAsync(first, 0xff, (size_t)ni * N_CHECK_CLASSES * 4, st));
  const unsigned gt = (unsigned)std::max<uint32_t>(1, std::min<uint32_t>((A.n_gate_on + 255) / 256, 64));
  k_check_gates<<<dim3(gt, ni), 256, 0, st>>>(A);
  CUDA_TRY(cudaGetLastError());
  const unsigned pt = (unsigned)std::max<uint32_t>(1, std::min<uint32_t>((A.n_pairs + 255) / 256, 128));
  k_check_pairs<<<dim3(pt, ni), 256, 0, st>>>(A);
  CUDA_TRY(cudaGetLastError());
  const unsigned rt = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((A.G.n_lookup + 255) / 256, 64));
  k_check_range<<<dim3(rt, ni), 256, 0, st>>>(A);
  CUDA_TRY(cudaGetLastError());
  const unsigned stl = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((A.G.n_limb + 1023) / 1024, 32));
  k_check_spread<<<dim3(stl, ni), 256, 0, st>>>(A);
  CUDA_TRY(cudaGetLastError());
  if (A.digests) {
    const uint64_t n = (uint64_t)ni * A.n_digests * 32;
    k_check_digest_bytes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(A, ni);
    CUDA_TRY(cudaGetLastError());
  }
  return H2SHA_OK;
}

}  // namespace

extern "C" {

int h2sha_check_batch(h2sha_engine_t* e, uint64_t n_instances, const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                      uint64_t* violations_host, void* stream) {
  if (!e || !gate || !lookup || !spread || !violations_host) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): there is no CPU path");
  memset(violations_host, 0, 5 * 8);
  if (n_instances == 0) return H2SHA_OK;
  CheckArgs A;
  int rc = check_setup(e, gate, lookup, spread, &A);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // per-instance counts of one chunk (<= 65535 x 5 u32 = 1.3 MB), summed into the five counters
  const uint64_t cap = std::min<uint64_t>(n_instances, 65535);
  if (cap > e->chk_counts_cap) {
    e->chk_counts_cap = 0;
    if ((rc = dev_realloc(e->d_chk_counts, cap * N_CHECK_CLASSES * 4))) return rc;
    e->chk_counts_cap = cap;
  }
  CUDA_TRY(cudaMemsetAsync(e->d_chk_viol, 0, 5 * 8, st));
  for (uint64_t i0 = 0; i0 < n_instances; i0 += 65535) {
    const unsigned ni = (unsigned)std::min<uint64_t>(65535, n_instances - i0);
    if ((rc = check_chunk(A, i0, ni, gate, lookup, spread, digests_dev, e->d_chk_counts, nullptr, st))) return rc;
    k_check_sum<<<(ni + 255) / 256, 256, 0, st>>>(e->d_chk_counts, ni, e->d_chk_viol);
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaMemcpyAsync(violations_host, e->d_chk_viol, 5 * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return H2SHA_OK;
}

int h2sha_check_batch_per_instance(h2sha_engine_t* e, uint64_t n_instances, const void* gate, const void* lookup, const void* spread,
                                   const uint8_t* digests_dev, uint32_t* counts_dev, uint32_t* first_dev, void* stream) {
  if (!counts_dev) return set_err(H2SHA_EINVAL, "null argument");
  CheckArgs A;
  int rc = check_setup(e, gate, lookup, spread, &A);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  for (uint64_t i0 = 0; i0 < n_instances; i0 += 65535) {
    const unsigned ni = (unsigned)std::min<uint64_t>(65535, n_instances - i0);
    if ((rc = check_chunk(A, i0, ni, gate, lookup, spread, digests_dev, counts_dev + i0 * N_CHECK_CLASSES,
                          first_dev ? first_dev + i0 * N_CHECK_CLASSES : nullptr, st)))
      return rc;
  }
  return H2SHA_OK;
}

int h2sha_check_site(h2sha_engine_t* e, uint32_t check_class, uint32_t item, h2sha_check_site_t* out) {
  if (!e || !out) return set_err(H2SHA_EINVAL, "null argument");
  const int rc = ensure_check_items(e);
  if (rc) return rc;
  const h2sha_check_items& I = *e->chk_items;
  if (check_class >= N_CHECK_CLASSES) return set_err(H2SHA_EINVAL, "check class out of range (0 .. 4)");
  if (item >= check_class_items(I, check_class)) return set_err(H2SHA_EINVAL, "check item out of range for its class");
  memset(out, 0, sizeof *out);
  auto put = [&](uint32_t kind, uint32_t index, uint32_t row) {
    out->kind[out->n_cells] = kind; out->index[out->n_cells] = index; out->row[out->n_cells] = row; out->n_cells++;
  };
  auto put_cell = [&](const h2sha_check_items::Cell& c) { put(c.kind, c.index, c.row); };
  switch (check_class) {
    case 0: for (uint32_t j = 0; j < 4; j++) put(H2SHA_COL_GATE, I.gate[item].index, I.gate[item].row + j); break;
    case 1: put_cell(I.copy[2 * (uint64_t)item]); put_cell(I.copy[2 * (uint64_t)item + 1]); break;
    case 2: { const LookupCell c = I.G.range_cell(item); put(H2SHA_COL_LOOKUP, c.col, c.row); break; }
    case 3: { const LookupCell c = I.G.spread_cell(item); put(H2SHA_COL_DENSE, c.col, c.row); put(H2SHA_COL_SPREAD, c.col, c.row); break; }
    default: put_cell(I.out_byte[item]); break;
  }
  return H2SHA_OK;
}

// ---------------------------------------------------------------------------------------------------
// The only collective of the path (SURVEY.md 8e): all-gather of digests and per-instance checksums (64 B per instance) over
// the caller's NCCL communicator.  NCCL is resolved at run time (dlopen of libnccl.so.2), so libh2sha_b200.so itself links
// nothing but the CUDA runtime; without NCCL the call fails with H2SHA_EINVAL and a message.
// ---------------------------------------------------------------------------------------------------
int h2sha_gather(void* nccl_comm, uint64_t n_instances_per_rank, uint32_t n_digests, const uint8_t* digests_dev, const uint64_t* checksums_dev,
                 uint8_t* all_digests_dev, uint64_t* all_checksums_dev, void* stream) {
  if (!nccl_comm) return set_err(H2SHA_EINVAL, "null NCCL communicator");
  if ((!digests_dev) != (!all_digests_dev) || (!checksums_dev) != (!all_checksums_dev)) return set_err(H2SHA_EINVAL, "send and receive buffers must be given in pairs");
  // resolved once per process; the static-local initialiser is thread-safe (C++11) and publishes the pointers only after all
  // of them are known, so one host thread per GPU may make its first call at the same moment (tools/native_runner.cc)
  struct Nccl {
    typedef int (*all_gather_fn)(const void*, void*, size_t, int, void*, cudaStream_t);
    typedef int (*group_fn)(void);
    typedef const char* (*err_fn)(int);
    void* lib = nullptr;
    all_gather_fn all_gather = nullptr;
    group_fn start = nullptr, end = nullptr;
    err_fn err = nullptr;
    std::string why;
  };
  static const Nccl nccl = [] {
    Nccl n;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) { n.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (n.lib) break; }
    if (!n.lib) { const char* de = dlerror(); n.why = std::string("NCCL is not loadable: ") + (de ? de : "dlopen failed"); return n; }
    n.all_gather = (Nccl::all_gather_fn)dlsym(n.lib, "ncclAllGather");
    n.start = (Nccl::group_fn)dlsym(n.lib, "ncclGroupStart");
    n.end = (Nccl::group_fn)dlsym(n.lib, "ncclGroupEnd");
    n.err = (Nccl::err_fn)dlsym(n.lib, "ncclGetErrorString");
    if (!n.all_gather || !n.start || !n.end) { n.why = "libnccl lacks ncclAllGather / ncclGroupStart / ncclGroupEnd"; n.all_gather = nullptr; }
    return n;
  }();
  if (!nccl.all_gather) return set_err(H2SHA_EINVAL, nccl.why);
  const auto p_all_gather = nccl.all_gather;
  const auto p_start = nccl.start, p_end = nccl.end;
  const auto p_err = nccl.err;
  const int kUint8 = 1, kUint64 = 5;   // ncclDataType_t values (nccl.h), stable across NCCL 2.x
  int rc = p_start();
  if (!rc && digests_dev) rc = p_all_gather(digests_dev, all_digests_dev, (size_t)n_instances_per_rank * n_digests * 32, kUint8, nccl_comm, (cudaStream_t)stream);
  if (!rc && checksums_dev) rc = p_all_gather(checksums_dev, all_checksums_dev, (size_t)n_instances_per_rank * 4, kUint64, nccl_comm, (cudaStream_t)stream);
  const int rc_end = p_end();
  if (!rc) rc = rc_end;
  if (rc) return set_err(H2SHA_ECUDA, std::string("NCCL: ") + (p_err ? p_err(rc) : "error"));
  return H2SHA_OK;
}

}  // extern "C"
