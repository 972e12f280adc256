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
// Result: five violation counters.  Not on the timed path; reads every cell a few times (L2-resident per instance).
#pragma once

namespace {

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
  unsigned long long* viol;      // [5]
};

__device__ __forceinline__ const uint64_t* tagged_cell(const CheckArgs& A, uint64_t inst, uint32_t t) {
  const uint32_t tag = t >> 30, pos = t & 0x3fffffffu;
  if (tag == 0) return A.gate + (inst * A.gate_inst_cells + pos) * 4;
  if (tag == 1) return A.lookup + (inst * A.lookup_inst_cells + pos) * 4;
  if (tag == 2) return A.spread + (inst * A.spread_inst_cells + pos) * 4;
  return A.fixed + (uint64_t)pos * 4;
}

// grid = (tiles, instances)
__global__ void __launch_bounds__(256) k_check_gates(const CheckArgs A) {
  const uint64_t inst = blockIdx.y;
  const uint64_t* g = A.gate + inst * A.gate_inst_cells * 4;
  uint32_t bad = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_gate_on; i += gridDim.x * blockDim.x) {
    const uint64_t* p = g + (uint64_t)A.gate_on[i] * 4;
    uint64_t a[4], b[4], c[4], d[4], bc[4], s[4];
    load_cell(p, a); load_cell(p + 4, b); load_cell(p + 8, c); load_cell(p + 12, d);
    mont_mul_dev(b, c, bc);
    fr_add_dev(a, bc, s);
    if ((s[0] ^ d[0]) | (s[1] ^ d[1]) | (s[2] ^ d[2]) | (s[3] ^ d[3])) bad++;
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&A.viol[0], (unsigned long long)bad);
}

__global__ void __launch_bounds__(256) k_check_pairs(const CheckArgs A) {
  const uint64_t inst = blockIdx.y;
  uint32_t bad = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < A.n_pairs; i += gridDim.x * blockDim.x) {
    const uint2 pr = reinterpret_cast<const uint2*>(A.pairs)[i];
    uint64_t x[4], y[4];
    load_cell(tagged_cell(A, inst, pr.x), x);
    load_cell(tagged_cell(A, inst, pr.y), y);
    if ((x[0] ^ y[0]) | (x[1] ^ y[1]) | (x[2] ^ y[2]) | (x[3] ^ y[3])) bad++;
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&A.viol[1], (unsigned long long)bad);
}

// one thread per output byte: grid = ceil(n_inst * n_digests * 32 / 256)
__global__ void __launch_bounds__(256) k_check_digest_bytes(const CheckArgs A, uint64_t n_inst) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t bad = 0;
  if (i < n_inst * A.n_digests * 32) {
    const uint64_t inst = i / (A.n_digests * 32u);
    const uint32_t r = (uint32_t)(i - inst * (A.n_digests * 32u));   // d * 32 + byte
    const uint64_t* cell = A.gate + (inst * A.gate_inst_cells + A.out_bytes[r]) * 4;
    const uint64_t* want = reinterpret_cast<const uint64_t*>(A.byte_tab) + (uint64_t)A.digests[i] * 4;
    uint64_t x[4], y[4];
    load_cell(cell, x); load_cell(want, y);
    if ((x[0] ^ y[0]) | (x[1] ^ y[1]) | (x[2] ^ y[2]) | (x[3] ^ y[3])) bad = 1;
  }
  bad = __reduce_add_sync(0xffffffffu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(&A.viol[4], (unsigned long long)bad);
}

// the static part of the check: built from a shape-recording plan of the same configuration, uploaded once
int ensure_check_tables(h2sha_engine* e) {
  if (e->d_chk_gate_on) return H2SHA_OK;
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
  if ((uint64_t)P.n_gate_cols * P.gate_col_rows >= (1u << 30)) return set_err(H2SHA_EINVAL, "instance too large for the checker's position tags");
  auto gate_pos = [&](uint32_t idx) {
    const uint32_t c = (uint32_t)(std::upper_bound(P.breaks.begin(), P.breaks.end(), idx) - P.breaks.begin()) - 1;
    return c * P.gate_col_rows + (idx - P.breaks[c]);
  };
  std::vector<uint32_t> gate_on;
  for (uint32_t i = 0; i < S->selectors.size(); i++)
    if (S->selectors[i]) {
      if (i + 3 >= P.n_gate || gate_pos(i + 3) != gate_pos(i) + 3) return set_err(H2SHA_EINVAL, "a gate straddles a column");
      gate_on.push_back(gate_pos(i));
    }
  std::vector<uint32_t> pairs;
  auto tag = [&](uint32_t kind, uint32_t idx) { return kind == CP_GATE ? gate_pos(idx) : ((3u << 30) | idx); };
  for (const CopyPair& cp : S->copies) { pairs.push_back(tag(cp.a_kind, cp.a_idx)); pairs.push_back(tag(cp.b_kind, cp.b_idx)); }
  const LookupGeom G = lookup_geom(P);
  for (uint32_t k = 0; k < S->lookup_cells.size(); k++) {   // range.finalize
    const LookupCell c = G.range_cell(k);
    pairs.push_back((1u << 30) | (c.col * P.lookup_col_rows + c.row));
    pairs.push_back(gate_pos(S->lookup_cells[k]));
  }
  for (uint32_t n = 0; n < S->limb_gate_dense.size(); n++) {   // the dense and the spread cell of limb n
    const LookupCell c = G.spread_cell(n);
    pairs.push_back((2u << 30) | (c.col * P.spread_rows + c.row));
    pairs.push_back(gate_pos(S->limb_gate_dense[n]));
    pairs.push_back((2u << 30) | ((G.spread_cols + c.col) * P.spread_rows + c.row));
    pairs.push_back(gate_pos(S->limb_gate_spread[n]));
  }
  std::vector<uint64_t> fixed(S->fixed_consts.size() * 4 + 4, 0);
  for (size_t i = 0; i < S->fixed_consts.size(); i++) { const U256 m = fr::to_mont(S->fixed_consts[i]); memcpy(&fixed[4 * i], m.l, 32); }
  std::vector<uint32_t> out_bytes;
  for (const DigestHandles& h : S->handles) for (int j = 0; j < 32; j++) out_bytes.push_back(gate_pos(h.output_bytes_idx[j]));
  std::vector<uint64_t> bytes(256 * 4);
  for (uint32_t v = 0; v < 256; v++) { const U256 m = fr::to_mont(fr::from_u64(v)); memcpy(&bytes[4 * v], m.l, 32); }
  auto up = [&](const void* src, size_t bytes_n, void** dst) -> int {
    CUDA_TRY(cudaMalloc(dst, std::max<size_t>(bytes_n, 16)));
    CUDA_TRY(cudaMemcpy(*dst, src, bytes_n, cudaMemcpyHostToDevice));
    return H2SHA_OK;
  };
  int rc;
  if ((rc = up(pairs.data(), pairs.size() * 4, (void**)&e->d_chk_pairs))) return rc;
  if ((rc = up(fixed.data(), fixed.size() * 8, (void**)&e->d_chk_fixed))) return rc;
  if ((rc = up(out_bytes.data(), out_bytes.size() * 4, (void**)&e->d_chk_out_bytes))) return rc;
  if ((rc = up(bytes.data(), bytes.size() * 8, (void**)&e->d_chk_bytes))) return rc;
  CUDA_TRY(cudaMalloc(&e->d_chk_viol, 5 * 8));
  e->n_chk_gate_on = (uint32_t)gate_on.size(); e->n_chk_pairs = (uint32_t)(pairs.size() / 2);
  if ((rc = up(gate_on.data(), gate_on.size() * 4, (void**)&e->d_chk_gate_on))) return rc;   // last: marks the tables as ready
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
  CUDA_TRY(cudaSetDevice(e->device));
  int rc = ensure_check_tables(e);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const Plan& P = e->plan;
  CheckArgs A{};
  A.gate_inst_cells = e->dplan.gate_inst_cells; A.lookup_inst_cells = e->dplan.lookup_inst_cells; A.spread_inst_cells = e->dplan.spread_inst_cells;
  A.gate_on = e->d_chk_gate_on; A.n_gate_on = e->n_chk_gate_on;
  A.pairs = e->d_chk_pairs; A.n_pairs = e->n_chk_pairs; A.fixed = e->d_chk_fixed;
  A.out_bytes = e->d_chk_out_bytes; A.n_digests = (uint32_t)P.digests.size(); A.byte_tab = (const uint32_t*)e->d_chk_bytes;
  A.viol = e->d_chk_viol;
  CUDA_TRY(cudaMemsetAsync(e->d_chk_viol, 0, 5 * 8, st));
  // lookups: the multiplicity kernels without bins (cells outside their table are counted)
  uint32_t* bad32 = reinterpret_cast<uint32_t*>(e->d_chk_viol + 2);   // [2] range (low word), [3] spread (low word)
  const LookupGeom G = lookup_geom(P);
  for (uint64_t i0 = 0; i0 < n_instances; i0 += 65535) {
    const unsigned ni = (unsigned)std::min<uint64_t>(65535, n_instances - i0);
    A.gate = (const uint64_t*)gate + i0 * A.gate_inst_cells * 4;
    A.lookup = (const uint64_t*)lookup + i0 * A.lookup_inst_cells * 4;
    A.spread = (const uint64_t*)spread + i0 * A.spread_inst_cells * 4;
    const unsigned gt = (unsigned)std::max<uint32_t>(1, std::min<uint32_t>((A.n_gate_on + 255) / 256, 64));
    k_check_gates<<<dim3(gt, ni), 256, 0, st>>>(A);
    CUDA_TRY(cudaGetLastError());
    const unsigned pt = (unsigned)std::max<uint32_t>(1, std::min<uint32_t>((A.n_pairs + 255) / 256, 128));
    k_check_pairs<<<dim3(pt, ni), 256, 0, st>>>(A);
    CUDA_TRY(cudaGetLastError());
    const unsigned rt = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((G.n_lookup + 255) / 256, 64));
    k_range_mult<<<dim3(rt, ni), 256, 0, st>>>(G, A.lookup, nullptr, bad32);
    CUDA_TRY(cudaGetLastError());
    const unsigned stl = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((G.n_limb + 1023) / 1024, 32));
    k_spread_mult<<<dim3(stl, ni), 256, 0, st>>>(G, A.spread, nullptr, bad32 + 2);   // check-only: no histogram, no shared memory
    CUDA_TRY(cudaGetLastError());
  }
  if (digests_dev) {
    A.gate = (const uint64_t*)gate; A.digests = digests_dev;
    const uint64_t n = n_instances * A.n_digests * 32;
    k_check_digest_bytes<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(A, n_instances);
    CUDA_TRY(cudaGetLastError());
  }
  CUDA_TRY(cudaMemcpyAsync(violations_host, e->d_chk_viol, 5 * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
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
