// export.cuh -- prover hand-off of whole batches (SURVEY.md §8f #2).  Included at the end of engine.cu.
//
// The consumer of the witness is halo2's prover (`create_proof`, reference benches/digest.rs:143-157), which holds one vector of
// 2^k field elements per advice column.  Two ways to get a batch there:
//   h2sha_export_batch     the cells themselves: three strided device-to-host copies for the whole batch (one per buffer kind)
//                          into [instance][column][2^k] host vectors -- PCIe-bound at 32 bytes per cell;
//   the compact hand-off   h2sha_batch_t.compact_dict makes the expansion kernel write every DISTINCT value of an instance once
//                          (the fill entries of its chunks: ~27 % of the cells); h2sha_get_compact_map says which dictionary
//                          entry (or which of a few constants) every cell copies -- a static, input-independent table --
//                          and h2sha_expand_compact rebuilds the [instance][column][2^k] vectors on the host with plain 32-byte
//                          copies, multi-threaded.  No field arithmetic happens on the host: it is a gather, not a CPU path
//                          for the witness (it also runs on a plan-only engine, i.e. on a prover box without a GPU).
#pragma once

#include <atomic>
#include <memory>
#include <thread>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

struct h2sha_compact_state {
  Plan plan;                       // the engine's configuration planned with record_compact_map
  std::vector<uint64_t> consts;    // Montgomery form of mont_table, 4 x u64 each
};

namespace {

int ensure_compact(h2sha_engine* e) {
  if (e->compact) return H2SHA_OK;
  std::unique_ptr<h2sha_compact_state> st(new h2sha_compact_state());
  Config c = e->plan.cfg;
  c.record_compact_map = 1; c.record_shape = 0;
  std::string err;
  if (!build_plan(c, &st->plan, &err)) return set_err(H2SHA_EINVAL, "compact map plan: " + err);
  if (st->plan.dict_cells != e->plan.dict_cells || st->plan.n_gate != e->plan.n_gate || st->plan.breaks != e->plan.breaks)
    return set_err(H2SHA_EINVAL, "compact map plan does not match the engine's plan");
  st->consts.resize(st->plan.mont_table.size() * 4);
  for (size_t i = 0; i < st->plan.mont_table.size(); i++) memcpy(&st->consts[4 * i], st->plan.mont_table[i].l, 32);
  e->compact = st.release();
  return H2SHA_OK;
}

struct HostGeom {   // [instance][column][rows_per_column] host layout shared by export_batch and expand_compact
  uint32_t n_gate_cols, n_lookup_cols, n_spread_cols, total_cols, rows;
  uint64_t inst_cells;
};
HostGeom host_geom(const Plan& P, uint32_t rows_per_column) {
  HostGeom g;
  g.n_gate_cols = P.n_gate_cols; g.n_lookup_cols = P.n_lookup_cols; g.n_spread_cols = 2 * P.cfg.spread_cols;
  g.total_cols = g.n_gate_cols + g.n_lookup_cols + g.n_spread_cols;
  g.rows = rows_per_column;
  g.inst_cells = (uint64_t)g.total_cols * rows_per_column;
  return g;
}
// assigned rows of the largest column of each buffer kind
void used_rows(const Plan& P, uint32_t used[3]) {
  used[0] = 0;
  for (size_t c = 0; c < P.breaks.size(); c++) used[0] = std::max(used[0], ((c + 1 < P.breaks.size()) ? P.breaks[c + 1] : P.n_gate) - P.breaks[c]);
  const LookupGeom G = lookup_geom(P);
  used[1] = G.max_range_used();
  used[2] = G.max_spread_used();
}

}  // namespace

extern "C" {

int h2sha_get_compact_info(const h2sha_engine_t* e, h2sha_compact_info_t* out) {
  if (!e || !out) return set_err(H2SHA_EINVAL, "null argument");
  memset(out, 0, sizeof *out);
  out->dict_cells_per_instance = e->plan.dict_cells;
  out->dict_bytes_per_instance = (uint64_t)e->plan.dict_cells * 32;
  out->cells_per_instance = e->plan.cells_per_instance();
  out->n_consts = (uint32_t)e->plan.mont_table.size();
  return H2SHA_OK;
}

int h2sha_get_compact_map(h2sha_engine_t* e, uint32_t* gate_map, uint32_t* lookup_map, uint32_t* dense_map, uint32_t* spread_map, uint64_t* consts) {
  if (!e) return set_err(H2SHA_EINVAL, "null argument");
  int rc = ensure_compact(e);
  if (rc) return rc;
  const Plan& C = e->compact->plan;
  if (gate_map) memcpy(gate_map, C.map_gate.data(), C.map_gate.size() * 4);
  if (lookup_map) memcpy(lookup_map, C.map_lookup.data(), C.map_lookup.size() * 4);
  if (dense_map) memcpy(dense_map, C.map_dense.data(), C.map_dense.size() * 4);
  if (spread_map) memcpy(spread_map, C.map_spread.data(), C.map_spread.size() * 4);
  if (consts) memcpy(consts, e->compact->consts.data(), e->compact->consts.size() * 8);
  return H2SHA_OK;
}

int h2sha_export_batch(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, const void* gate, const void* lookup, const void* spread,
                       void* host_out, uint32_t rows_per_column, int zero_fill, void* stream) {
  if (!e || !host_out) return set_err(H2SHA_EINVAL, "null argument");
  if (e->device < 0) return set_err(H2SHA_ECUDA, "plan-only engine (device = -1): nothing to export; there is no CPU path");
  if (n_instances == 0) return H2SHA_OK;
  const Plan& P = e->plan;
  uint32_t used[3];
  used_rows(P, used);
  const void* bufs[3] = {gate, lookup, spread};
  for (int b = 0; b < 3; b++)
    if (bufs[b] && used[b] > rows_per_column) return set_err(H2SHA_EINVAL, "rows_per_column is smaller than the assigned rows of a column");
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const HostGeom G = host_geom(P, rows_per_column);
  if (zero_fill) memset(host_out, 0, (size_t)n_instances * G.inst_cells * 32);   // the rows nobody assigns; needed once per host buffer (the shape is static)
  const uint32_t col_rows[3] = {P.gate_col_rows, P.lookup_col_rows, P.spread_rows};
  const uint32_t n_cols[3] = {G.n_gate_cols, G.n_lookup_cols, G.n_spread_cols};
  const uint32_t col0[3] = {0, G.n_gate_cols, G.n_gate_cols + G.n_lookup_cols};
  const uint64_t inst_cells[3] = {e->dplan.gate_inst_cells, e->dplan.lookup_inst_cells, e->dplan.spread_inst_cells};
  for (int b = 0; b < 3; b++) {
    if (!bufs[b]) continue;
    // one 3-D copy per buffer kind: x = the assigned prefix of a column, y = the columns of the kind, z = the instances
    cudaMemcpy3DParms p{};
    p.srcPtr = make_cudaPitchedPtr((void*)((const uint8_t*)bufs[b] + first_instance * inst_cells[b] * 32), (size_t)col_rows[b] * 32, (size_t)col_rows[b] * 32, n_cols[b]);
    p.dstPtr = make_cudaPitchedPtr(host_out, (size_t)rows_per_column * 32, (size_t)rows_per_column * 32, G.total_cols);
    p.dstPos = make_cudaPos(0, col0[b], 0);
    p.extent = make_cudaExtent((size_t)std::min(col_rows[b], rows_per_column) * 32, n_cols[b], n_instances);
    p.kind = cudaMemcpyDeviceToHost;
    CUDA_TRY(cudaMemcpy3DAsync(&p, st));
  }
  return H2SHA_OK;
}

int h2sha_expand_compact(h2sha_engine_t* e, const void* dict_host, uint64_t n_instances, void* host_out, uint32_t rows_per_column, int zero_fill,
                         uint32_t n_threads) {
  if (!e || !dict_host || !host_out) return set_err(H2SHA_EINVAL, "null argument");
  int rc = ensure_compact(e);
  if (rc) return rc;
  const Plan& P = e->plan;
  const Plan& C = e->compact->plan;
  const LookupGeom L = lookup_geom(P);
  uint32_t used[3];
  used_rows(P, used);
  if (std::max(used[0], std::max(used[1], used[2])) > rows_per_column) return set_err(H2SHA_EINVAL, "rows_per_column is smaller than the assigned rows of a column");
  const HostGeom G = host_geom(P, rows_per_column);
  const uint64_t* consts = e->compact->consts.data();
  const uint64_t dict_cells = P.dict_cells;
  // work units: (instance, segment); segments = the gate columns, then the lookup stream, then the spread limbs
  const uint32_t n_seg = G.n_gate_cols + 2;
  std::atomic<uint64_t> next{0};
  const uint64_t n_units = n_instances * n_seg;
  // every output cell is written exactly once and not read again by this call: non-temporal stores skip the read-for-ownership of
  // the destination line, which is half of the memory traffic of a plain 32-byte copy (the expander is memory-bound)
  const bool aligned16 = ((uintptr_t)host_out & 15u) == 0;
  auto put = [&](uint64_t* dst, const uint64_t* dict, uint32_t m) {
    const uint64_t* src = (m & 0x80000000u) ? consts + (uint64_t)(m & 0x7fffffffu) * 4 : dict + (uint64_t)m * 4;
#if defined(__SSE2__)
    if (aligned16) {
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst), _mm_loadu_si128(reinterpret_cast<const __m128i*>(src)));
      _mm_stream_si128(reinterpret_cast<__m128i*>(dst) + 1, _mm_loadu_si128(reinterpret_cast<const __m128i*>(src) + 1));
      return;
    }
#endif
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
  };
  auto worker = [&]() {
    for (;;) {
      const uint64_t u = next.fetch_add(1);
      if (u >= n_units) break;
      const uint64_t inst = u / n_seg;
      const uint32_t seg = (uint32_t)(u - inst * n_seg);
      const uint64_t* dict = (const uint64_t*)dict_host + inst * dict_cells * 4;
      uint64_t* out = (uint64_t*)host_out + inst * G.inst_cells * 4;
      if (seg < G.n_gate_cols) {
        const uint32_t lo = P.breaks[seg], hi = (seg + 1 < P.breaks.size()) ? P.breaks[seg + 1] : P.n_gate;
        uint64_t* col = out + (uint64_t)seg * G.rows * 4;
        for (uint32_t i = lo; i < hi; i++) put(col + (uint64_t)(i - lo) * 4, dict, C.map_gate[i]);
        if (zero_fill) memset(col + (uint64_t)(hi - lo) * 4, 0, (size_t)(G.rows - (hi - lo)) * 32);
      } else if (seg == G.n_gate_cols) {
        for (uint32_t c = 0; c < G.n_lookup_cols; c++) {
          uint64_t* col = out + (uint64_t)(G.n_gate_cols + c) * G.rows * 4;
          const uint32_t lo = L.range_first(c), hi = lo + L.range_used(c);
          for (uint32_t k = lo; k < hi; k++) put(col + (uint64_t)(k - lo) * 4, dict, C.map_lookup[k]);
          if (zero_fill) memset(col + (uint64_t)(hi - lo) * 4, 0, (size_t)(G.rows - (hi - lo)) * 32);
        }
      } else {
        const uint32_t nc = L.spread_cols;
        uint64_t* base = out + (uint64_t)(G.n_gate_cols + G.n_lookup_cols) * G.rows * 4;
        for (uint32_t n = 0; n < P.n_limb; n++) {
          const LookupCell c = L.spread_cell(n);
          put(base + ((uint64_t)c.col * G.rows + c.row) * 4, dict, C.map_dense[n]);
          put(base + ((uint64_t)(nc + c.col) * G.rows + c.row) * 4, dict, C.map_spread[n]);
        }
        if (zero_fill)
          for (uint32_t c = 0; c < 2 * nc; c++) {
            const uint32_t rows_used = L.spread_used(c % nc);
            memset(base + ((uint64_t)c * G.rows + rows_used) * 4, 0, (size_t)(G.rows - rows_used) * 32);
          }
      }
    }
#if defined(__SSE2__)
    _mm_sfence();   // non-temporal stores are weakly ordered: make them visible before the thread is joined
#endif
  };
  uint32_t nt = n_threads ? n_threads : std::max(1u, std::thread::hardware_concurrency());
  nt = (uint32_t)std::min<uint64_t>(nt, n_units);
  if (nt <= 1) { worker(); return H2SHA_OK; }
  std::vector<std::thread> th;
  for (uint32_t t = 0; t < nt; t++) th.emplace_back(worker);
  for (auto& t : th) t.join();
  return H2SHA_OK;
}

}  // extern "C"
