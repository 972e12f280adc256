// planner.h -- host planner: configuration -> static plan (layout, templates, slot programs, shape).
//
// The plan is input-independent: for a given `Config` every instance has the same cell at the same
// (column,row); only the values differ.  The planner walks the reference's program order
// (lib.rs:71-349 -> compression.rs:19-213 -> spread.rs:76-233; halo2-base op patterns per SURVEY.md 8a-B)
// symbolically and records, per unit type, how each cell's value derives from a handful of u32 trace words.
#pragma once
#include <string>
#include <vector>

#include "fr_host.h"
#include "h2sha_defs.h"

namespace h2sha {

// Mirrors the constructor arguments of the reference: Sha256DynamicConfig::configure (lib.rs:49-56),
// RangeConfig::configure (lib.rs:409-418) and ContextParams (lib.rs:354-358).
struct Config {
  std::vector<uint32_t> max_variable_byte_sizes;  // one entry per digest() call sharing a Context
  uint32_t max_rows = (1u << 17) - 9;             // range.gate.max_rows
  uint32_t lookup_bits = 16;                      // RangeConfig lookup_bits
  uint32_t limb_bits = 8;                         // SpreadConfig num_bits_lookup
  uint32_t spread_cols = 2;                       // SpreadConfig num_advice_columns
  uint32_t is_input_range_check = 1;
  uint32_t record_shape = 1;                      // also build selectors / copy constraints / fixed column
  uint32_t record_compact_map = 0;                // also build the cell -> dictionary-entry map of the compact hand-off (host side)
  uint32_t block_parts = 3;                       // engine tuning: jobs per sha256_compression (load balance vs. overhead)
  uint32_t max_fill = 144;                        // engine tuning: distinct values per chunk (size of a warp's scratch table)
  uint32_t digest_batch = 0;                      // engine tuning: instances per digest job (0 = as many as fit, <= 32)
  uint32_t resident_consts = 16;                  // engine tuning: most-used constants kept permanently in every warp's scratch
};

enum : uint32_t { CP_GATE = 0, CP_FIXED = 1 };
struct CopyPair {
  uint32_t a_kind, a_idx, b_kind, b_idx;
};
struct DigestHandles {  // AssignedHashResult (lib.rs:31-36) as gate-stream indices
  uint32_t input_len_idx;
  std::vector<uint32_t> input_bytes_idx;
  uint32_t output_bytes_idx[32];
};
// cells of the column-major buffers nobody assigns (column tails, alignment padding): zero-filled by the engine
enum : uint32_t { BUF_GATE = 0, BUF_LOOKUP = 1, BUF_SPREAD = 2 };
struct ZeroRange {
  uint32_t buf, pos, count;
};

struct Plan {
  Config cfg;
  // ---- device-side data ----
  std::vector<UnitType> types;
  std::vector<std::string> type_names;
  std::vector<VmIns> prog;
  std::vector<FillEntry> fill;          // fill lists of all chunks
  std::vector<uint32_t> resident;       // static-table indices of the constants every warp keeps in scratch slots [0, n)
  std::vector<CellEntry> cells;         // cell lists of all chunks
  std::vector<Chunk> chunks;
  std::vector<ItemDesc> items;          // phase-2 work items of all classes
  std::vector<uint32_t> item_dict;      // per item: dictionary index of its chunk's first distinct value, relative to the job's dictionary base
  uint32_t n_block_parts = 1;
  std::vector<UnitGroup> groups;
  std::vector<WarpTask> tasks;
  std::vector<JobClass> classes;        // classes [0, n_block_parts) = block-job parts; then one digest job class per digest
  std::vector<uint64_t> raw_consts;     // VM constants
  std::vector<U256> mont_table;         // Montgomery-form table: [fixed constants | byte | spread-byte | inverses]
  uint32_t tb_byte = 0, tb_sbyte = 0, tb_inv = 0, inv_bias = 0;
  std::vector<DigestPlace> digests;
  std::vector<ZeroRange> zero_ranges;
  // ---- layout (per instance) ----
  uint32_t n_gate = 0, n_lookup = 0, n_limb = 0;  // stream lengths
  std::vector<uint32_t> breaks;                   // gate-stream index at which column c starts (breaks[0] == 0)
  uint32_t n_gate_cols = 0, gate_col_rows = 0;
  uint32_t n_lookup_cols = 0, lookup_col_rows = 0;
  uint32_t spread_rows = 0;
  uint32_t max_slots = 0, max_trace_words = 0;
  // ---- shape (host only; record_shape) ----
  std::vector<uint8_t> selectors;            // per gate-stream index
  std::vector<CopyPair> copies;
  std::vector<U256> fixed_consts;            // canonical values, first-use order (fixed column cells)
  std::vector<uint32_t> lookup_cells;        // cells_to_lookup as gate-stream indices
  std::vector<uint32_t> limb_gate_dense, limb_gate_spread;
  std::vector<DigestHandles> handles;
  // ---- compact hand-off (host only): which dictionary entry every cell copies.  Entry = index into the instance's dictionary of
  // distinct values, or 0x80000000 | index into mont_table for the constants every warp keeps resident ----
  uint32_t dict_cells = 0;                   // distinct values per instance
  std::vector<uint32_t> map_gate;            // per gate-stream index
  std::vector<uint32_t> map_lookup;          // per cells_to_lookup index
  std::vector<uint32_t> map_dense, map_spread;   // per spread limb
  // ---- statistics ----
  uint64_t cells_per_instance() const { return (uint64_t)n_gate + n_lookup + 2ull * n_limb; }
};

// Recomputes Plan::zero_ranges from the current column strides (call after widening gate_col_rows etc.).
void compute_zero_ranges(Plan* plan);

// Returns false and sets *err when the reference would panic / is unsupported.
bool build_plan(const Config& cfg, Plan* out, std::string* err);

}  // namespace h2sha
