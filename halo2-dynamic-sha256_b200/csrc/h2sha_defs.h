// h2sha_defs.h -- data structures shared by the host planner and the sm_100a kernels.
//
// The engine is a two-phase, plan-driven expander (see DESIGN.md):
//   phase 1 ("slots"):  per unit instance (one SHA-256 round, one schedule step, ...) a tiny
//                       straight-line VM program turns a few u32 trace words into <= 255 raw u64 "slots";
//   phase 2 ("cells"):  per chunk of a unit, every distinct value ((slot >> sh) & mask, a table lookup of it, a
//                       constant, ...) is converted once to BN254 Fr Montgomery form in a per-warp scratch table
//                       (fill), then every advice / lookup / spread-column cell is a 32-byte copy from that table
//                       to its final (column,row).
// The VM programs, fill lists and cell lists are produced once per configuration by the host planner
// (planner.cc), which walks the reference's call order (lib.rs:71-349 -> compression.rs:19-213 ->
// spread.rs:76-233) symbolically.
#pragma once
#include <stdint.h>

namespace h2sha {

// ---------------------------------------------------------------------------------------------
// Value descriptor ("template entry"): how one Fr value derives from the unit's slots.  8 bytes.
//   lo: dst (16)  | tbl (16)
//   hi: slot (8) | sh (6) | w (7) | shl (5) | kind (2) | neg (1)
// value(raw)  = ((slots[slot] >> sh) & mask(w)) << shl          (w == 0 -> 0, w == 64 -> all bits)
// KIND_TABLE  : cell = mont_table[tbl + value(raw)]             (constants: w == 0)
// KIND_GENERIC: cell = Mont(value(raw)), negated mod p if neg
// KIND_SIGNED : slots[slot] is an int64; cell = Mont(|v|), negated if v < 0
// ---------------------------------------------------------------------------------------------
enum : uint32_t { KIND_TABLE = 0, KIND_GENERIC = 1, KIND_SIGNED = 2 };

struct TmplEntry {
  uint32_t lo, hi;
};
static inline TmplEntry tmpl_pack(uint32_t dst, uint32_t tbl, uint32_t slot, uint32_t sh, uint32_t w, uint32_t shl, uint32_t kind,
                                  uint32_t neg) {
  TmplEntry e;
  e.lo = (dst & 0xffffu) | (tbl << 16);
  e.hi = (slot & 0xffu) | ((sh & 63u) << 8) | ((w & 127u) << 14) | ((shl & 31u) << 21) | ((kind & 3u) << 26) | ((neg & 1u) << 28);
  return e;
}
#define H2SHA_TE_DST(e) ((e).lo & 0xffffu)
#define H2SHA_TE_TBL(e) ((e).lo >> 16)
#define H2SHA_TE_SLOT(e) ((e).hi & 0xffu)
#define H2SHA_TE_SH(e) (((e).hi >> 8) & 63u)
#define H2SHA_TE_W(e) (((e).hi >> 14) & 127u)
#define H2SHA_TE_SHL(e) (((e).hi >> 21) & 31u)
#define H2SHA_TE_KIND(e) (((e).hi >> 26) & 3u)
#define H2SHA_TE_NEG(e) (((e).hi >> 28) & 1u)

// ---------------------------------------------------------------------------------------------
// Slot VM.  Operand (32 bit): is_const (1) | slot-or-const-index (12) | sh (6) | w (7)
//   is_const: value = raw_consts[index]   else: value = (slots[slot] >> sh) & mask(w)
// ---------------------------------------------------------------------------------------------
enum : uint32_t {
  OP_ADD = 0,        // dst = A + B
  OP_SUB = 1,        // dst = A - B            (wrapping; read back as int64 by KIND_SIGNED)
  OP_MULADD = 2,     // dst = A * B + C
  OP_SPREAD = 3,     // dst = bit-interleave of the low 32 bits of A with zeros (bit i -> bit 2i)
  OP_COMPRESS2 = 4,  // dst = even16(A) | even16(B)<<16 | odd16(A)<<32 | odd16(B)<<48   (A,B 32-bit)
  OP_EQ = 5,         // dst = (A == B)
  OP_GT = 6,         // dst = (A > B), unsigned
  OP_SEL = 7,        // dst = A ? B : C
  OP_MOV = 8,        // dst = A
};
struct VmIns {
  uint32_t op_dst;  // op (8) | dst slot (8)
  uint32_t a, b, c;
};
static inline uint32_t vm_operand_slot(uint32_t slot, uint32_t sh, uint32_t w) { return (slot << 1) | ((sh & 63u) << 13) | ((w & 127u) << 19); }
static inline uint32_t vm_operand_const(uint32_t idx) { return 1u | (idx << 1); }

// ---------------------------------------------------------------------------------------------
// Phase 2 works chunk by chunk (a chunk = up to a few hundred consecutive cells of one unit):
//   fill:  every DISTINCT value of the chunk is materialised once (TmplEntry, `dst` = scratch slot) in the warp's scratch
//          table: KIND_TABLE entries (constants, 8-bit limbs, spread limbs, inverses) are copied from the static
//          Montgomery table, the others go through the Barrett conversion; entries are sorted
//          TABLE | GENERIC <= 32 bit | GENERIC > 32 bit / SIGNED;
//   copy:  every cell is a 32-byte copy  scratch[src] -> its (column,row)  (CellEntry).
// ---------------------------------------------------------------------------------------------
struct CellEntry {
  uint32_t v;  // gate / lookup cells: src (16) | dst (16).  src = index into the warp's scratch table
               // spread-column cells: src (8) | dst (10) | slot (8) | sh (6): slot / sh say where the limb's raw value sits in the
               // unit's slots (width = limb bits), so that the table-row multiplicities can be counted while the cells are written
};
#define H2SHA_CE_SRC(e) ((e).v & 0xffffu)
#define H2SHA_CE_DST(e) ((e).v >> 16)
#define H2SHA_LE_SRC(e) ((e).v & 0xffu)
#define H2SHA_LE_DST(e) (((e).v >> 8) & 0x3ffu)
#define H2SHA_LE_SLOT(e) (((e).v >> 18) & 0xffu)
#define H2SHA_LE_SH(e) ((e).v >> 26)
enum { H2SHA_MAX_FILL_LIMIT = 256 };   // the actual limit is Config::max_fill (runtime, <= this)

// Fill entry: how to materialise one distinct value (same packing as TmplEntry, dst = scratch slot) plus the weight of
// the value in the gate checksum: it is carried by `cnt & 0xffff` gate cells of the chunk whose unit-relative offsets sum to
// `sumdst`.  `cnt >> 16` = lookup-column cells of the chunk that carry the value (its multiplicity in the range lookup).
struct alignas(16) FillEntry {
  uint32_t lo, hi;
  uint32_t cnt, sumdst;
};
#define H2SHA_FE_GATE_CNT(e) ((e).cnt & 0xffffu)
#define H2SHA_FE_LK_CNT(e) ((e).cnt >> 16)

// multipliers of the cell checksum hash (include/h2sha_b200.h: H2SHA_CK_M)
static const uint32_t kCkM[8] = {0x9E3779B1u, 0x85EBCA77u, 0xC2B2AE3Du, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};

struct alignas(16) Chunk {
  uint64_t res_a, res_b;   // gate-checksum contribution of the resident constants of the chunk: res_a + res_b * (2*pos0 + 1)
  uint32_t fill_off;   // FillEntry index
  uint16_t n_fill, n_fill_table;   // distinct values to materialise; the first n_fill_table are table copies
  uint32_t gate_off;   // CellEntry index; dst = gate-stream offset inside the unit
  uint16_t gate_len, n_fill32;     // n_fill32: Barrett entries known to be < 2^32 (they follow the table copies)
  uint32_t lk_off;     // dst = lookup index inside the unit
  uint16_t lk_len, gate_dst_min;   // smallest / largest gate dst of the chunk (to detect a column break inside it)
  uint32_t limb_off;   // dst = (limb index inside the unit) << 1 | (0 dense, 1 spread)
  uint16_t limb_len, gate_dst_max;
};

// Unit type: slot program + chunks (offsets into the plan's flat arrays).
struct UnitType {
  uint32_t n_in, n_slots;        // input slots, total slots (slot stride is n_slots | 1)
  uint32_t prog_off, prog_len;   // VmIns
  uint32_t chunk_off, n_chunks;  // Chunk
  uint32_t gate_len, lk_len, limb_len;   // cells per instance (limb_len = 2 per limb)
  uint32_t dict_len;                     // distinct values per instance = fill entries of all its chunks (compact hand-off)
};

// Input source of slot k of a unit instance u: trace[in_base + in_stride * u]; or the instance index u itself.
struct InputMap {
  int32_t base;    // index into the job's trace array (u32 words); -1: value = u
  int32_t stride;
};
enum { MAX_UNIT_INPUTS = 20 };

// A group = `count` consecutive instances of one unit type inside a job.
struct UnitGroup {
  uint32_t type;
  uint32_t count;                // unit instances in the job = per_inst * (instances the job covers)
  uint32_t per_inst;             // unit instances per circuit instance (== count for block jobs, which cover one instance)
  uint32_t slot_base;            // offset (in u64) of instance 0's slots in the job's slot area
  uint32_t gate_base, gate_stride;   // gate-stream index of instance 0 relative to the job's gate base, and per-instance stride
  uint32_t lk_base, lk_stride;       // same for the lookup stream
  uint32_t limb_base, limb_stride;   // same for spread limbs
  uint32_t dict_base;                // dictionary index of instance 0's first distinct value, relative to the job's dictionary base
  InputMap in[MAX_UNIT_INPUTS];
};

// Warp task of phase 1: lanes = instances [first, first+32) of a group.
struct WarpTask {
  uint32_t group, first;
};

// Work item of phase 2: one chunk of one unit instance, with everything that does not depend on the job precomputed.
struct alignas(16) ItemDesc {
  uint32_t gate_rel;   // gate-stream index of the unit's first cell, relative to the job's gate base
  uint32_t lk_rel;     // same for the lookup stream
  uint32_t limb_rel;   // same for spread limbs
  uint32_t slot_chunk; // slot_off (16: offset in u64 units of the unit's slots in the job's slot area) | Chunk index (11) |
                       // inst_off (5: which of the job's circuit instances the unit belongs to)
};
#define H2SHA_ITEM_SLOT(x) ((x) & 0xffffu)
#define H2SHA_ITEM_CHUNK(x) (((x) >> 16) & 0x7ffu)
#define H2SHA_ITEM_INST(x) ((x) >> 27)
enum { H2SHA_MAX_JOB_BATCH = 32 };

// A job class: (a part of) the block job (one sha256_compression) or the per-digest prologue/epilogue job.
struct JobClass {
  uint32_t group_off, n_groups;  // UnitGroup
  uint32_t task_off, n_tasks;    // WarpTask (phase 1)
  uint32_t item_off, n_items;    // phase-2 work items, heaviest first
  uint32_t n_slots_total;        // u64 slots needed in shared memory
  uint32_t n_trace_words;        // u32 words of trace the job loads, per circuit instance
  uint32_t batch;                // circuit instances one job covers (1 for block jobs; digest jobs are batched so that the
                                 // lanes of the slot VM are filled and its latency is amortised)
  uint32_t digest;               // digest-job classes: the digest() call the class belongs to (0 for block-job parts)
};

// Trace layout of a block job (u32 words), written by the trace kernel:
//   W[64] | A[68] | E[68]          A[k+4] / E[k+4] = working variables a / e after round k;
//                                  A[3..0] = a,b,c,d and E[3..0] = e,f,g,h of the input state
enum { TR_W = 0, TR_A = 64, TR_E = 132, TR_K = 200, TR_BLOCK_WORDS = 200, TR_BLOCK_WORDS_WITH_K = 264 };
// Trace layout of a digest job: scalars | H[8] | states[(R+1)][8] | msg words [R][16]
enum { TD_LEN = 0, TD_NUM_ROUND = 1, TD_PRE_ROUND = 2, TD_TARGET = 3, TD_H = 4, TD_STATES = 12 };

// Per-digest placement inside one instance (all stream indices are instance-relative).
struct DigestPlace {
  uint32_t max_bytes, n_blocks;
  uint32_t gate_base, lk_base, limb_base;   // start of this digest's prologue
  uint32_t blk_gate_base, blk_lk_base, blk_limb_base;   // block 0 of this digest (after the one-time zero cell, if any)
  uint32_t blk_gate_stride, blk_lk_stride, blk_limb_stride;
  uint32_t dict_base, dict_dig_len, dict_blk_len;   // compact hand-off: the digest's dictionary range starts at dict_base with the prologue /
                                 // epilogue units (dict_dig_len values), followed by n_blocks x dict_blk_len values of its compressions
  uint32_t job_class;            // first digest-job class of this digest (block-job parts are classes 0 .. n_block_parts-1; a digest
                                 // whose slots exceed one stage is cut into several consecutive classes, JobClass::digest names the owner)
  uint32_t trace_words;          // digest-job trace words
};

}  // namespace h2sha
