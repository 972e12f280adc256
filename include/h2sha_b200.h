/*
 * h2sha_b200.h -- C ABI of the B200-native SHA-256 witness-generation engine.
 *
 * Drop-in boundary for ONE path of zhmolly/halo2-dynamic-sha256: the value-producing half of
 * `Sha256DynamicConfig::digest` (reference src/lib.rs:71-349) together with `sha256_compression`
 * (src/compression.rs:19-213) and `SpreadConfig::{spread,spread_limb,decompose_even_and_odd_unchecked}`
 * (src/spread.rs:76-233).  The reference has no FFI of its own: its boundary is the Rust API
 *   configure(meta, max_variable_byte_sizes, range, num_bits_lookup, num_advice_columns, is_input_range_check)  lib.rs:49-56
 *   digest(&mut self, ctx, input: &[u8], precomputed_input_len: Option<usize>) -> AssignedHashResult           lib.rs:71-76
 *   new_context / range / load                                                                                  lib.rs:351-368
 * Each entry point below names the reference item it replaces.  INTEGRATION.md shows the Rust binding.
 *
 * Model: one *instance* = one halo2 region / `Context` in which `n_digests` digest() calls are made in
 * order (the reference's tests use 2, its bench 1).  For a given configuration every instance has the
 * same shape; the engine produces, for a batch of instances, every advice cell as BN254 Fr in
 * Montgomery form (4 x u64 little-endian limbs = halo2curves bn256::Fr memory layout), column-major:
 *
 *   gate   [instance][n_gate_cols  ][gate_col_rows  ]  FlexGate advice columns (halo2-base, Vertical)
 *   lookup [instance][n_lookup_cols][lookup_col_rows]  range-lookup advice column(s) filled by range.finalize
 *   spread [instance][2*num_advice_columns][spread_rows]  SpreadConfig denses[0..], then spreads[0..]
 *
 * Cells the reference never assigns are NOT written (zero the buffers once; the shape is static, so they
 * stay zero across reuse).  All pointers are plain C; no C++ or torch types cross this boundary.
 * Every call returns 0 on success or a negative H2SHA_E* code; h2sha_last_error() gives the message
 * (thread-local).  The engine never falls back to the CPU: without a CUDA device every call fails.
 */
#ifndef H2SHA_B200_H
#define H2SHA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define H2SHA_OK 0
#define H2SHA_EINVAL (-1)      /* bad argument / configuration the reference would reject (lib.rs:57-59, spread.rs:37) */
#define H2SHA_EPANIC (-2)      /* input the reference would panic on (lib.rs:89-90: bad precomputed length, message too long) */
#define H2SHA_ECUDA (-3)       /* CUDA runtime error (no device, launch failure, out of memory) */
#define H2SHA_ENOMEM (-4)

typedef struct h2sha_engine h2sha_engine_t;

/* Replaces the arguments of Sha256DynamicConfig::configure (lib.rs:49-56), RangeConfig::configure
 * (lib.rs:409-418: lookup_bits, k) and ContextParams.max_rows (lib.rs:354-358). */
typedef struct {
  uint32_t n_digests;                       /* max_variable_byte_sizes.len()                                   */
  const uint32_t* max_variable_byte_sizes;  /* each a positive multiple of 64 (lib.rs:57-59); this engine: <= 7808 (122 blocks) per digest
                                               (inverse table of is_zero); larger -> H2SHA_EINVAL */
  uint32_t max_rows;                        /* range.gate.max_rows = 2^k - minimum_rows; 0 -> 2^17 - 9          */
  uint32_t lookup_bits;                     /* RangeConfig lookup_bits; 0 -> 16                                 */
  uint32_t num_bits_lookup;                 /* SpreadConfig limb bits, divides 16 (1, 2, 4, 8, 16); 0 -> 8      */
  uint32_t num_advice_columns;              /* SpreadConfig column pairs; 0 -> 2                                */
  uint32_t is_input_range_check;            /* lib.rs:55,174-178                                                */
  uint32_t gate_col_rows;                   /* row stride of a gate column in the output; 0 -> tight            */
  uint32_t lookup_col_rows;                 /* 0 -> tight                                                       */
  uint32_t spread_rows;                     /* 0 -> tight                                                       */
  int32_t device;                           /* CUDA device ordinal; -1 = plan-only (host queries, no witness)   */
  uint32_t build_shape;                     /* also build selectors / copy constraints / fixed column (host)    */
  uint32_t block_parts;                     /* tuning: GPU jobs per sha256_compression; 0 -> default (3: throughput).
                                               >= 12 = latency setting for one digest at a time (e.g. 24): the compression is
                                               cut into 8-instance jobs for as many SMs; not for batches                        */
  uint32_t num_lookup_advice;               /* RangeConfig's NUM_LOOKUP_ADVICE (lib.rs:413,492): lookup advice columns the circuit has;
                                               0 -> as many as the looked-up cells need.  Fewer than needed -> H2SHA_EINVAL (halo2-base
                                               would panic); more -> the extra columns stay empty.  Cells fill column 0 up to max_rows,
                                               then column 1: for more than ONE column this order is an unpinned recollection of halo2-base */
} h2sha_config_t;

typedef struct {
  uint32_t n_digests;
  uint32_t n_gate_cells, n_lookup_cells, n_spread_limbs;   /* stream lengths per instance                    */
  uint32_t n_gate_cols, gate_col_rows;
  uint32_t n_lookup_cols, lookup_col_rows;
  uint32_t n_spread_cols, spread_rows;                     /* n_spread_cols = 2 * num_advice_columns          */
  uint32_t n_blocks;                                       /* sha256_compression calls per instance           */
  uint32_t n_fixed, n_copies, n_selectors_on;              /* shape sizes (0 unless build_shape)              */
  uint64_t cells_per_instance;                             /* assigned Fr per instance over all three buffers */
  uint64_t gate_bytes, lookup_bytes, spread_bytes;         /* buffer bytes per instance                       */
} h2sha_layout_t;

/* Sha256DynamicConfig::configure + new_context (lib.rs:49-69, 351-360): builds the static plan and uploads it. */
int h2sha_create(const h2sha_config_t* cfg, h2sha_engine_t** out);
void h2sha_destroy(h2sha_engine_t* e);
const char* h2sha_last_error(void);
/* Stamp of the sources and flags this library was built from (halo2-dynamic-sha256_b200/build.py compares it with the tree). */
const char* h2sha_build_id(void);
int h2sha_get_layout(const h2sha_engine_t* e, h2sha_layout_t* out);

/* Gate-stream index -> (column,row): column c holds stream indices [breaks[c], breaks[c+1]).  `breaks` gets n_gate_cols entries. */
int h2sha_get_breaks(const h2sha_engine_t* e, uint32_t* breaks);
/* AssignedHashResult (lib.rs:31-36, 342-346) of digest d as gate-stream indices:
 * input_len (1), input_bytes (max_variable_byte_sizes[d]), output_bytes (32). */
int h2sha_get_handles(const h2sha_engine_t* e, uint32_t d, uint32_t* input_len_idx, uint32_t* input_bytes_idx, uint32_t* output_bytes_idx);
/* The stream ranges each digest() call owns (what that call appends in the reference, lib.rs:122-341):
 * ranges [n_digests][6] = gate_lo, gate_hi, lookup_lo, lookup_hi, limb_lo, limb_hi (half-open; gate-stream indices,
 * cells_to_lookup indices, spread-limb indices).  A facade that assigns cells digest() call by digest() call uses them. */
int h2sha_get_digest_ranges(const h2sha_engine_t* e, uint32_t* ranges);

/* Shape (needs build_shape): what keygen needs and what MockProver checks.
 *   selectors  [n_gate_cells] u8        gate selector per gate-stream index (q * (a + b*c - d) = 0 over 4 rows)
 *   copies     [n_copies][4] u32        (a_kind,a_idx,b_kind,b_idx); kind 0 = gate stream, 1 = fixed column cell
 *   fixed      [n_fixed][4] u64         canonical (non-Montgomery) constants, first-use order (Context::assign_fixed)
 *   lookup_src [n_lookup_cells] u32     gate-stream index each lookup-column cell copies (range.finalize, lib.rs:469)
 *   limb_dense_src / limb_spread_src [n_spread_limbs] u32   gate cells the spread-column cells are copy-constrained to (spread.rs:209-227)
 * Any pointer may be NULL. */
int h2sha_get_shape(const h2sha_engine_t* e, uint8_t* selectors, uint32_t* copies, uint64_t* fixed, uint32_t* lookup_src,
                    uint32_t* limb_dense_src, uint32_t* limb_spread_src);

/* The fixed lookup tables keygen has to load next to the shape:
 *   SpreadConfig::load (spread.rs:165-194): 2^num_bits_lookup rows (dense i, spread(i)) with bit b of i at bit 2b of spread(i);
 *   range.load_lookup_table (lib.rs:442): 2^lookup_bits rows holding 0 .. 2^lookup_bits - 1 (only the row count is returned).
 * table_dense / table_spread: [2^num_bits_lookup] u64 canonical values, may be NULL. */
int h2sha_get_lookup_tables(const h2sha_engine_t* e, uint64_t* table_dense, uint64_t* table_spread, uint32_t* n_spread_rows, uint32_t* n_range_rows);

/* One batch = n_instances instances; message m = instance * n_digests + d. */
typedef struct {
  uint64_t n_instances;
  const uint8_t* msgs;               /* packed message bytes                                                     */
  int32_t msgs_on_device;            /* 0: `msgs` is host memory (copied H2D on `stream`), 1: device memory       */
  uint64_t msgs_bytes;               /* total bytes in `msgs`                                                     */
  const uint64_t* offsets;           /* host, [n_msgs]: byte offset of message m in `msgs`                        */
  const uint32_t* lens;              /* host, [n_msgs]: input.len()                                               */
  const uint32_t* precomputed_lens;  /* host, [n_msgs] or NULL (= None): precomputed_input_len (lib.rs:75,88)     */
  void* gate;                        /* device, n_instances * gate_bytes, or NULL to skip                         */
  void* lookup;                      /* device, n_instances * lookup_bytes, or NULL                               */
  void* spread;                      /* device, n_instances * spread_bytes, or NULL                               */
  uint8_t* digests_dev;              /* device [n_msgs][32] or NULL                                               */
  uint64_t* checksums_dev;           /* device [n_instances][4] or NULL: gate, lookup, spread, total              */
  uint8_t* digests_host;             /* host [n_msgs][32] or NULL: copied D2H on `stream`                         */
  uint64_t* checksums_host;          /* host [n_instances][4] or NULL                                             */
  void* stream;                      /* cudaStream_t (NULL = default stream); the call only enqueues              */
  int32_t reuse_inputs;              /* 1: messages / offsets / lens uploaded by the previous call on this engine are
                                        still resident in HBM and are reused (no validation, no H2D); n_instances
                                        must not exceed that call's                                                */
  int32_t time_kernels;              /* 1: bracket each kernel with CUDA events on `stream` (h2sha_last_kernel_ms) */
  uint32_t only_digest;              /* 0: every digest() call of every instance; d + 1: only the cells digest() call d owns
                                        (h2sha_get_digest_ranges) are generated -- for a facade that assigns call by call */
  uint32_t* lookup_mult_dev;         /* device [n_instances][mult_words_per_instance] u32 or NULL: the table-row multiplicities
                                        h2sha_lookup_multiplicities would compute from the finished witness, counted here while the
                                        cells are written (no second pass over HBM).  Needs gate, lookup and spread.            */
  uint32_t mult_usable_rows;         /* rows every lookup is evaluated on (2^k - blinding factors - 1), for lookup_mult_dev     */
  uint32_t* mult_not_in_table_dev;   /* device u32 or NULL: looked-up cells that are no table row (0 for an honest witness)     */
  void* compact_dict;                /* device [n_instances][dict_cells_per_instance] Fr or NULL: the compact hand-off -- every DISTINCT
                                        value of an instance once (3.7x fewer bytes than its cells); h2sha_get_compact_map says which
                                        entry each cell copies, h2sha_expand_compact rebuilds the columns on the host.  gate / lookup /
                                        spread may be NULL then (nothing but the dictionary is written)                         */
  uint32_t keep_lookup_raw;          /* 1: like lookup_mult_dev, but nothing dense is written: the raw values of the looked-up cells stay in the
                                        engine (17.6 KB per block) and h2sha_permute_lookup_from_raw bins them per lookup on the fly.  Needs
                                        gate, lookup and spread; valid until the next batch with lookup_mult_dev / keep_lookup_raw       */
} h2sha_batch_t;

/* Replaces `digest` (lib.rs:71-349) for a whole batch: padding and length selection, the precomputed
 * prefix state (sha2::compress256, lib.rs:153-160), every compression and every cell.
 * The call only enqueues: every host INPUT array (msgs when it is host memory, offsets, lens, precomputed_lens) is copied
 * into the engine's pinned staging ring before the call returns and may be reused at once; the call never waits for
 * the device (exception: more than 8 calls in flight, when the oldest staging slot is still being copied from).
 * Results reach digests_host / checksums_host in stream order: synchronise `stream` (or an event recorded after the
 * call) before reading them; they must stay valid until then and should be pinned (a pageable destination makes the
 * CUDA runtime block inside the call).  With host messages and host result buffers the H2D copy and the trace kernel
 * run on an engine-owned stream and overlap the previous batch's expansion kernel. */
int h2sha_digest_batch(h2sha_engine_t* e, const h2sha_batch_t* batch);

/* Prover hand-off: copy ONE instance's advice columns from the batch buffers to host memory, one vector per advice
 * column, `rows_per_column` (normally 2^k) Fr each, zero-padded -- the layout halo2's witness collection / MockProver
 * hold (`advice[column][row]`).  Column order = allocation order of the reference's configure (lib.rs:409-428,
 * spread.rs:39-52): gate advice columns, lookup advice column(s), SpreadConfig denses[0..], spreads[0..].
 * `host_columns` has n_gate_cols + n_lookup_cols + n_spread_cols pointers.  Asynchronous on `stream` when the host
 * memory is pinned; any of the device buffers may be NULL (its columns are skipped). */
int h2sha_export_instance(h2sha_engine_t* e, uint64_t instance, const void* gate, const void* lookup, const void* spread,
                          uint64_t* const* host_columns, uint32_t rows_per_column, void* stream);

/* Prover hand-off of a whole batch: instances [first_instance, first_instance + n_instances) of the batch buffers to host memory
 * laid out [instance][column][rows_per_column] Fr (column order as h2sha_export_instance; rows_per_column normally 2^k) with three
 * strided copies in total (one per buffer kind) on `stream`; asynchronous when host_out is pinned.  Rows nobody assigns are not
 * written: zero_fill != 0 clears host_out first (needed once per host buffer -- the shape is static).  NULL buffers are skipped. */
int h2sha_export_batch(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, const void* gate, const void* lookup, const void* spread,
                       void* host_out, uint32_t rows_per_column, int zero_fill, void* stream);

/* ---- Compact hand-off: h2sha_batch_t.compact_dict holds every DISTINCT value of an instance once (~27 % of its cells, 3.7x fewer
 * bytes over PCIe); which entry each cell copies is static (input-independent) and comes from h2sha_get_compact_map:
 *   gate_map [n_gate_cells], lookup_map [n_lookup_cells], dense_map / spread_map [n_spread_limbs]: per gate-stream index /
 *   cells_to_lookup index / spread limb, either an index into the instance's dictionary or 0x80000000 | index into `consts`
 *   ([n_consts][4] u64 Montgomery: the few constants the kernel keeps resident instead of writing them per instance).
 * h2sha_expand_compact rebuilds [instance][column][rows_per_column] host vectors (the layout of h2sha_export_batch) from a
 * dictionary in host memory with n_threads host threads (0 = all cores): 32-byte copies only, no field arithmetic.  Both
 * calls work on a plan-only engine (device = -1), i.e. on a prover box without a GPU. */
typedef struct {
  uint64_t dict_cells_per_instance, dict_bytes_per_instance;
  uint64_t cells_per_instance;
  uint32_t n_consts;
} h2sha_compact_info_t;
int h2sha_get_compact_info(const h2sha_engine_t* e, h2sha_compact_info_t* out);
int h2sha_get_compact_map(h2sha_engine_t* e, uint32_t* gate_map, uint32_t* lookup_map, uint32_t* dense_map, uint32_t* spread_map, uint64_t* consts);
int h2sha_expand_compact(h2sha_engine_t* e, const void* dict_host, uint64_t n_instances, void* host_out, uint32_t rows_per_column, int zero_fill,
                         uint32_t n_threads);

/* ---- Lookup-argument pre-work on the witness in HBM (the step after assignment in create_proof) --------------------
 * The chip has two kinds of lookups, neither with a selector (every usable row is looked up):
 *   range lookup l  (l < n_range_lookups = n_lookup_cols): lookup advice column l against the table 0 .. 2^lookup_bits - 1
 *                   (halo2-base RangeConfig, lib.rs:409-418; filled by range.finalize, lib.rs:469);
 *   spread lookup c (index n_range_lookups + c, c < num_advice_columns): (denses[c], spreads[c]) against
 *                   (table_dense, table_spread) (spread.rs:53-62, 165-194).
 * halo2's lookup prover (halo2_proofs plonk/lookup/prover.rs, `permute_expression_pair`) needs per lookup A' = the
 * (compressed) input column sorted and S' = the table column permuted so that A'[i] == S'[i] or A'[i] == A'[i-1].
 * Never-assigned advice rows hold 0; table columns are padded with their first row.  `usable_rows` = 2^k - (blinding
 * factors + 1); the trailing blinding rows are random and stay with the prover. */
typedef struct {
  uint32_t n_range_lookups, n_spread_lookups;
  uint32_t range_table_rows, spread_table_rows;   /* 2^lookup_bits, 2^num_bits_lookup                                    */
  uint32_t min_usable_rows;                       /* largest assigned lookup / spread column or table                     */
  uint64_t mult_words_per_instance;               /* n_range_lookups * range_table_rows + n_spread_lookups * spread_table_rows */
} h2sha_lookup_info_t;
int h2sha_get_lookup_info(const h2sha_engine_t* e, h2sha_lookup_info_t* out);

/* Challenge-independent half: how often each table row is hit by the first `usable_rows` rows of each lookup's input.
 *   mult_dev [n_instances][mult_words_per_instance] u32 (device): range lookups first ([l][2^lookup_bits]), then the spread
 *   lookups ([c][2^num_bits_lookup]).  `lookup` / `spread` are the batch buffers of h2sha_digest_batch; one of them may be
 *   NULL (its half of mult_dev is left untouched).  not_in_table_dev (device u32, may be NULL) counts cells that are no
 *   table row (a witness the lookup argument would reject).  Asynchronous on `stream`. */
int h2sha_lookup_multiplicities(h2sha_engine_t* e, uint64_t n_instances, const void* lookup, const void* spread, uint32_t usable_rows,
                                uint32_t* mult_dev, uint32_t* not_in_table_dev, void* stream);

/* Permuted pair of lookup `lookup_idx` for every instance: permuted_input_dev / permuted_table_dev [n_instances][usable_rows]
 * Fr (Montgomery, device).  theta_mont (host, 4 x u64 Montgomery) compresses the two expressions of a spread lookup
 * (dense * theta + spread); NULL for range lookups (one expression).  errors_dev (device u32, may be NULL) is incremented
 * for every instance whose multiplicities do not sum to usable_rows (its rows are then not written). */
int h2sha_permute_lookup(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows,
                         const uint64_t* theta_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream);

/* The same permuted pair straight from the raw value lists of the last batch generated with keep_lookup_raw (or lookup_mult_dev):
 * instances [first_instance, first_instance + n_instances) of that batch.  The multiplicities of the one lookup are binned into the
 * engine's workspace (L2-resident) right before the scan; no dense multiplicity array is ever written to or read from HBM. */
int h2sha_permute_lookup_from_raw(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, uint32_t lookup_idx, uint32_t usable_rows,
                                  const uint64_t* theta_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream);

/* The grand-product column z of lookup `lookup_idx` for every instance, once beta and gamma are drawn (halo2_proofs
 * plonk/lookup/prover.rs `Permuted::commit_product`), with A / S the (theta-compressed) input and table expressions and
 * A' / S' the permuted pair:
 *   u_i = (A[i] + beta)(S[i] + gamma),  v_i = (A'[i] + beta)(S'[i] + gamma),  z[0] = 1,  z[j+1] = z[j] * u_j / v_j,  j < usable_rows.
 * A row with v_i = 0 has the fraction 0 (ff's batch_invert leaves a zero as zero), so every later z is 0.
 *   lookup / spread        the batch buffers of h2sha_digest_batch; only the one this lookup reads is needed (the other may be NULL)
 *   permuted_input_dev / permuted_table_dev   [n_instances][usable_rows] Fr (device): A', S', e.g. from h2sha_permute_lookup
 *   theta_mont / beta_mont / gamma_mont       host, 4 x u64 Montgomery, reduced (< p) or H2SHA_EINVAL; theta only for spread lookups
 *   z_dev                  [n_instances][usable_rows + 1] Fr (device): z[0 .. usable_rows]; the blinding rows after them are the prover's
 *   errors_dev             device u32, may be NULL: incremented for every instance whose z[usable_rows] != 1 (A', S' are then no
 *                          permutation of the input and table expressions, or a denominator was 0)
 * Instance i of the four device buffers belongs together: a slice of a batch is passed by offsetting all of them.  Fr buffers
 * must be 32-byte aligned.  Every num_bits_lookup works (the table's compressed values are computed per call).  Asynchronous on
 * `stream`. */
int h2sha_lookup_product(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                         const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows,
                         const uint64_t* theta_mont, const uint64_t* beta_mont, const uint64_t* gamma_mont,
                         void* z_dev, uint32_t* errors_dev, void* stream);

/* ---- Permutation argument (copy constraints): halo2_proofs plonk/permutation ------------------------------------------
 * The columns with equality enabled, in the order of `cs.permutation.columns` (the order of the enable_equality calls), as
 * (kind, index) pairs.  Kinds are numbered like chip::ColumnKind (csrc/chip_api.hpp); the instance column is new. */
#define H2SHA_COL_GATE 0u      /* gate advice column `index` (< n_gate_cols)                                       */
#define H2SHA_COL_LOOKUP 1u    /* lookup advice column `index` (< n_lookup_cols)                                   */
#define H2SHA_COL_DENSE 2u     /* SpreadConfig denses[index] (< num_advice_columns)                                */
#define H2SHA_COL_SPREAD 3u    /* SpreadConfig spreads[index]                                                      */
#define H2SHA_COL_FIXED 4u     /* fixed (constants) column `index` (< num_fixed)                                   */
#define H2SHA_COL_INSTANCE 6u  /* the instance column (index 0) the output bytes are bound to                      */
typedef struct {
  uint32_t n_columns;
  const uint32_t* columns;      /* [n_columns][2] (kind, index): every column the chip copies from or to, each once        */
  uint32_t num_fixed;           /* fixed columns Context::assign_fixed fills round-robin (constant k -> column k % num_fixed,
                                   row k / num_fixed); 0 -> 1                                                            */
  uint32_t columns_per_chunk;   /* cs.degree() - 2: columns per product column z                                          */
  uint32_t bind_output_bytes;   /* 1: constrain_instance(output_bytes[i], instance, i) for the 32 * n_digests output bytes
                                   in order (the reference's TestCircuit, lib.rs:480-482); the list then has the instance
                                   column, and only then                                                                 */
  uint32_t k;                   /* domain size 2^k; 0 -> the smallest 2^k > usable_rows + 1                              */
} h2sha_perm_desc_t;

/* Keygen half: the permutation mapping halo2's `permutation::keygen::Assembly` builds from the chip's copy constraints, replayed
 * in the order the chip API issues them (chip_api.hpp `assign_digest`: per digest() call its shape copies, then per spread limb
 * the dense and the spread copy; then range.finalize's lookup copies; then the instance binding).  Region rows = circuit rows
 * (the region starts at row 0).  mapping: [n_columns][usable_rows][2] u32 (column position in desc->columns, row), or NULL to
 * validate only.  sigma_c(w^r) = delta^c' w^r' with (c', r') = mapping[c][r].  Works on a plan-only engine (device = -1); needs
 * build_shape.  H2SHA_EINVAL when a column the chip copies is missing, a column is listed twice or out of range, an assigned
 * cell lies at or above usable_rows, or columns_per_chunk == 0. */
int h2sha_get_permutation(h2sha_engine_t* e, const h2sha_perm_desc_t* desc, uint32_t usable_rows, uint32_t* mapping);

/* The permutation argument's product columns for every instance, once beta and gamma are drawn (halo2_proofs
 * plonk/permutation/prover.rs `Argument::commit` without the blinding rows): chunk h covers columns [h*m, min(C, (h+1)*m)),
 * m = columns_per_chunk, and with one deltaomega running over all columns,
 *   z_h[0] = z_{h-1}[U] (1 for h = 0),  z_h[i+1] = z_h[i] * prod_j (p_j(w^i) + beta delta^j w^i + gamma) / prod_j (p_j(w^i) + beta sigma_j(w^i) + gamma)
 * for i < U = usable_rows.  A zero denominator gives the fraction 0 (ff's batch_invert leaves a zero as zero), so the rest of
 * that chunk and every later chunk is 0.  The fixed column holds the shape's constants at their round-robin rows and 0 elsewhere;
 * the instance column holds byte i of the instance's digests at row i and 0 above.
 *   gate / lookup / spread    the batch buffers of h2sha_digest_batch (each may be NULL when no listed column reads it)
 *   digests_dev               device [n_instances * n_digests][32]; needed only with bind_output_bytes
 *   beta_mont / gamma_mont    host, 4 x u64 Montgomery, reduced (< p) or H2SHA_EINVAL
 *   z_dev                     [n_instances][n_chunks][usable_rows + 1] Fr (device, 32-byte aligned), n_chunks = ceil(C / m)
 *   errors_dev                device u32, may be NULL: incremented for every instance whose last chunk ends with z[U] != 1
 * Only cells whose sigma is not the identity enter the products; a cell with sigma = id contributes exactly 1.  The one departure
 * from halo2: a zero term p + beta delta^j w^i + gamma at such a cell (probability ~2^-230 over beta, gamma) is taken as 1 where
 * halo2 would zero the fraction.  The moved cells are planned once per (desc, usable_rows) and kept on the device.  Asynchronous
 * on `stream` after the first call for a desc. */
int h2sha_permutation_product(h2sha_engine_t* e, uint64_t n_instances, const h2sha_perm_desc_t* desc, uint32_t usable_rows,
                              const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                              const uint64_t* beta_mont, const uint64_t* gamma_mont, void* z_dev, uint32_t* errors_dev, void* stream);

/* ---- Per-instance challenges ---------------------------------------------------------------------------------------------
 * The four calls above take one theta / beta / gamma for the whole batch: right when the batch holds the circuits of ONE
 * create_proof over many circuits.  A batch of independent proofs (one per message or request) has one transcript, and so one
 * (theta_i, beta_i, gamma_i), per instance; these four calls take them, at batch speed:
 *   thetas_mont / betas_mont / gammas_mont   host [n_instances][4] u64 Montgomery; row i belongs to instance i of the call (for
 *                          from_raw: instance first_instance + i, like the output rows).  Every row must be reduced (< p), or the
 *                          call returns H2SHA_EINVAL naming the row.  thetas_mont may be NULL for a range lookup.  The rows are
 *                          staged before the call returns (the caller may reuse the arrays at once); the call stays asynchronous.
 *   errors_dev             device [n_instances] u32, or NULL: entry i is incremented (never zeroed) when instance i fails for a
 *                          reason that increments the shared calls' single counter, and, for the permuted pair of a spread lookup,
 *                          when theta_i makes two compressed table rows equal (the shared call refuses such a theta with
 *                          H2SHA_EINVAL; here only that instance is counted and its A', S' rows are left unwritten).
 * Every other argument is that of the matching shared call.  For every instance the outputs are bit-identical to the shared call
 * on that instance alone with row i's challenges; with all rows equal they are bit-identical to the shared call on the batch, and
 * the per-instance errors sum to its counter.  A slice of a batch is passed by offsetting every pointer, the challenge arrays too.
 * The spread table of each instance is compressed, sorted by canonical value and checked on the device. */
int h2sha_permute_lookup_per_instance(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const uint32_t* mult_dev, uint32_t usable_rows,
                                      const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream);
int h2sha_permute_lookup_from_raw_per_instance(h2sha_engine_t* e, uint64_t first_instance, uint64_t n_instances, uint32_t lookup_idx, uint32_t usable_rows,
                                               const uint64_t* thetas_mont, void* permuted_input_dev, void* permuted_table_dev, uint32_t* errors_dev, void* stream);
int h2sha_lookup_product_per_instance(h2sha_engine_t* e, uint64_t n_instances, uint32_t lookup_idx, const void* lookup, const void* spread,
                                      const void* permuted_input_dev, const void* permuted_table_dev, uint32_t usable_rows,
                                      const uint64_t* thetas_mont, const uint64_t* betas_mont, const uint64_t* gammas_mont,
                                      void* z_dev, uint32_t* errors_dev, void* stream);
int h2sha_permutation_product_per_instance(h2sha_engine_t* e, uint64_t n_instances, const h2sha_perm_desc_t* desc, uint32_t usable_rows,
                                           const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                                           const uint64_t* betas_mont, const uint64_t* gammas_mont, void* z_dev, uint32_t* errors_dev, void* stream);

/* MockProver-style check of a whole batch where it lies, in HBM -- what the reference's tests accept a witness by
 * (`MockProver::run(..).verify() == Ok(())`, lib.rs:525-526), for every instance instead of one:
 *   violations[0] gates           q * (a + b*c - d) = 0 on every enabled gate row (halo2-base FlexGate, Vertical)
 *   violations[1] copies          the chip's copy constraints (cell <-> cell, cell <-> fixed constant), the lookup-column cells
 *                                 against the cells range.finalize copies (lib.rs:469), the spread-column cells against their gate
 *                                 cells (spread.rs:209-227)
 *   violations[2] range lookups   lookup-column cells that are not < 2^lookup_bits
 *   violations[3] spread lookups  (dense, spread) pairs that are no row of the spread table (spread.rs:53-62,165-194)
 *   violations[4] digest bytes    output-byte cells (lib.rs:311-341) that differ from digests_dev [n_msgs][32] (skipped when NULL)
 * `violations_host` gets the five counters; the call synchronises `stream`.  The static shape is built on first use. */
int h2sha_check_batch(h2sha_engine_t* e, uint64_t n_instances, const void* gate, const void* lookup, const void* spread, const uint8_t* digests_dev,
                      uint64_t* violations_host, void* stream);

/* The same check with a verdict per instance, for batches of independent proofs and for finding a wrong cell:
 *   counts_dev  device [n_instances][5] u32: instance i's violations per class, classes and order of h2sha_check_batch
 *   first_dev   device [n_instances][5] u32, or NULL: the smallest failing item number (below) per class, 0xFFFFFFFF when none fails
 * Both arrays are overwritten, never accumulated into.  Asynchronous on `stream`; the static shape is built on first use.
 * Summed over the instances, counts_dev equals h2sha_check_batch's counters.  A slice of a batch is passed by offsetting every pointer.
 *
 * Item numbers, per instance (the cells of an item are what h2sha_check_site returns):
 *   class 0 gates          item i = the i-th enabled selector in gate-stream order; 4 cells: gate-stream indices s .. s+3
 *   class 1 copies         first the n_copies copies of h2sha_get_shape, in its order; then one item per lookup cell k (the lookup
 *                          cell against lookup_src[k], range.finalize); then two items per spread limb n (the dense cell against
 *                          limb_dense_src[n], then the spread cell against limb_spread_src[n]); 2 cells each.  A fixed constant k is
 *                          the cell (H2SHA_COL_FIXED, 0, k): row k of the single fixed column the check assumes
 *   class 2 range lookups  item k = lookup cell k in cells_to_lookup order; 1 cell (its column is the lookup_idx of the range lookup)
 *   class 3 spread lookups item n = spread limb n; 2 cells, the dense and the spread cell of column pair n % num_advice_columns
 *                          (lookup_idx n_range_lookups + n % num_advice_columns)
 *   class 4 digest bytes   item d * 32 + j = output byte j of digest() call d; 1 cell, the output-byte gate cell */
int h2sha_check_batch_per_instance(h2sha_engine_t* e, uint64_t n_instances, const void* gate, const void* lookup, const void* spread,
                                   const uint8_t* digests_dev, uint32_t* counts_dev, uint32_t* first_dev, void* stream);

/* The cells check item `item` of class `check_class` reads, as halo2's MockProver names a failure's place (VerifyFailure): cell c is
 * column (kind[c], index[c]) -- kinds H2SHA_COL_* -- at row[c]; the region starts at row 0.  Host only: works on a plan-only engine
 * and builds the shape on first use when the engine was made without build_shape.  H2SHA_EINVAL for a class >= 5 or an item
 * beyond the class. */
typedef struct {
  uint32_t n_cells;
  uint32_t kind[4], index[4], row[4];
} h2sha_check_site_t;
int h2sha_check_site(h2sha_engine_t* e, uint32_t check_class, uint32_t item, h2sha_check_site_t* out);

/* The only collective of the path: all-gather of digests [n_instances_per_rank * n_digests][32] and per-instance checksums
 * [n_instances_per_rank][4] over the caller's communicator (`ncclComm_t`, one per GPU/rank; inside an ncclGroup when one
 * thread drives several GPUs).  Receive buffers hold n_ranks x the send size, rank-major.  Either pair may be NULL.
 * NCCL is loaded at run time (libnccl.so.2); the library itself links only the CUDA runtime. */
int h2sha_gather(void* nccl_comm, uint64_t n_instances_per_rank, uint32_t n_digests, const uint8_t* digests_dev, const uint64_t* checksums_dev,
                 uint8_t* all_digests_dev, uint64_t* all_checksums_dev, void* stream);

/* Zero-fill output buffers (or just the never-assigned ranges when only_unassigned != 0). */
int h2sha_zero_outputs(h2sha_engine_t* e, uint64_t n_instances, void* gate, void* lookup, void* spread, int only_unassigned, void* stream);

/* Checksum definition (so a consumer can re-verify): for every assigned cell at position `pos` (Fr index inside the
 * instance's buffer of that kind) with 32-bit limbs x[0..8):  h = sum_k x[k] * H2SHA_CK_M[k] mod 2^32;
 * checksum += (u64)h * (u32)(2*pos+1)  mod 2^64. */
extern const uint32_t H2SHA_CK_M[8];

/* Test hook: Montgomery form of n raw u64 values (device pointers), through the same device function the
 * expansion kernel uses.  out: [n][4] u64. */
int h2sha_debug_mont_from_u64(h2sha_engine_t* e, const uint64_t* vals_dev, uint64_t* out_dev, uint64_t n, void* stream);
/* Same for the 32-bit fast path (the low 32 bits of each value are converted). */
int h2sha_debug_mont_from_u32(h2sha_engine_t* e, const uint64_t* vals_dev, uint64_t* out_dev, uint64_t n, void* stream);

/* Measurement hook: overwrite `bytes` of device memory with incompressible 32-byte cells by plain coalesced 256-bit stores
 * (no shared memory, no arithmetic) -- the write-bandwidth ceiling bench.py reports next to the expansion kernel. */
int h2sha_debug_store_probe(h2sha_engine_t* e, void* buf_dev, uint64_t bytes, void* stream);

/* Measurement hook for the other roofline the path could hit: `iters` x 16 dependent-chain integer instructions (8 IMAD +
 * 8 LOP3 over 8 independent chains) per thread on n_sms * 8 CTAs of 256 threads, no memory traffic.  scratch_dev: device
 * buffer of n_sms * 8 * 256 u32 (practically never written).  *thread_instructions = integer instructions the launch executes. */
int h2sha_debug_int_probe(h2sha_engine_t* e, uint32_t* scratch_dev, uint32_t iters, uint64_t* thread_instructions, void* stream);

/* Kernel launch statistics of the last h2sha_digest_batch (for bench.py's gpu_launches). */
int h2sha_last_launch_count(const h2sha_engine_t* e);
/* Device time of the two kernels of the last batch run with time_kernels = 1; synchronises on the recorded events. */
int h2sha_last_kernel_ms(h2sha_engine_t* e, float* trace_ms, float* expand_ms);

#ifdef __cplusplus
}
#endif
#endif /* H2SHA_B200_H */
