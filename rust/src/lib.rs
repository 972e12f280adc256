//! Drop-in for `halo2_dynamic_sha256::Sha256DynamicConfig` (reference src/lib.rs:38-369) whose cell values come from
//! the B200 engine (`libh2sha_b200.so`, C-ABI `include/h2sha_b200.h`).
//!
//! SOURCE ONLY.  The build image has no cargo/rustc and no network, so this crate has never been compiled; the SAME design
//! is implemented and tested in C++ (`halo2-dynamic-sha256_b200/csrc/chip_api.hpp`, `tests/test_gpu_chip_api.py`: the
//! reference's TestCircuit replayed into a recording region and accepted by the MockProver-style checker).  What a
//! maintainer has to check on the first `cargo build` is marked `CHECK:` below (field names of halo2-base @ 40ba7e3).
//!
//! Public API = the reference's, signature for signature:
//!   configure(meta, max_variable_byte_sizes, range, num_bits_lookup, num_advice_columns, is_input_range_check)  lib.rs:49-56
//!   digest(&mut self, ctx, input, precomputed_input_len) -> Result<AssignedHashResult<F>, Error>                lib.rs:71-76
//!   new_context(&self, region) -> Context<F>                                                                    lib.rs:351-360
//!   range(&self) -> &RangeConfig<F>                                                                             lib.rs:362-364
//!   load(&self, layouter) -> Result<(), Error>                                                                  lib.rs:366-368
//! `digest` assigns exactly the cells the reference's `digest` would assign, at the same (column, row), by replaying the
//! engine's static shape (selectors, fixed cells, copy constraints: `h2sha_get_shape`) and the exported columns of the
//! region (`h2sha_export_instance`).  `range.finalize(ctx)` stays halo2-base's own: `digest` pushes the looked-up cells
//! into `ctx.cells_to_lookup` in the reference's order.
#![allow(non_camel_case_types, dead_code)]
include!(concat!(env!("OUT_DIR"), "/bindings.rs"));

use std::ffi::CStr;
use std::marker::PhantomData;

use halo2_base::gates::range::RangeConfig;
use halo2_base::halo2_proofs::{
    circuit::{Cell, Layouter, Region, Value},
    halo2curves::bn256::Fr,
    plonk::{Advice, Any, Column, ConstraintSystem, Error, Instance, TableColumn},
    poly::Rotation,
};
use halo2_base::{AssignedValue, Context, ContextParams};

pub const NUM_ROUND: usize = 64; // compression.rs:990
pub const NUM_STATE_WORD: usize = 8; // compression.rs:991
pub const INIT_STATE: [u32; 8] = [0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19]; // compression.rs:1003-1012

fn engine_err(rc: i32) -> Error {
    let msg = unsafe { CStr::from_ptr(h2sha_last_error()) }.to_string_lossy().into_owned();
    if rc == H2SHA_EPANIC {
        panic!("{msg}"); // the reference panics on these inputs (lib.rs:89-90)
    }
    eprintln!("h2sha engine error {rc}: {msg}");
    Error::Synthesis
}
fn check(rc: i32) -> Result<(), Error> {
    if rc == H2SHA_OK as i32 { Ok(()) } else { Err(engine_err(rc)) }
}

#[derive(Debug, Clone)]
pub struct AssignedHashResult { // lib.rs:31-36
    pub input_len: AssignedValue<Fr>,
    pub input_bytes: Vec<AssignedValue<Fr>>,
    pub output_bytes: Vec<AssignedValue<Fr>>,
}

/// The columns `SpreadConfig::configure` creates (spread.rs:32-74), in the same order, with the same lookups.
#[derive(Debug, Clone)]
struct SpreadColumns {
    denses: Vec<Column<Advice>>,
    spreads: Vec<Column<Advice>>,
    table_dense: TableColumn,
    table_spread: TableColumn,
    num_bits_lookup: usize,
}

/// The static plan of one configuration, fetched once through the C-ABI.
struct Shape {
    layout: h2sha_layout_t,
    breaks: Vec<u32>,
    selectors: Vec<u8>,
    copies: Vec<[u32; 4]>,
    fixed: Vec<[u64; 4]>,
    lookup_src: Vec<u32>,
    limb_dense_src: Vec<u32>,
    limb_spread_src: Vec<u32>,
    /// per digest: [gate_lo, gate_hi), [lookup_lo, lookup_hi), [limb_lo, limb_hi) of the stream ranges its `digest` call owns
    ranges: Vec<[u32; 6]>,
}

pub struct Sha256DynamicConfig {
    pub max_variable_byte_sizes: Vec<usize>, // lib.rs:40
    range: RangeConfig<Fr>,
    spread: SpreadColumns,
    pub cur_hash_idx: usize, // lib.rs:43
    is_input_range_check: bool,
    engine: *mut h2sha_engine_t,
    shape: std::rc::Rc<Shape>,
    inputs: Vec<Vec<u8>>,
    pre_lens: Vec<u32>,
    /// halo2 cells of the gate stream assigned so far in the current Context (index = gate-stream index)
    cells: Vec<AssignedValue<Fr>>,
    fixed_cells: Vec<Option<Cell>>,
    /// witness taken from a batch generated earlier: (gate, lookup, spread device pointers, instance)
    attached: Option<(u64, u64, u64, u64)>,
    _f: PhantomData<Fr>,
}

impl Sha256DynamicConfig {
    const ONE_ROUND_INPUT_BYTES: usize = 64; // lib.rs:48

    /// lib.rs:49-69.  CUDA device: `H2SHA_DEVICE` (default 0; -1 = plan only, for keygen on a machine without a GPU).
    pub fn configure(
        meta: &mut ConstraintSystem<Fr>,
        max_variable_byte_sizes: Vec<usize>,
        range: RangeConfig<Fr>,
        num_bits_lookup: usize,
        num_advice_columns: usize,
        is_input_range_check: bool,
    ) -> Self {
        for byte in max_variable_byte_sizes.iter() {
            debug_assert_eq!(byte % Self::ONE_ROUND_INPUT_BYTES, 0); // lib.rs:57-59
        }
        // SpreadConfig::configure (spread.rs:32-74): same column allocation order, same lookups
        debug_assert_eq!(16 % num_bits_lookup, 0);
        let mk = |meta: &mut ConstraintSystem<Fr>| {
            let c = meta.advice_column();
            meta.enable_equality(c);
            c
        };
        let denses: Vec<_> = (0..num_advice_columns).map(|_| mk(meta)).collect();
        let spreads: Vec<_> = (0..num_advice_columns).map(|_| mk(meta)).collect();
        let table_dense = meta.lookup_table_column();
        let table_spread = meta.lookup_table_column();
        for (dense, spread) in denses.iter().zip(spreads.iter()) {
            meta.lookup("spread lookup", |meta| {
                let dense = meta.query_advice(*dense, Rotation::cur());
                let spread = meta.query_advice(*spread, Rotation::cur());
                vec![(dense, table_dense), (spread, table_spread)]
            });
        }
        let device: i32 = std::env::var("H2SHA_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        let sizes: Vec<u32> = max_variable_byte_sizes.iter().map(|&x| x as u32).collect();
        let cfg = h2sha_config_t {
            n_digests: sizes.len() as u32,
            max_variable_byte_sizes: sizes.as_ptr(),
            max_rows: range.gate.max_rows as u32, // lib.rs:355
            lookup_bits: range.lookup_bits as u32,
            num_bits_lookup: num_bits_lookup as u32,
            num_advice_columns: num_advice_columns as u32,
            is_input_range_check: is_input_range_check as u32,
            gate_col_rows: 0,
            lookup_col_rows: 0,
            spread_rows: 0,
            device,
            build_shape: 1,
            block_parts: 0,
            num_lookup_advice: range.lookup_advice.iter().map(|v| v.len()).sum::<usize>() as u32, // CHECK: RangeConfig.lookup_advice
        };
        let mut engine = std::ptr::null_mut();
        let rc = unsafe { h2sha_create(&cfg, &mut engine) };
        assert_eq!(rc, H2SHA_OK as i32, "{}", unsafe { CStr::from_ptr(h2sha_last_error()) }.to_string_lossy());
        let shape = Self::fetch_shape(engine, &sizes);
        // the plan needs this many FlexGate advice columns; halo2-base would panic "NOT ENOUGH ADVICE COLUMNS" later
        assert!(shape.layout.n_gate_cols as usize <= range.gate.basic_gates[0].len(), "NOT ENOUGH ADVICE COLUMNS"); // CHECK: FlexGateConfig.basic_gates
        Self {
            max_variable_byte_sizes,
            range,
            spread: SpreadColumns { denses, spreads, table_dense, table_spread, num_bits_lookup },
            cur_hash_idx: 0,
            is_input_range_check,
            engine,
            shape: std::rc::Rc::new(shape),
            inputs: vec![],
            pre_lens: vec![],
            cells: vec![],
            fixed_cells: vec![],
            attached: None,
            _f: PhantomData,
        }
    }

    fn fetch_shape(engine: *mut h2sha_engine_t, sizes: &[u32]) -> Shape {
        unsafe {
            let mut layout: h2sha_layout_t = std::mem::zeroed();
            h2sha_get_layout(engine, &mut layout);
            let mut breaks = vec![0u32; layout.n_gate_cols as usize];
            h2sha_get_breaks(engine, breaks.as_mut_ptr());
            let mut selectors = vec![0u8; layout.n_gate_cells as usize];
            let mut copies = vec![[0u32; 4]; layout.n_copies as usize];
            let mut fixed = vec![[0u64; 4]; layout.n_fixed as usize];
            let mut lookup_src = vec![0u32; layout.n_lookup_cells as usize];
            let mut limb_dense_src = vec![0u32; layout.n_spread_limbs as usize];
            let mut limb_spread_src = vec![0u32; layout.n_spread_limbs as usize];
            h2sha_get_shape(engine, selectors.as_mut_ptr(), copies.as_mut_ptr() as *mut u32, fixed.as_mut_ptr() as *mut u64, lookup_src.as_mut_ptr(),
                            limb_dense_src.as_mut_ptr(), limb_spread_src.as_mut_ptr());
            let mut ranges = vec![[0u32; 6]; sizes.len()];
            h2sha_get_digest_ranges(engine, ranges.as_mut_ptr() as *mut u32);
            Shape { layout, breaks, selectors, copies, fixed, lookup_src, limb_dense_src, limb_spread_src, ranges }
        }
    }

    /// lib.rs:351-360
    pub fn new_context<'a, 'b>(&'b self, region: Region<'a, Fr>) -> Context<'a, Fr> {
        Context::new(region, ContextParams { max_rows: self.range.gate.max_rows, num_context_ids: 1, fixed_columns: self.range.gate.constants.clone() })
    }
    /// lib.rs:362-364
    pub fn range(&self) -> &RangeConfig<Fr> { &self.range }
    /// lib.rs:366-368 -> SpreadConfig::load (spread.rs:165-194)
    pub fn load(&self, layouter: &mut impl Layouter<Fr>) -> Result<(), Error> {
        let n = 1usize << self.spread.num_bits_lookup;
        let (mut dense, mut spread) = (vec![0u64; n], vec![0u64; n]);
        let (mut ns, mut nr) = (0u32, 0u32);
        check(unsafe { h2sha_get_lookup_tables(self.engine, dense.as_mut_ptr(), spread.as_mut_ptr(), &mut ns, &mut nr) })?;
        layouter.assign_table(|| "spread table", |mut table| {
            for i in 0..n {
                table.assign_cell(|| "table_dense", self.spread.table_dense, i, || Value::known(Fr::from(dense[i])))?;
                table.assign_cell(|| "table_spread", self.spread.table_spread, i, || Value::known(Fr::from(spread[i])))?;
            }
            Ok(())
        })
    }

    /// Prover path: take the region's witness from a batch generated earlier with `h2sha_digest_batch` (device pointers).
    pub fn attach(&mut self, gate: u64, lookup: u64, spread: u64, instance: u64) { self.attached = Some((gate, lookup, spread, instance)); }

    /// lib.rs:71-349: same preconditions and panics, same cells at the same (column,row), same `cur_hash_idx` advance.
    pub fn digest<'a>(&mut self, ctx: &mut Context<'a, Fr>, input: &[u8], precomputed_input_len: Option<usize>) -> Result<AssignedHashResult, Error> {
        let d = self.cur_hash_idx;
        let max_variable_byte_size = self.max_variable_byte_sizes[d]; // lib.rs:86 (index panic like the reference)
        let precomputed_input_len = precomputed_input_len.unwrap_or(0); // lib.rs:88
        assert_eq!(precomputed_input_len % Self::ONE_ROUND_INPUT_BYTES, 0); // lib.rs:89
        let padded_size = (input.len() + 9 + 63) / 64 * 64; // lib.rs:80-85
        assert!(padded_size - precomputed_input_len <= max_variable_byte_size); // lib.rs:90
        let sh = self.shape.clone();
        let lay = &sh.layout;
        // ---- values: this region with the inputs known so far (later digests: the empty message, replaced when their turn comes) ----
        let k_rows = (self.range.gate.max_rows as usize).next_power_of_two(); // rows per column = 2^k (max_rows = 2^k - minimum_rows)
        let n_cols = (lay.n_gate_cols + lay.n_lookup_cols + lay.n_spread_cols) as usize;
        let mut cols: Vec<Vec<u64>> = vec![vec![0u64; k_rows * 4]; n_cols];
        {
            self.inputs.truncate(d);
            self.pre_lens.truncate(d);
            self.inputs.push(input.to_vec());
            self.pre_lens.push(precomputed_input_len as u32);
            let ptrs: Vec<*mut u64> = cols.iter_mut().map(|c| c.as_mut_ptr()).collect();
            let dev = cudarc::driver::CudaDevice::new(0).map_err(|_| Error::Synthesis)?;
            let (gate, lookup, spread, inst, _keep) = match self.attached {
                Some((g, l, s, i)) => (g, l, s, i, None),
                None => {
                    let g = dev.alloc_zeros::<u64>(lay.gate_bytes as usize / 8).map_err(|_| Error::Synthesis)?;
                    let l = dev.alloc_zeros::<u64>(lay.lookup_bytes as usize / 8).map_err(|_| Error::Synthesis)?;
                    let s = dev.alloc_zeros::<u64>(lay.spread_bytes as usize / 8).map_err(|_| Error::Synthesis)?;
                    let (mut blob, mut offs, mut lens, mut pre) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
                    for k in 0..self.max_variable_byte_sizes.len() {
                        offs.push(blob.len() as u64);
                        let m: &[u8] = if k <= d { &self.inputs[k] } else { &[] };
                        lens.push(m.len() as u32);
                        pre.push(if k <= d { self.pre_lens[k] } else { 0 });
                        blob.extend_from_slice(m);
                    }
                    use cudarc::driver::DevicePtr;
                    let (gp, lp, sp) = (*g.device_ptr(), *l.device_ptr(), *s.device_ptr());
                    let batch = h2sha_batch_t {
                        n_instances: 1, msgs: blob.as_ptr(), msgs_on_device: 0, msgs_bytes: blob.len() as u64, offsets: offs.as_ptr(), lens: lens.as_ptr(),
                        precomputed_lens: pre.as_ptr(), gate: gp as *mut _, lookup: lp as *mut _, spread: sp as *mut _,
                        only_digest: d as u32 + 1, // only the cells this digest() call owns
                        ..unsafe { std::mem::zeroed() }
                    };
                    check(unsafe { h2sha_digest_batch(self.engine, &batch) })?;
                    (gp, lp, sp, 0u64, Some((g, l, s)))
                }
            };
            check(unsafe { h2sha_export_instance(self.engine, inst, gate as *const _, lookup as *const _, spread as *const _, ptrs.as_ptr(), k_rows as u32, std::ptr::null_mut()) })?;
            dev.synchronize().map_err(|_| Error::Synthesis)?;
        }
        let fr_at = |col: usize, row: usize| -> Fr {
            let l = &cols[col][row * 4..row * 4 + 4];
            Fr::from_raw_montgomery([l[0], l[1], l[2], l[3]]) // CHECK: halo2curves constructor from Montgomery limbs (Fr([u64;4]) is pub(crate) in some versions)
        };
        let gate_pos = |idx: u32| -> (usize, usize) {
            let c = sh.breaks.partition_point(|&b| b <= idx) - 1;
            (c, (idx - sh.breaks[c]) as usize)
        };
        let [g_lo, g_hi, l_lo, l_hi, m_lo, m_hi] = sh.ranges[d];
        // ---- (1) this digest's gate cells, stream order, + selectors (Context::assign_region of halo2-base) ----
        if d == 0 { self.cells.clear(); self.fixed_cells = vec![None; sh.fixed.len()]; }
        for idx in g_lo..g_hi {
            let (c, row) = gate_pos(idx);
            let gate_cfg = &self.range.gate.basic_gates[0][c]; // CHECK: BasicGateConfig { q_enable, value }
            let v = fr_at(c, row);
            let cell = ctx.region.assign_advice(|| "", gate_cfg.value, row, || Value::known(v))?;
            if sh.selectors[idx as usize] != 0 { gate_cfg.q_enable.enable(&mut ctx.region, row)?; }
            self.cells.push(AssignedValue { cell: cell.cell(), value: Value::known(v), row_offset: row, context_id: 0 }); // CHECK: AssignedValue fields
        }
        // ---- (2) copy constraints recorded while these cells were emitted; fixed cells on first use (Context::assign_fixed) ----
        let n_fixed_cols = self.range.gate.constants.len();
        for cp in sh.copies.iter().filter(|cp| cp[1] >= g_lo && cp[1] < g_hi) {
            let a = self.cells[cp[1] as usize].cell;
            let b = if cp[2] == 0 { self.cells[cp[3] as usize].cell } else {
                let k = cp[3] as usize;
                if self.fixed_cells[k].is_none() {
                    let f = sh.fixed[k];
                    let fc = ctx.region.assign_fixed(|| "", self.range.gate.constants[k % n_fixed_cols], k / n_fixed_cols, || Value::known(Fr::from_raw(f)))?;
                    self.fixed_cells[k] = Some(fc.cell());
                }
                self.fixed_cells[k].unwrap()
            };
            ctx.region.constrain_equal(a, b)?;
        }
        // ---- (3) spread-table columns (spread.rs:202-231) ----
        let nc = self.spread.denses.len();
        for n in m_lo as usize..m_hi as usize {
            let (col, row) = (n % nc, n / nc);
            let base = (lay.n_gate_cols + lay.n_lookup_cols) as usize;
            let dc = ctx.region.assign_advice(|| "dense", self.spread.denses[col], row, || Value::known(fr_at(base + col, row)))?;
            ctx.region.constrain_equal(dc.cell(), self.cells[sh.limb_dense_src[n] as usize].cell)?;
            let sc = ctx.region.assign_advice(|| "spread", self.spread.spreads[col], row, || Value::known(fr_at(base + nc + col, row)))?;
            ctx.region.constrain_equal(sc.cell(), self.cells[sh.limb_spread_src[n] as usize].cell)?;
        }
        // ---- (4) looked-up cells, push order: halo2-base's own range.finalize(ctx) copies them into the lookup column (lib.rs:469) ----
        for k in l_lo..l_hi { ctx.cells_to_lookup.push(self.cells[sh.lookup_src[k as usize] as usize].clone()); }
        // ---- (5) Context bookkeeping, so that gates placed after this call continue where the reference's would ----
        let (c_end, r_end) = if g_hi == lay.n_gate_cells { gate_pos(g_hi - 1) } else { gate_pos(g_hi) };
        ctx.advice_alloc[0] = (c_end, if g_hi == lay.n_gate_cells { r_end + 1 } else { r_end }); // CHECK: Context.advice_alloc
        ctx.total_advice += (g_hi - g_lo) as usize;
        // ---- AssignedHashResult (lib.rs:342-346) ----
        let mut input_len_idx = 0u32;
        let mut in_idx = vec![0u32; max_variable_byte_size];
        let mut out_idx = vec![0u32; 32];
        check(unsafe { h2sha_get_handles(self.engine, d as u32, &mut input_len_idx, in_idx.as_mut_ptr(), out_idx.as_mut_ptr()) })?;
        let result = AssignedHashResult {
            input_len: self.cells[input_len_idx as usize].clone(),
            input_bytes: in_idx.iter().map(|&i| self.cells[i as usize].clone()).collect(),
            output_bytes: out_idx.iter().map(|&i| self.cells[i as usize].clone()).collect(),
        };
        self.cur_hash_idx += 1; // lib.rs:347
        Ok(result)
    }
}

impl Sha256DynamicConfig {
    /// The permutation argument's column list for `h2sha_perm_desc_t`: `meta`'s equality-enabled columns in the order of
    /// `cs.permutation.columns`, each as (H2SHA_COL_* kind, index) of the chip's columns; `instance` is the column the output bytes
    /// are bound to (`constrain_instance`), if any.  Panics on an equality column the chip does not own.
    pub fn permutation_columns(&self, meta: &ConstraintSystem<Fr>, instance: Option<Column<Instance>>) -> Vec<[u32; 2]> {
        let gates: Vec<Column<Any>> = self.range.gate.basic_gates[0].iter().map(|g| g.value.into()).collect(); // CHECK: BasicGateConfig.value
        let lookups: Vec<Column<Any>> = self.range.lookup_advice[0].iter().map(|c| (*c).into()).collect(); // CHECK: RangeConfig.lookup_advice
        let fixed: Vec<Column<Any>> = self.range.gate.constants.iter().map(|c| (*c).into()).collect(); // CHECK: FlexGateConfig.constants
        let denses: Vec<Column<Any>> = self.spread.denses.iter().map(|c| (*c).into()).collect();
        let spreads: Vec<Column<Any>> = self.spread.spreads.iter().map(|c| (*c).into()).collect();
        let inst: Option<Column<Any>> = instance.map(|c| c.into());
        meta.permutation().get_columns().into_iter() // CHECK: ConstraintSystem::permutation() / permutation::Argument::get_columns()
            .map(|col| {
                let pos = |v: &[Column<Any>]| v.iter().position(|c| *c == col).map(|i| i as u32);
                if let Some(i) = pos(&gates) { [H2SHA_COL_GATE, i] }
                else if let Some(i) = pos(&lookups) { [H2SHA_COL_LOOKUP, i] }
                else if let Some(i) = pos(&denses) { [H2SHA_COL_DENSE, i] }
                else if let Some(i) = pos(&spreads) { [H2SHA_COL_SPREAD, i] }
                else if let Some(i) = pos(&fixed) { [H2SHA_COL_FIXED, i] }
                else if inst == Some(col) { [H2SHA_COL_INSTANCE, 0] }
                else { panic!("equality-enabled column {col:?} is none of the chip's") }
            })
            .collect()
    }

    /// keygen `Assembly` mapping of the chip's copy constraints: per listed column and usable row, (column position, row).
    pub fn permutation_mapping(&self, desc: &h2sha_perm_desc_t, usable_rows: u32) -> Result<Vec<[u32; 2]>, Error> {
        let mut m = vec![[0u32; 2]; desc.n_columns as usize * usable_rows as usize];
        check(unsafe { h2sha_get_permutation(self.engine, desc, usable_rows, m.as_mut_ptr() as *mut u32) })?;
        Ok(m)
    }
}

impl Drop for Sha256DynamicConfig {
    fn drop(&mut self) { unsafe { h2sha_destroy(self.engine) } }
}

/// Batch side for provers that generate many regions up front (what the reference cannot do): thin, typed pass-throughs.
pub mod batch {
    use super::*;
    /// The path's only collective: all-gather of digests and per-instance checksums over the caller's `ncclComm_t`.
    pub fn gather(comm: *mut std::ffi::c_void, n_per_rank: usize, n_digests: u32, digests: u64, checksums: u64, all_digests: u64, all_checksums: u64,
                  stream: *mut std::ffi::c_void) -> Result<(), Error> {
        check(unsafe { h2sha_gather(comm, n_per_rank as u64, n_digests, digests as *const u8, checksums as *const u64, all_digests as *mut u8, all_checksums as *mut u64, stream) })
    }
    /// halo2 `permutation::prover` commit without the blinding rows, for every instance of a batch: z [n][n_chunks][usable_rows + 1]
    /// Fr at `z_dev`; beta / gamma as Montgomery limbs (the memory layout of halo2curves bn256::Fr).
    pub fn permutation_product(engine: *mut h2sha_engine_t, n: usize, desc: &h2sha_perm_desc_t, usable_rows: u32, gate: u64, lookup: u64, spread: u64,
                               digests_dev: u64, beta_mont: &[u64; 4], gamma_mont: &[u64; 4], z_dev: u64, errors_dev: u64,
                               stream: *mut std::ffi::c_void) -> Result<(), Error> {
        check(unsafe { h2sha_permutation_product(engine, n as u64, desc, usable_rows, gate as *const _, lookup as *const _, spread as *const _,
                                                 digests_dev as *const u8, beta_mont.as_ptr(), gamma_mont.as_ptr(), z_dev as *mut _, errors_dev as *mut u32, stream) })
    }
    /// Per-instance challenges, for a batch of independent proofs: row i of `thetas_mont` ([n][4] Montgomery limbs) belongs to
    /// instance i; `thetas_mont` may be empty for a range lookup.  errors_dev: device [n] u32 (or 0), entry i counts instance i's failures.
    pub fn permute_lookup_per_instance(engine: *mut h2sha_engine_t, n: usize, lookup_idx: u32, mult_dev: u64, usable_rows: u32, thetas_mont: &[[u64; 4]],
                                       permuted_input_dev: u64, permuted_table_dev: u64, errors_dev: u64, stream: *mut std::ffi::c_void) -> Result<(), Error> {
        if !thetas_mont.is_empty() && thetas_mont.len() != n { return Err(Error::Synthesis); }
        let th = if thetas_mont.is_empty() { std::ptr::null() } else { thetas_mont.as_ptr() as *const u64 };
        check(unsafe { h2sha_permute_lookup_per_instance(engine, n as u64, lookup_idx, mult_dev as *const u32, usable_rows, th, permuted_input_dev as *mut _,
                                                         permuted_table_dev as *mut _, errors_dev as *mut u32, stream) })
    }
    /// `permute_lookup_per_instance` from the raw value lists of the last keep_lookup_raw batch: row i of `thetas_mont` belongs to
    /// instance first_instance + i.
    pub fn permute_lookup_from_raw_per_instance(engine: *mut h2sha_engine_t, first_instance: usize, n: usize, lookup_idx: u32, usable_rows: u32,
                                                thetas_mont: &[[u64; 4]], permuted_input_dev: u64, permuted_table_dev: u64, errors_dev: u64,
                                                stream: *mut std::ffi::c_void) -> Result<(), Error> {
        if !thetas_mont.is_empty() && thetas_mont.len() != n { return Err(Error::Synthesis); }
        let th = if thetas_mont.is_empty() { std::ptr::null() } else { thetas_mont.as_ptr() as *const u64 };
        check(unsafe { h2sha_permute_lookup_from_raw_per_instance(engine, first_instance as u64, n as u64, lookup_idx, usable_rows, th,
                                                                  permuted_input_dev as *mut _, permuted_table_dev as *mut _, errors_dev as *mut u32, stream) })
    }
    /// halo2 `commit_product` of one lookup with per-instance (theta_i, beta_i, gamma_i); `thetas_mont` may be empty for a range lookup.
    pub fn lookup_product_per_instance(engine: *mut h2sha_engine_t, n: usize, lookup_idx: u32, lookup: u64, spread: u64, permuted_input_dev: u64,
                                       permuted_table_dev: u64, usable_rows: u32, thetas_mont: &[[u64; 4]], betas_mont: &[[u64; 4]],
                                       gammas_mont: &[[u64; 4]], z_dev: u64, errors_dev: u64, stream: *mut std::ffi::c_void) -> Result<(), Error> {
        if (!thetas_mont.is_empty() && thetas_mont.len() != n) || betas_mont.len() != n || gammas_mont.len() != n {
            return Err(Error::Synthesis); // one challenge row per instance
        }
        let th = if thetas_mont.is_empty() { std::ptr::null() } else { thetas_mont.as_ptr() as *const u64 };
        check(unsafe { h2sha_lookup_product_per_instance(engine, n as u64, lookup_idx, lookup as *const _, spread as *const _, permuted_input_dev as *const _,
                                                         permuted_table_dev as *const _, usable_rows, th, betas_mont.as_ptr() as *const u64,
                                                         gammas_mont.as_ptr() as *const u64, z_dev as *mut _, errors_dev as *mut u32, stream) })
    }
    /// `permutation_product` with per-instance (beta_i, gamma_i).
    pub fn permutation_product_per_instance(engine: *mut h2sha_engine_t, n: usize, desc: &h2sha_perm_desc_t, usable_rows: u32, gate: u64, lookup: u64,
                                            spread: u64, digests_dev: u64, betas_mont: &[[u64; 4]], gammas_mont: &[[u64; 4]], z_dev: u64, errors_dev: u64,
                                            stream: *mut std::ffi::c_void) -> Result<(), Error> {
        if betas_mont.len() != n || gammas_mont.len() != n {
            return Err(Error::Synthesis); // one challenge row per instance
        }
        check(unsafe { h2sha_permutation_product_per_instance(engine, n as u64, desc, usable_rows, gate as *const _, lookup as *const _, spread as *const _,
                                                              digests_dev as *const u8, betas_mont.as_ptr() as *const u64, gammas_mont.as_ptr() as *const u64,
                                                              z_dev as *mut _, errors_dev as *mut u32, stream) })
    }
    /// `MockProver::run(..).verify()` (lib.rs:525-526) for every instance of a batch, on the device.
    pub fn check_batch(engine: *mut h2sha_engine_t, n: usize, gate: u64, lookup: u64, spread: u64, digests_dev: u64, stream: *mut std::ffi::c_void) -> Result<[u64; 5], Error> {
        let mut v = [0u64; 5];
        check(unsafe { h2sha_check_batch(engine, n as u64, gate as *const _, lookup as *const _, spread as *const _, digests_dev as *const u8, v.as_mut_ptr(), stream) })?;
        Ok(v)
    }
    /// The same check per instance, asynchronous on `stream`: counts / first failing item per instance and class into the device
    /// arrays [n][5] u32 at `counts_dev` / `first_dev` (`first_dev` may be 0).  Item numbering: `h2sha_check_batch_per_instance`.
    pub fn check_batch_per_instance(engine: *mut h2sha_engine_t, n: usize, gate: u64, lookup: u64, spread: u64, digests_dev: u64, counts_dev: u64,
                                    first_dev: u64, stream: *mut std::ffi::c_void) -> Result<(), Error> {
        check(unsafe { h2sha_check_batch_per_instance(engine, n as u64, gate as *const _, lookup as *const _, spread as *const _, digests_dev as *const u8,
                                                      counts_dev as *mut u32, first_dev as *mut u32, stream) })
    }
    /// The cells (`VerifyFailure`'s column and row) check item `item` of class `check_class` reads; host only.
    pub fn check_site(engine: *mut h2sha_engine_t, check_class: u32, item: u32) -> Result<h2sha_check_site_t, Error> {
        let mut s: h2sha_check_site_t = unsafe { std::mem::zeroed() };
        check(unsafe { h2sha_check_site(engine, check_class, item, &mut s) })?;
        Ok(s)
    }
}
