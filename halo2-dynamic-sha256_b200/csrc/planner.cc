// planner.cc -- symbolic walk of the reference program -> static plan.  See planner.h.
//
// Every function below that mirrors a reference function cites it.  The "symbolic value" of a cell
// (struct Sym) says how the kernel derives the cell from the unit's raw u64 slots; the gate/range op
// patterns are those of halo2-base v0.2.x (SURVEY.md 8a Table B).
#include "planner.h"

#include "lookup_geom.h"

#include <algorithm>
#include <array>
#include <map>
#include <set>
#include <stdexcept>
#include <stdio.h>
#include <stdlib.h>

namespace h2sha {
namespace {

enum : uint8_t { T_CONST = 0, T_BYTE = 1, T_SBYTE = 2, T_INV = 3 };

struct Sym {
  uint8_t kind = KIND_GENERIC;
  uint8_t neg = 0;
  uint8_t slot = 0, sh = 0, w = 0, shl = 0;
  uint8_t table = T_CONST;
  uint16_t tbl_off = 0;
  bool operator==(const Sym& o) const {
    return kind == o.kind && neg == o.neg && slot == o.slot && sh == o.sh && w == o.w && shl == o.shl && table == o.table && tbl_off == o.tbl_off;
  }
};

struct AV {  // AssignedValue: global gate-stream index + symbolic value valid inside unit `serial`
  uint32_t idx = 0;
  Sym s;
  uint32_t serial = 0;  // 0: valid everywhere (constants)
};
enum { QC_EXISTING, QC_CONSTANT, QC_WITNESS };
struct QC {
  int kind;
  AV ex;
  U256 cval;  // QC_CONSTANT: canonical value
  Sym s;
  bool has_raw = false;  // QC_CONSTANT: fits a u64 -> usable as VM operand
  uint64_t raw = 0;
  bool dyn = false;      // QC_CONSTANT whose value differs per unit instance (cell comes from a slot)
};

enum : uint8_t { EV_GATE = 0, EV_LK = 1, EV_LIMB = 2 };
struct Event {
  uint8_t kind;
  Sym s;
};
struct UnitRec {
  std::vector<Sym> gate, lk, limb;
  std::vector<Event> ev;  // the same cells in emission order (chunking needs the interleaving)
  std::vector<VmIns> prog;
  std::vector<InputMap> in;
  uint32_t n_slots = 0;
  bool same_as(const UnitRec& o) const {
    if (!(gate == o.gate && lk == o.lk && limb == o.limb) || n_slots != o.n_slots || prog.size() != o.prog.size()) return false;
    for (size_t i = 0; i < prog.size(); i++)
      if (prog[i].op_dst != o.prog[i].op_dst || prog[i].a != o.prog[i].a || prog[i].b != o.prog[i].b || prog[i].c != o.prog[i].c) return false;
    return true;
  }
};

struct GroupRec {
  std::string type;
  uint32_t count = 0, seen = 0;
  uint32_t gate_base = 0, gate_stride = 0, lk_base = 0, lk_stride = 0, limb_base = 0, limb_stride = 0;
  uint32_t dict_base = 0;   // set in finalize: dictionary index of instance 0 relative to the job's dictionary base
  std::vector<InputMap> in;
  bool same_as(const GroupRec& o) const {
    if (type != o.type || count != o.count || gate_base != o.gate_base || gate_stride != o.gate_stride || lk_base != o.lk_base ||
        lk_stride != o.lk_stride || limb_base != o.limb_base || limb_stride != o.limb_stride || in.size() != o.in.size())
      return false;
    for (size_t i = 0; i < in.size(); i++)
      if (in[i].base != o.in[i].base || in[i].stride != o.in[i].stride) return false;
    return true;
  }
};
struct ClassRec {
  uint32_t gate_origin = 0, lk_origin = 0, limb_origin = 0;
  std::vector<GroupRec> groups;
};

[[noreturn]] void fail(const std::string& m) { throw std::runtime_error(m); }

U256 pow2(uint32_t n) {
  if (n >= 254) fail("pow2 too large");
  U256 r = {{0, 0, 0, 0}};
  r.l[n / 64] = 1ULL << (n % 64);
  return r;
}

class Builder {
 public:
  Builder(const Config& cfg, Plan* plan) : cfg_(cfg), P_(plan) {}

  void run() {
    if (cfg_.max_variable_byte_sizes.empty()) fail("max_variable_byte_sizes is empty");
    if (cfg_.limb_bits == 0 || 16 % cfg_.limb_bits != 0) fail("num_bits_lookup must divide 16 (spread.rs:37)");
    if (cfg_.spread_cols == 0) fail("num_advice_columns must be >= 1");
    if (cfg_.lookup_bits < 8 || cfg_.lookup_bits > 32) fail("lookup_bits must be in [8, 32]");
    if (cfg_.max_rows < 64) fail("max_rows too small");
    if (cfg_.max_fill < 64 || cfg_.max_fill > H2SHA_MAX_FILL_LIMIT || cfg_.max_fill % 8) fail("max_fill must be a multiple of 8 in [64, 256]");
    uint32_t max_r = 0;
    for (uint32_t m : cfg_.max_variable_byte_sizes) {
      if (m == 0 || m % 64 != 0) fail("max_variable_byte_size must be a positive multiple of 64 (lib.rs:57-59)");
      max_r = std::max(max_r, m / 64);
    }
    inv_bias_ = max_r + 2;
    if (2 * inv_bias_ + 1 > 250) fail("max_variable_byte_size too large for the inverse table");
    const_id(U256{{0, 0, 0, 0}});  // table entry 0 is the zero constant
    for (uint32_t d = 0; d < cfg_.max_variable_byte_sizes.size(); d++) digest(d);
    finalize();
  }

 private:
  const Config& cfg_;
  Plan* P_;
  // ---- global stream state (Context) ----
  uint32_t n_gate_ = 0, col_ = 0, row_ = 0;
  uint32_t n_lk_ = 0, n_limb_ = 0;
  bool has_zero_ = false;
  AV zero_;
  std::vector<U256> consts_;  // Montgomery table consts (superset of fixed cells; same order for fixed ones)
  std::map<std::pair<std::pair<uint64_t, uint64_t>, std::pair<uint64_t, uint64_t>>, uint32_t> const_map_;
  std::map<uint64_t, uint32_t> raw_map_;
  uint32_t inv_bias_ = 0;
  // ---- unit / group / class recording ----
  std::map<std::string, uint32_t> type_idx_;
  std::vector<UnitRec> type_recs_;
  UnitRec cur_;
  bool in_unit_ = false;
  uint32_t serial_ = 0;
  uint32_t unit_gate0_ = 0, unit_lk0_ = 0, unit_limb0_ = 0;
  ClassRec* cls_ = nullptr;
  GroupRec* grp_ = nullptr;
  std::vector<ClassRec> class_recs_;  // index = class id
  std::vector<bool> class_set_;

  // ======================================================================================
  // symbolic values
  // ======================================================================================
  static Sym ext(uint32_t slot, uint32_t sh, uint32_t w) {
    Sym s;
    s.kind = KIND_GENERIC;
    s.slot = (uint8_t)slot; s.sh = (uint8_t)sh; s.w = (uint8_t)w;
    if (slot > 255 || sh > 63 || w > 64 || sh + w > 64) fail("bad extract");
    return s;
  }
  static bool plain(const Sym& s) { return s.kind == KIND_GENERIC && !s.neg && s.shl == 0; }
  // bits [sh2, sh2+w2) of an extract
  static Sym sub(const Sym& s, uint32_t sh2, uint32_t w2) {
    if (!plain(s)) fail("sub-extract of a non-plain value");
    uint32_t w = sh2 >= s.w ? 0 : std::min<uint32_t>(w2, s.w - sh2);
    return ext(s.slot, w ? s.sh + sh2 : 0, w);
  }
  static Sym shl(const Sym& s, uint32_t n) {
    if (!plain(s) || n > 31) fail("bad shl");
    Sym r = s; r.shl = (uint8_t)n; return r;
  }
  static Sym negated(const Sym& s) {
    if (!plain(s)) fail("bad neg");
    Sym r = s; r.neg = 1; return r;
  }
  static Sym table(uint8_t t, const Sym& idx, uint32_t off = 0) {
    if (!plain(idx)) fail("table index must be a plain extract");
    Sym r = idx; r.kind = KIND_TABLE; r.table = t; r.tbl_off = (uint16_t)off; return r;
  }
  static Sym signed_slot(uint32_t slot) {
    Sym r; r.kind = KIND_SIGNED; r.slot = (uint8_t)slot; r.w = 64; return r;
  }

  // index of a constant in the Montgomery table
  uint32_t const_id(const U256& v) {
    auto key = std::make_pair(std::make_pair(v.l[0], v.l[1]), std::make_pair(v.l[2], v.l[3]));
    auto it = const_map_.find(key);
    if (it != const_map_.end()) return it->second;
    uint32_t id = (uint32_t)consts_.size();
    consts_.push_back(v);
    fixed_of_const_.push_back(~0u);
    const_map_[key] = id;
    return id;
  }
  // Context::assign_fixed: the fixed-column cell of a constant, de-duplicated, in first-use order
  uint32_t fixed_id(uint32_t cid) {
    if (fixed_of_const_[cid] == ~0u) {
      fixed_of_const_[cid] = n_fixed_++;
      if (cfg_.record_shape) P_->fixed_consts.push_back(consts_[cid]);
    }
    return fixed_of_const_[cid];
  }
  std::vector<uint32_t> fixed_of_const_;
  uint32_t n_fixed_ = 0;

  uint32_t raw_const(uint64_t v) {
    auto it = raw_map_.find(v);
    if (it != raw_map_.end()) return it->second;
    uint32_t id = (uint32_t)P_->raw_consts.size();
    P_->raw_consts.push_back(v);
    raw_map_[v] = id;
    return id;
  }

  // ---- QuantumCell constructors ----
  QC EX(const AV& a) { QC q; q.kind = QC_EXISTING; q.ex = a; q.s = a.s; return q; }
  QC CU(const U256& v) {  // Constant(F)
    QC q; q.kind = QC_CONSTANT; q.cval = v;
    uint32_t id = const_id(v);
    q.s = Sym(); q.s.kind = KIND_TABLE; q.s.table = T_CONST; q.s.tbl_off = (uint16_t)id; q.s.w = 0;
    q.has_raw = (v.l[1] | v.l[2] | v.l[3]) == 0; q.raw = v.l[0];
    return q;
  }
  QC C(uint64_t v) { return CU(fr::from_u64(v)); }
  // Constant whose value differs per unit instance (round constant K[t], loop counter n): the cell is
  // produced from an input slot; the fixed-column bookkeeping uses this instance's concrete value.
  QC Cdyn(const Sym& s, const U256& this_instance_value) {
    QC q; q.kind = QC_CONSTANT; q.s = s; q.has_raw = false; q.dyn = true; q.cval = this_instance_value; return q;
  }
  QC W(const Sym& s) { QC q; q.kind = QC_WITNESS; q.s = s; return q; }

  uint32_t operand(const QC& q) {
    if (q.kind == QC_CONSTANT && !q.dyn) {
      if (!q.has_raw) fail("constant does not fit a VM operand");
      return vm_operand_const(raw_const(q.raw));
    }
    return operand(q.s);
  }
  uint32_t operand(const Sym& s) {
    if (!plain(s)) fail("VM operand must be a plain extract");
    return vm_operand_slot(s.slot, s.sh, s.w);
  }

  // ======================================================================================
  // unit / group / class bookkeeping
  // ======================================================================================
  void use_class(ClassRec* c) { cls_ = c; }
  void begin_group(const std::string& type, uint32_t count) {
    if (grp_) fail("nested group");
    cls_->groups.emplace_back();
    grp_ = &cls_->groups.back();
    grp_->type = type; grp_->count = count;
  }
  void end_group() {
    if (!grp_ || grp_->seen != grp_->count) fail("group instance count mismatch: " + (grp_ ? grp_->type : std::string("?")));
    grp_ = nullptr;
  }
  void begin_unit() {
    if (in_unit_ || !grp_) fail("begin_unit outside group");
    in_unit_ = true; serial_++;
    cur_ = UnitRec();
    unit_gate0_ = n_gate_; unit_lk0_ = n_lk_; unit_limb0_ = n_limb_;
  }
  // declares input slot k = trace[base + stride * u]  (base < 0: the instance index u)
  Sym input(uint32_t k, int32_t base, int32_t stride, uint32_t w = 32) {
    if (k != cur_.in.size() || k >= MAX_UNIT_INPUTS) fail("inputs must be declared in order");
    cur_.in.push_back(InputMap{base, stride});
    cur_.n_slots = k + 1;
    return ext(k, 0, w);
  }
  uint32_t new_slot() {
    if (cur_.n_slots >= 255) fail("too many slots in unit " + grp_->type);
    return cur_.n_slots++;
  }
  Sym emit(uint32_t op, uint32_t a, uint32_t b, uint32_t c, uint32_t width) {
    uint32_t dst = new_slot();
    cur_.prog.push_back(VmIns{op | (dst << 8), a, b, c});
    return ext(dst, 0, width);
  }
  void end_unit() {
    if (!in_unit_) fail("end_unit");
    in_unit_ = false;
    uint32_t u = grp_->seen++;
    // per-instance input base: the declared base is that of instance u -> normalise to instance 0
    std::vector<InputMap> in0 = cur_.in;
    for (auto& m : in0)
      if (m.base >= 0) m.base -= m.stride * (int32_t)u;
    cur_.in = in0;
    auto it = type_idx_.find(grp_->type);
    if (it == type_idx_.end()) {
      type_idx_[grp_->type] = (uint32_t)type_recs_.size();
      type_recs_.push_back(cur_);
    } else if (!type_recs_[it->second].same_as(cur_)) {
      fail("unit instances of type " + grp_->type + " differ");
    }
    uint32_t g = unit_gate0_ - cls_->gate_origin, l = unit_lk0_ - cls_->lk_origin, m = unit_limb0_ - cls_->limb_origin;
    if (u == 0) {
      grp_->gate_base = g; grp_->lk_base = l; grp_->limb_base = m; grp_->in = in0;
    } else {
      if (u == 1) { grp_->gate_stride = g - grp_->gate_base; grp_->lk_stride = l - grp_->lk_base; grp_->limb_stride = m - grp_->limb_base; }
      if (g != grp_->gate_base + u * grp_->gate_stride || l != grp_->lk_base + u * grp_->lk_stride || m != grp_->limb_base + u * grp_->limb_stride)
        fail("non-uniform unit stride in " + grp_->type);
      for (size_t i = 0; i < in0.size(); i++)
        if (in0[i].base != grp_->in[i].base || in0[i].stride != grp_->in[i].stride) fail("non-affine input map in " + grp_->type);
    }
  }
  AV rebind(const AV& a, const Sym& s) { AV r = a; r.s = s; r.serial = serial_; return r; }

  // ======================================================================================
  // halo2-base Context / FlexGate / Range (symbolic)
  // ======================================================================================
  void add_copy(uint32_t ak, uint32_t ai, uint32_t bk, uint32_t bi) {
    if (cfg_.record_shape) P_->copies.push_back(CopyPair{ak, ai, bk, bi});
  }
  // FlexGateConfig::assign_region_in: break to the next column when `row + len >= max_rows`
  void assign_region(const std::vector<QC>& cells, std::initializer_list<int> gate_offs, std::vector<AV>* out) {
    if (!in_unit_) fail("assign_region outside a unit");
    uint32_t n = (uint32_t)cells.size();
    if (P_->breaks.empty()) P_->breaks.push_back(0);
    if (row_ + n >= cfg_.max_rows) {
      if (row_ == 0) fail("max_rows too small for one op");
      row_ = 0; col_++;
      P_->breaks.push_back(n_gate_);
    }
    uint32_t base = n_gate_;
    if (out) out->resize(n);
    for (uint32_t i = 0; i < n; i++) {
      const QC& q = cells[i];
      if (q.kind == QC_EXISTING && q.ex.serial != 0 && q.ex.serial != serial_) fail("cell from another unit used without rebind in " + grp_->type);
      cur_.gate.push_back(q.s);
      cur_.ev.push_back(Event{EV_GATE, q.s});
      if (cfg_.record_shape) {
        P_->selectors.push_back(0);
        if (q.kind == QC_EXISTING) add_copy(CP_GATE, base + i, CP_GATE, q.ex.idx);
      }
      if (q.kind == QC_CONSTANT) {
        uint32_t fid = fixed_id(q.dyn ? const_id(q.cval) : q.s.tbl_off);
        add_copy(CP_GATE, base + i, CP_FIXED, fid);
      }
      if (out) { (*out)[i].idx = base + i; (*out)[i].s = q.s; (*out)[i].serial = (q.s.kind == KIND_TABLE && q.s.w == 0) ? 0 : serial_; }
    }
    if (cfg_.record_shape)
      for (int o : gate_offs) P_->selectors[base + o] = 1;
    n_gate_ += n; row_ += n;
  }

  AV load_witness(const Sym& s) { std::vector<AV> o; assign_region({W(s)}, {}, &o); return o[0]; }
  AV load_zero() {
    if (has_zero_) return zero_;
    std::vector<AV> o; assign_region({C(0)}, {}, &o);
    has_zero_ = true; zero_ = o[0]; zero_.serial = 0;
    return zero_;
  }
  AV add(const QC& a, const QC& b, const Sym& out) { std::vector<AV> o; assign_region({a, b, C(1), W(out)}, {0}, &o); return o[3]; }
  AV sub(const QC& a, const QC& b, const Sym& out) { std::vector<AV> o; assign_region({W(out), b, C(1), a}, {0}, &o); return o[0]; }
  AV neg(const QC& a, const Sym& out) { std::vector<AV> o; assign_region({a, W(out), C(1), C(0)}, {0}, &o); return o[1]; }
  AV mul(const QC& a, const QC& b, const Sym& out) { std::vector<AV> o; assign_region({C(0), a, b, W(out)}, {0}, &o); return o[3]; }
  AV mul_add(const QC& a, const QC& b, const QC& c, const Sym& out) { std::vector<AV> o; assign_region({c, a, b, W(out)}, {0}, &o); return o[3]; }
  AV select(const QC& a, const QC& b, const QC& sel, const Sym& diff, const Sym& out) {
    std::vector<AV> o;
    assign_region({W(diff), C(1), b, a, b, sel, W(diff), W(out)}, {0, 4}, &o);
    add_copy(CP_GATE, o[0].idx, CP_GATE, o[6].idx);
    return o[7];
  }
  AV is_zero(const AV& a, const Sym& z, const Sym& inv) {
    std::vector<AV> o;
    assign_region({W(z), EX(a), W(inv), C(1), C(0), EX(a), W(z), C(0)}, {0, 4}, &o);
    add_copy(CP_GATE, o[0].idx, CP_GATE, o[6].idx);
    return o[0];
  }
  void assert_equal(const AV& a, const AV& b) { add_copy(CP_GATE, a.idx, CP_GATE, b.idx); }
  void assert_is_const(const AV& a, const U256& v) {
    add_copy(CP_GATE, a.idx, CP_FIXED, fixed_id(const_id(v)));
  }
  // new-slot flavours
  AV add_new(const QC& a, const QC& b, uint32_t width) { return add(a, b, emit(OP_ADD, operand(a), operand(b), 0, width)); }

  void lk_push(const AV& a) {
    cur_.lk.push_back(a.s);
    cur_.ev.push_back(Event{EV_LK, a.s});
    if (a.serial != 0 && a.serial != serial_) fail("lookup of a cell from another unit");
    if (cfg_.record_shape) P_->lookup_cells.push_back(a.idx);
    n_lk_++;
  }
  // RangeConfig::range_check (Vertical)
  AV range_check(const AV& a, uint32_t range_bits) {
    uint32_t lb = cfg_.lookup_bits;
    uint32_t k = (range_bits + lb - 1) / lb, rem = range_bits % lb;
    AV last = a;
    if (k == 1) {
      lk_push(a);
    } else {
      std::vector<QC> cells;
      std::vector<int> limb_pos;
      std::vector<int> offs;
      for (uint32_t i = 0; i < k; i++) {
        Sym limb = sub(a.s, lb * i, lb);
        if (i == 0) { limb_pos.push_back(0); cells.push_back(W(limb)); }
        else {
          offs.push_back((int)cells.size() - 1);
          limb_pos.push_back((int)cells.size());
          cells.push_back(W(limb));
          cells.push_back(CU(pow2(lb * i)));
          cells.push_back(W(sub(a.s, 0, lb * (i + 1))));
        }
      }
      std::vector<AV> o;
      assign_region_offs(cells, offs, &o);
      for (uint32_t i = 0; i < k; i++) lk_push(o[limb_pos[i]]);
      last = o[limb_pos[k - 1]];
      add_copy(CP_GATE, a.idx, CP_GATE, o.back().idx);
    }
    if (rem == 1) fail("range_check with rem_bits == 1 (assert_bit) is not used by the reference");
    if (rem > 1) {
      std::vector<AV> o;
      assign_region({C(0), EX(last), CU(pow2(lb - rem)), W(shl(last.s, lb - rem))}, {0}, &o);
      lk_push(o[3]);
      last = o[3];
    }
    return last;  // the most recently looked-up cell (ctx.cells_to_lookup.last())
  }
  void assign_region_offs(const std::vector<QC>& cells, const std::vector<int>& offs, std::vector<AV>* out) {
    assign_region(cells, {}, out);
    if (cfg_.record_shape)
      for (int o : offs) P_->selectors[(*out)[0].idx + o] = 1;
  }

  // ======================================================================================
  // src/spread.rs
  // ======================================================================================
  // spread.rs:196-233
  // `whole_spread`: with 16-bit limbs (num_bits_lookup = 16: one limb per `spread`, no 2^16-entry table in shared memory) the limb's
  // spread is the caller's 32-bit spread slot itself, a plain extract the Barrett path converts
  AV spread_limb(const AV& limb, const Sym* whole_spread = nullptr) {
    Sym sp = whole_spread ? *whole_spread : table(T_SBYTE, limb.s);
    cur_.limb.push_back(limb.s);  // dense column cell (:203-208)
    cur_.limb.push_back(sp);      // spread column cell (:219-224)
    cur_.ev.push_back(Event{EV_LIMB, limb.s});
    cur_.ev.push_back(Event{EV_LIMB, sp});
    AV as = load_witness(sp);     // :225
    if (cfg_.record_shape) { P_->limb_gate_dense.push_back(limb.idx); P_->limb_gate_spread.push_back(as.idx); }
    n_limb_++;
    return as;
  }
  // spread.rs:76-123; `out` = symbolic 32-bit spread of `dense` (the caller owns the slot)
  AV spread(const AV& dense, const Sym& out) {
    uint32_t lb = cfg_.limb_bits, nl = 16 / lb;
    if (!plain(dense.s) || dense.s.w != 16) fail("spread() of a value that is not a 16-bit extract");
    std::vector<AV> limbs;
    for (uint32_t i = 0; i < nl; i++) limbs.push_back(load_witness(sub(dense.s, lb * i, lb)));           // :85-88
    AV sum = load_zero();                                                                                 // :90
    for (uint32_t i = 0; i < nl; i++) sum = mul_add(EX(limbs[i]), C(1ULL << (lb * i)), EX(sum), sub(dense.s, 0, lb * (i + 1)));  // :91-98
    assert_equal(sum, dense);                                                                             // :104-108
    AV acc = load_zero();                                                                                 // :110
    for (uint32_t i = 0; i < nl; i++) {                                                                   // :112-121
      const Sym whole = sub(out, 0, 32);
      AV sl = spread_limb(limbs[i], lb == 16 ? &whole : nullptr);
      Sym partial = (i == 0) ? (lb == 16 ? whole : table(T_SBYTE, limbs[0].s)) : sub(out, 0, 2 * lb * (i + 1));
      acc = mul_add(EX(sl), C(1ULL << (2 * lb * i)), EX(acc), partial);
    }
    return acc;
  }
  // spread.rs:139-163
  void decompose_even_and_odd_unchecked(const Sym& even, const Sym& odd, AV* e, AV* o) {
    *e = load_witness(even);   // :158
    *o = load_witness(odd);    // :159
    range_check(*e, 16);       // :160
    range_check(*o, 16);       // :161
  }

  // ======================================================================================
  // src/compression.rs
  // ======================================================================================
  struct SpreadU32 { AV lo, hi; };  // compression.rs:17

  // compression.rs:215-246; x must be a 32-bit plain extract.  Allocates the slot S = spread32(x).
  SpreadU32 state_to_spread_u32(const AV& x) {
    Sym S = emit(OP_SPREAD, operand(sub(x.s, 0, 32)), 0, 0, 64);
    AV lo = load_witness(sub(x.s, 0, 16));                                   // :222-230
    AV hi = load_witness(sub(x.s, 16, 16));                                  // :226-231
    AV composed = mul_add(EX(hi), C(1ULL << 16), EX(lo), sub(x.s, 0, 32));   // :232-237
    assert_equal(x, composed);                                               // :238-242
    SpreadU32 r;
    r.lo = spread(lo, sub(S, 0, 32));                                        // :243
    r.hi = spread(hi, sub(S, 32, 32));                                       // :244
    return r;
  }
  // compression.rs:266-295; x is a plain extract of a slot holding the (< 2^64) sum
  AV mod_u32(const AV& x) {
    AV lo = load_witness(sub(x.s, 0, 32));                                   // :272-280
    AV hi = load_witness(sub(x.s, 32, 32));                                  // :276-281
    range_check(lo, 32);                                                     // :282
    AV composed = mul_add(EX(hi), C(1ULL << 32), EX(lo), x.s);               // :283-288
    assert_equal(x, composed);                                               // :289-293
    return lo;
  }
  // shared tail of ch / maj / sigma_generic (compression.rs:344-354 etc.)
  void check_even_odd(const AV& even, const AV& odd, const AV& v, const Sym& even_spread, const Sym& odd_spread) {
    AV es = spread(even, even_spread);
    AV os = spread(odd, odd_spread);
    AV sum = mul_add(C(2), EX(os), EX(es), v.s);
    assert_equal(sum, v);
  }
  // even/odd decomposition of two 32-bit values packed by OP_COMPRESS2, plus their re-spreads
  struct EvenOdd { Sym lo_e, lo_o, hi_e, hi_o, se_lo, so_lo, se_hi, so_hi, evens32, odds32; };
  EvenOdd compress_pair(const Sym& lo32, const Sym& hi32) {
    Sym Cx = emit(OP_COMPRESS2, operand(lo32), operand(hi32), 0, 64);
    Sym SE = emit(OP_SPREAD, operand(sub(Cx, 0, 32)), 0, 0, 64);
    Sym SO = emit(OP_SPREAD, operand(sub(Cx, 32, 32)), 0, 0, 64);
    EvenOdd r;
    r.lo_e = sub(Cx, 0, 16); r.hi_e = sub(Cx, 16, 16); r.lo_o = sub(Cx, 32, 16); r.hi_o = sub(Cx, 48, 16);
    r.se_lo = sub(SE, 0, 32); r.se_hi = sub(SE, 32, 32); r.so_lo = sub(SO, 0, 32); r.so_hi = sub(SO, 32, 32);
    r.evens32 = sub(Cx, 0, 32); r.odds32 = sub(Cx, 32, 32);
    return r;
  }
  // compression.rs:297-405
  AV ch(const SpreadU32& x, const SpreadU32& y, const SpreadU32& z) {
    AV p_lo = add_new(EX(x.lo), EX(y.lo), 32);                               // :309-313
    AV p_hi = add_new(EX(x.hi), EX(y.hi), 32);                               // :314-318
    const uint64_t MASK_EVEN_32 = 0x55555555ULL;                             // :319
    AV x_neg_lo = neg(EX(x.lo), negated(x.lo.s));                            // :320
    AV x_neg_hi = neg(EX(x.hi), negated(x.hi.s));                            // :321
    // three_add(mask, -x, z) (:322-335, :521-530): add1 = mask - x, add2 = add1 + z
    QC mask = C(MASK_EVEN_32);
    AV q1_lo = add(mask, EX(x_neg_lo), emit(OP_SUB, operand(mask), operand(x.lo.s), 0, 32));
    AV q_lo = add_new(EX(q1_lo), EX(z.lo), 32);
    AV q1_hi = add(mask, EX(x_neg_hi), emit(OP_SUB, operand(mask), operand(x.hi.s), 0, 32));
    AV q_hi = add_new(EX(q1_hi), EX(z.hi), 32);
    EvenOdd p = compress_pair(p_lo.s, p_hi.s), q = compress_pair(q_lo.s, q_hi.s);
    AV p_lo_e, p_lo_o, p_hi_e, p_hi_o, q_lo_e, q_lo_o, q_hi_e, q_hi_o;
    decompose_even_and_odd_unchecked(p.lo_e, p.lo_o, &p_lo_e, &p_lo_o);      // :336-343
    decompose_even_and_odd_unchecked(p.hi_e, p.hi_o, &p_hi_e, &p_hi_o);
    decompose_even_and_odd_unchecked(q.lo_e, q.lo_o, &q_lo_e, &q_lo_o);
    decompose_even_and_odd_unchecked(q.hi_e, q.hi_o, &q_hi_e, &q_hi_o);
    check_even_odd(p_lo_e, p_lo_o, p_lo, p.se_lo, p.so_lo);                  // :344-354
    check_even_odd(p_hi_e, p_hi_o, p_hi, p.se_hi, p.so_hi);                  // :355-365
    check_even_odd(q_lo_e, q_lo_o, q_lo, q.se_lo, q.so_lo);                  // :366-376
    check_even_odd(q_hi_e, q_hi_o, q_hi, q.se_hi, q.so_hi);                  // :377-387
    // odd(P) and odd(Q) have disjoint bits, so both 16-bit halves add without carry: one packed slot
    Sym OUT = emit(OP_ADD, operand(p.odds32), operand(q.odds32), 0, 32);
    AV out_lo = add(EX(p_lo_o), EX(q_lo_o), sub(OUT, 0, 16));                // :388-392
    AV out_hi = add(EX(p_hi_o), EX(q_hi_o), sub(OUT, 16, 16));               // :393-397
    return mul_add(EX(out_hi), C(1ULL << 16), EX(out_lo), OUT);              // :398-403
  }
  // compression.rs:460-519
  AV maj(const SpreadU32& x, const SpreadU32& y, const SpreadU32& z) {
    AV m1_lo = add_new(EX(x.lo), EX(y.lo), 32);                              // :472-478 (three_add)
    AV m_lo = add_new(EX(m1_lo), EX(z.lo), 32);
    AV m1_hi = add_new(EX(x.hi), EX(y.hi), 32);                              // :479-485
    AV m_hi = add_new(EX(m1_hi), EX(z.hi), 32);
    EvenOdd m = compress_pair(m_lo.s, m_hi.s);
    AV lo_e, lo_o, hi_e, hi_o;
    decompose_even_and_odd_unchecked(m.lo_e, m.lo_o, &lo_e, &lo_o);          // :486-489
    decompose_even_and_odd_unchecked(m.hi_e, m.hi_o, &hi_e, &hi_o);
    check_even_odd(lo_e, lo_o, m_lo, m.se_lo, m.so_lo);                      // :490-500
    check_even_odd(hi_e, hi_o, m_hi, m.se_hi, m.so_hi);                      // :501-511
    return mul_add(EX(hi_o), C(1ULL << 16), EX(lo_o), m.odds32);             // :512-517
  }
  // compression.rs:702-882.  xs.lo / xs.hi must be extracts [0,32) / [32,64) of one slot S = spread32(x).
  AV sigma_generic(const SpreadU32& xs, const int starts[4], const int ends[4], const uint64_t coeffs[4]) {
    const Sym& lo = xs.lo.s;
    if (!plain(lo) || !plain(xs.hi.s) || lo.slot != xs.hi.s.slot || lo.sh != 0 || lo.w != 32 || xs.hi.s.sh != 32 || xs.hi.s.w != 32)
      fail("sigma_generic: x_spread must be the two halves of one spread slot");
    Sym S = ext(lo.slot, 0, 64);
    AV piece[4];
    for (int k = 0; k < 4; k++) piece[k] = load_witness(sub(S, 2 * starts[k], 2 * (ends[k] - starts[k])));   // :719-734
    {                                                                        // :735-766
      AV sum = piece[0];
      for (int k = 1; k < 4; k++) sum = mul_add(EX(piece[k]), C(1ULL << (2 * starts[k])), EX(sum), sub(S, 0, 2 * ends[k]));
      AV x_composed = mul_add(EX(xs.hi), C(1ULL << 32), EX(xs.lo), S);
      assert_equal(x_composed, sum);
    }
    AV r_spread = load_zero();                                               // :775-810
    for (int k = 0; k < 4; k++) {
      QC coeff = C(coeffs[k]);
      uint32_t prev = (k == 0) ? vm_operand_const(raw_const(0)) : operand(r_spread.s);
      Sym acc = emit(OP_MULADD, operand(coeff), operand(piece[k].s), prev, 64);
      r_spread = mul_add(coeff, EX(piece[k]), EX(r_spread), acc);
    }
    Sym Rr = r_spread.s;
    AV r_lo = load_witness(sub(Rr, 0, 32));                                  // :811-821
    AV r_hi = load_witness(sub(Rr, 32, 32));
    range_check(r_lo, 32);                                                   // :822
    range_check(r_hi, 32);                                                   // :823
    AV composed = mul_add(EX(r_hi), C(1ULL << 32), EX(r_lo), Rr);            // :824-829
    assert_equal(r_spread, composed);                                        // :830-834
    EvenOdd eo = compress_pair(r_lo.s, r_hi.s);
    AV lo_e, lo_o, hi_e, hi_o;
    decompose_even_and_odd_unchecked(eo.lo_e, eo.lo_o, &lo_e, &lo_o);        // :843-846
    decompose_even_and_odd_unchecked(eo.hi_e, eo.hi_o, &hi_e, &hi_o);
    check_even_odd(lo_e, lo_o, r_lo, eo.se_lo, eo.so_lo);                    // :852-862
    check_even_odd(hi_e, hi_o, r_hi, eo.se_hi, eo.so_hi);                    // :863-873
    return mul_add(EX(hi_e), C(1ULL << 16), EX(lo_e), eo.evens32);           // :874-879
  }
#define B_(n) (1ULL << (n))
  AV sigma_upper0(const SpreadU32& x) {  // compression.rs:594-619
    static const int S[4] = {0, 2, 13, 22}, E[4] = {2, 13, 22, 32};
    static const uint64_t K[4] = {B_(60) + B_(38) + B_(20), B_(0) + B_(42) + B_(24), B_(22) + B_(0) + B_(46), B_(40) + B_(18) + B_(0)};
    return sigma_generic(x, S, E, K);
  }
  AV sigma_upper1(const SpreadU32& x) {  // compression.rs:621-646
    static const int S[4] = {0, 6, 11, 25}, E[4] = {6, 11, 25, 32};
    static const uint64_t K[4] = {B_(52) + B_(42) + B_(14), B_(0) + B_(54) + B_(26), B_(10) + B_(0) + B_(36), B_(38) + B_(28) + B_(0)};
    return sigma_generic(x, S, E, K);
  }
  AV sigma_lower0(const SpreadU32& x) {  // compression.rs:648-673
    static const int S[4] = {0, 3, 7, 18}, E[4] = {3, 7, 18, 32};
    static const uint64_t K[4] = {B_(50) + B_(28), B_(0) + B_(56) + B_(34), B_(8) + B_(0) + B_(42), B_(30) + B_(22) + B_(0)};
    return sigma_generic(x, S, E, K);
  }
  AV sigma_lower1(const SpreadU32& x) {  // compression.rs:675-700
    static const int S[4] = {0, 10, 17, 19}, E[4] = {10, 17, 19, 32};
    static const uint64_t K[4] = {B_(30) + B_(26), B_(0) + B_(50) + B_(46), B_(14) + B_(0) + B_(60), B_(18) + B_(4) + B_(0)};
    return sigma_generic(x, S, E, K);
  }
#undef B_
  // a SpreadU32 living in another unit, re-derived in this unit from the u32 input `x`
  SpreadU32 rebind_spread(const SpreadU32& src, const Sym& x) {
    Sym S = emit(OP_SPREAD, operand(sub(x, 0, 32)), 0, 0, 64);
    SpreadU32 r;
    r.lo = rebind(src.lo, sub(S, 0, 32));
    r.hi = rebind(src.hi, sub(S, 32, 32));
    return r;
  }

  static const uint32_t* round_constants() {
    static const uint32_t K[64] = {
        0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
        0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
        0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
        0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
        0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
        0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
    return K;
  }

  // compression.rs:19-213, split into units.  `blk` is the block-class recorder, `dig` the enclosing digest's.
  void sha256_compression(ClassRec* blk, ClassRec* dig, const std::vector<AV>& in_bytes /*64*/, const AV pre[8], AV next[8]) {
    if (!has_zero_) {  // the one-time `C 0` cell of the first load_zero in the Context (:34) belongs to the digest job
      use_class(dig);
      begin_group("ZERO", 1); begin_unit(); load_zero(); end_unit(); end_group();
    }
    use_class(blk);
    blk->gate_origin = n_gate_; blk->lk_origin = n_lk_; blk->limb_origin = n_limb_;
    blk->groups.clear();
    AV w[64]; SpreadU32 ws[64];
    begin_group("WORD", 16);                                                 // :31-47
    for (int i = 0; i < 16; i++) {
      begin_unit();
      Sym Wi = input(0, TR_W + i, 1);
      AV sum = load_zero();
      for (int idx = 0; idx < 4; idx++) {
        AV byte = rebind(in_bytes[4 * i + 3 - idx], sub(Wi, 8 * idx, 8));
        sum = mul_add(EX(byte), C(1ULL << (8 * idx)), EX(sum), sub(Wi, 0, 8 * (idx + 1)));
      }
      w[i] = sum;
      end_unit();
    }
    end_group();
    begin_group("STSW", 16);                                                 // :53-56
    for (int i = 0; i < 16; i++) {
      begin_unit();
      Sym Wi = input(0, TR_W + i, 1);
      ws[i] = state_to_spread_u32(rebind(w[i], Wi));
      end_unit();
    }
    end_group();
    begin_group("SCHED", 48);                                                // :57-96
    for (int idx = 16; idx < 64; idx++) {
      begin_unit();
      Sym w2 = input(0, TR_W + idx - 2, 1), w15 = input(1, TR_W + idx - 15, 1), w7 = input(2, TR_W + idx - 7, 1), w16 = input(3, TR_W + idx - 16, 1);
      AV term1 = sigma_lower1(rebind_spread(ws[idx - 2], w2));
      AV term3 = sigma_lower0(rebind_spread(ws[idx - 15], w15));
      AV sum = add_new(EX(term1), EX(rebind(w[idx - 7], w7)), 33);
      sum = add_new(EX(sum), EX(term3), 34);
      sum = add_new(EX(sum), EX(rebind(w[idx - 16], w16)), 35);
      w[idx] = mod_u32(sum);
      ws[idx] = state_to_spread_u32(w[idx]);
      end_unit();
    }
    end_group();
    AV a = pre[0], b = pre[1], c = pre[2], d = pre[3], e = pre[4], f = pre[5], g = pre[6], h = pre[7];   // :99-108
    SpreadU32 a_s, b_s, c_s, e_s, f_s, g_s;
    begin_group("STSA", 3);                                                  // :109-111
    { AV* src[3] = {&a, &b, &c}; SpreadU32* dst[3] = {&a_s, &b_s, &c_s};
      for (int i = 0; i < 3; i++) { begin_unit(); Sym x = input(0, TR_A + 3 - i, -1); *dst[i] = state_to_spread_u32(rebind(*src[i], x)); end_unit(); } }
    end_group();
    begin_group("STSE", 3);                                                  // :113-115
    { AV* src[3] = {&e, &f, &g}; SpreadU32* dst[3] = {&e_s, &f_s, &g_s};
      for (int i = 0; i < 3; i++) { begin_unit(); Sym x = input(0, TR_E + 3 - i, -1); *dst[i] = state_to_spread_u32(rebind(*src[i], x)); end_unit(); } }
    end_group();
    // :123-124 two load_zero calls: cached, no cells
    begin_group("ROUND", 64);                                                // :125-196
    for (int idx = 0; idx < 64; idx++) {
      begin_unit();
      Sym ia = input(0, TR_A + idx + 3, 1), ib = input(1, TR_A + idx + 2, 1), ic = input(2, TR_A + idx + 1, 1), id = input(3, TR_A + idx, 1);
      Sym ie = input(4, TR_E + idx + 3, 1), if_ = input(5, TR_E + idx + 2, 1), ig = input(6, TR_E + idx + 1, 1), ih = input(7, TR_E + idx, 1);
      Sym iw = input(8, TR_W + idx, 1), ik = input(9, TR_K + idx, 1);
      SpreadU32 es = rebind_spread(e_s, ie), fs = rebind_spread(f_s, if_), gs = rebind_spread(g_s, ig);
      AV sigma_term = sigma_upper1(es);                                      // :130
      AV ch_term = ch(es, fs, gs);                                           // :131
      AV add1 = add_new(EX(rebind(h, ih)), EX(sigma_term), 33);              // :138-142
      AV add2 = add_new(EX(add1), EX(ch_term), 34);                          // :143-147
      QC kc = Cdyn(ik, fr::from_u64(round_constants()[idx]));
      AV add3 = add(EX(add2), kc, emit(OP_ADD, operand(add2.s), operand(ik), 0, 35));   // :148-152
      AV add4 = add_new(EX(add3), EX(rebind(w[idx], iw)), 36);               // :153-157
      AV t1 = mod_u32(add4);                                                 // :158
      SpreadU32 as = rebind_spread(a_s, ia), bs = rebind_spread(b_s, ib), cs = rebind_spread(c_s, ic);
      AV sigma0 = sigma_upper0(as);                                          // :164
      AV maj_term = maj(as, bs, cs);                                         // :165
      AV addt2 = add_new(EX(sigma0), EX(maj_term), 33);                      // :166-170
      AV t2 = mod_u32(addt2);                                                // :171
      h = g; g = f; g_s = f_s; f = e; f_s = e_s;                             // :174-179
      AV adde = add_new(EX(rebind(d, id)), EX(t1), 33);                      // :181
      e = mod_u32(adde);                                                     // :182
      e_s = state_to_spread_u32(e);                                          // :184
      d = c; c = b; c_s = b_s; b = a; b_s = a_s;                             // :185-190
      AV adda = add_new(EX(t1), EX(t2), 33);                                 // :192
      a = mod_u32(adda);                                                     // :193
      a_s = state_to_spread_u32(a);                                          // :195
      end_unit();
    }
    end_group();
    AV ns[8] = {a, b, c, d, e, f, g, h};                                     // :197-212
    begin_group("FFA", 4);
    for (int i = 0; i < 4; i++) {
      begin_unit();
      Sym x = input(0, TR_A + 67 - i, -1), y = input(1, TR_A + 3 - i, -1);
      next[i] = mod_u32(add_new(EX(rebind(ns[i], x)), EX(rebind(pre[i], y)), 33));
      end_unit();
    }
    end_group();
    begin_group("FFE", 4);
    for (int i = 0; i < 4; i++) {
      begin_unit();
      Sym x = input(0, TR_E + 67 - i, -1), y = input(1, TR_E + 3 - i, -1);
      next[4 + i] = mod_u32(add_new(EX(rebind(ns[4 + i], x)), EX(rebind(pre[4 + i], y)), 33));
      end_unit();
    }
    end_group();
    commit_class(0, *blk);
  }

  void commit_class(uint32_t id, const ClassRec& c) {
    if (class_recs_.size() <= id) { class_recs_.resize(id + 1); class_set_.resize(id + 1, false); }
    if (!class_set_[id]) { class_recs_[id] = c; class_set_[id] = true; return; }
    const ClassRec& o = class_recs_[id];
    if (o.groups.size() != c.groups.size()) fail("job class shape differs between instances");
    for (size_t i = 0; i < c.groups.size(); i++)
      if (!o.groups[i].same_as(c.groups[i])) fail("job class group differs between instances: " + c.groups[i].type);
  }

  // ======================================================================================
  // src/lib.rs:71-349  Sha256DynamicConfig::digest
  // ======================================================================================
  void digest(uint32_t d) {
    const uint32_t M = cfg_.max_variable_byte_sizes[d], Rn = M / 64;
    const uint32_t lb = cfg_.lookup_bits;
    ClassRec dig, blk;
    use_class(&dig);
    DigestPlace dp{};
    dp.max_bytes = M; dp.n_blocks = Rn; dp.gate_base = n_gate_; dp.lk_base = n_lk_; dp.limb_base = n_limb_;
    dp.job_class = 1 + d;
    const int32_t words_base = TD_STATES + 8 * (int32_t)(Rn + 1);
    dp.trace_words = (uint32_t)words_base + 16 * Rn;
    DigestHandles hd;
    AV a_target, st0[8];
    // ---- prologue: length check (:122-151) + precomputed state words (:162-165) ----
    begin_group("PRO", 1); begin_unit();
    {
      Sym len = input(0, TD_LEN, 0), nr = input(1, TD_NUM_ROUND, 0), pr = input(2, TD_PRE_ROUND, 0), tg = input(3, TD_TARGET, 0);
      Sym s0[8]; for (int i = 0; i < 8; i++) s0[i] = input(4 + i, TD_STATES + i, 0);
      AV a_len = load_witness(len);                                          // :124-125
      AV a_nr = load_witness(nr);                                            // :126
      QC c64 = C(64);
      AV a_padded = mul(EX(a_nr), c64, emit(OP_MULADD, operand(nr), operand(c64), vm_operand_const(raw_const(0)), 40));   // :127-131
      QC c9 = C(9);
      AV a_with9 = add(EX(a_len), c9, emit(OP_ADD, operand(len), operand(c9), 0, 33));                                   // :132-136
      AV padding = sub(EX(a_padded), EX(a_with9), emit(OP_SUB, operand(a_padded.s), operand(a_with9.s), 0, 32));         // :137-141
      // range.is_less_than_safe(padding, 64) (:142-143)
      uint32_t range_bits = (7 + lb - 1) / lb * lb;  // bit_length(64) == 7
      range_check(padding, range_bits);
      uint32_t k = (range_bits + lb - 1) / lb, padded_bits = k * lb;
      if (padded_bits + lb > 62) fail("lookup_bits too large for is_less_than");
      U256 pw = pow2(padded_bits);
      Sym shift_a = emit(OP_ADD, operand(padding.s), vm_operand_const(raw_const(1ULL << padded_bits)), 0, padded_bits + 1);
      Sym shifted = emit(OP_SUB, operand(shift_a), operand(c64), 0, padded_bits + 1);
      std::vector<AV> o;
      assign_region({W(shifted), c64, C(1), W(shift_a), CU(fr::neg(pw)), C(1), EX(padding)}, {0, 3}, &o);
      AV last = range_check(o[0], padded_bits + lb);
      // is_zero(last limb): in a valid witness the limb is 0 (padding < 64), but stay general (limb in {0,1})
      Sym z = emit(OP_EQ, operand(last.s), vm_operand_const(raw_const(0)), 0, 1);
      Sym ib = emit(OP_ADD, operand(last.s), vm_operand_const(raw_const(inv_bias_)), 0, 8);
      AV lt = is_zero(last, z, table(T_INV, ib));
      assert_is_const(lt, fr::from_u64(1));                                  // :144
      AV a_pre = load_witness(pr);                                           // :145-146
      a_target = sub(EX(a_nr), EX(a_pre), tg);                               // :147-151
      for (int i = 0; i < 8; i++) st0[i] = load_witness(s0[i]);              // :162-165
      hd.input_len_idx = a_len.idx;
    }
    end_unit(); end_group();
    // ---- input bytes (:170-173) ----
    std::vector<AV> in_bytes(M);
    begin_group("INB", Rn);
    for (uint32_t j = 0; j < Rn; j++) {
      begin_unit();
      Sym wj[16]; for (int i = 0; i < 16; i++) wj[i] = input(i, words_base + 16 * (int32_t)j + i, 16);
      for (int b = 0; b < 64; b++) in_bytes[64 * j + b] = load_witness(sub(wj[b / 4], 24 - 8 * (b % 4), 8));
      end_unit();
    }
    end_group();
    for (uint32_t i = 0; i < M; i++) hd.input_bytes_idx.push_back(in_bytes[i].idx);
    if (cfg_.is_input_range_check) {                                         // :174-178
      begin_group("INRC", Rn);
      for (uint32_t j = 0; j < Rn; j++) {
        begin_unit();
        Sym wj[16]; for (int i = 0; i < 16; i++) wj[i] = input(i, words_base + 16 * (int32_t)j + i, 16);
        for (int b = 0; b < 64; b++) range_check(rebind(in_bytes[64 * j + b], sub(wj[b / 4], 24 - 8 * (b % 4), 8)), 8);
        end_unit();
      }
      end_group();
    }
    // ---- the block loop (:179-238) ----
    std::vector<std::array<AV, 8>> states(Rn + 1);
    for (int i = 0; i < 8; i++) states[0][i] = st0[i];
    for (uint32_t j = 0; j < Rn; j++) {
      std::vector<AV> bytes(in_bytes.begin() + 64 * j, in_bytes.begin() + 64 * (j + 1));
      uint32_t g0 = n_gate_, l0 = n_lk_, m0 = n_limb_;
      bool had_zero = has_zero_;
      sha256_compression(&blk, &dig, bytes, states[j].data(), states[j + 1].data());
      if (!had_zero) g0 += 1;
      if (j == 0) { dp.blk_gate_base = g0; dp.blk_lk_base = l0; dp.blk_limb_base = m0; }
      if (j == 1) { dp.blk_gate_stride = g0 - dp.blk_gate_base; dp.blk_lk_stride = l0 - dp.blk_lk_base; dp.blk_limb_stride = m0 - dp.blk_limb_base; }
      if (j >= 1 && (g0 != dp.blk_gate_base + j * dp.blk_gate_stride || l0 != dp.blk_lk_base + j * dp.blk_lk_stride ||
                     m0 != dp.blk_limb_base + j * dp.blk_limb_stride))
        fail("non-uniform block stride");
    }
    use_class(&dig);
    // ---- round selection (:294-310) ----
    AV zero = load_zero();  // cached by now
    AV out_h[8]; for (int i = 0; i < 8; i++) out_h[i] = zero;
    begin_group("SEL", Rn + 1);
    for (uint32_t n = 0; n <= Rn; n++) {
      begin_unit();
      Sym in_n = input(0, -1, 0), tg = input(1, TD_TARGET, 0);
      Sym st[8], H[8];
      for (int i = 0; i < 8; i++) st[i] = input(2 + i, TD_STATES + 8 * (int32_t)n + i, 8);
      for (int i = 0; i < 8; i++) H[i] = input(10 + i, TD_H + i, 0);
      // is_equal(Constant(n), target) = is_zero(sub(n, target))
      Sym Dn = emit(OP_SUB, operand(in_n), operand(tg), 0, 64);
      std::vector<AV> o;
      assign_region({W(signed_slot(Dn.slot)), EX(rebind(a_target, tg)), C(1), Cdyn(in_n, fr::from_u64(n))}, {0}, &o);
      Sym z = emit(OP_EQ, operand(in_n), operand(tg), 0, 1);
      Sym ib = emit(OP_ADD, operand(Dn), vm_operand_const(raw_const(inv_bias_)), 0, 8);
      AV selector = is_zero(o[0], z, table(T_INV, ib));
      Sym gt = emit(OP_GT, operand(in_n), operand(tg), 0, 1);
      for (int i = 0; i < 8; i++) {
        // output_h_out[i] before this step: state[target] once n > target, else the zero cell
        Sym bprev = emit(OP_MULADD, operand(gt), operand(H[i]), vm_operand_const(raw_const(0)), 32);
        Sym df = emit(OP_SUB, operand(st[i]), operand(bprev), 0, 64);
        Sym ov = emit(OP_SEL, operand(z), operand(st[i]), operand(bprev), 32);
        // every instance uses the same template symbol for b (for n == 0 b is the cached zero cell and bprev == 0)
        QC bq = EX((n == 0) ? out_h[i] : rebind(out_h[i], bprev));
        bq.s = bprev;
        out_h[i] = select(EX(rebind(states[n][i], st[i])), bq, EX(selector), signed_slot(df.slot), ov);
      }
      end_unit();
    }
    end_group();
    // ---- digest bytes (:311-341) ----
    begin_group("DIG", 1); begin_unit();
    {
      Sym H[8]; for (int i = 0; i < 8; i++) H[i] = input(i, TD_H + i, 0);
      for (int wi = 0; wi < 8; wi++) {
        AV bytes[4];
        for (int idx = 0; idx < 4; idx++) {
          bytes[idx] = load_witness(sub(H[wi], 24 - 8 * idx, 8));            // :319-320
          range_check(bytes[idx], 8);                                        // :321
          hd.output_bytes_idx[4 * wi + idx] = bytes[idx].idx;
        }
        AV sum = load_zero();                                                // :325
        for (int idx = 0; idx < 4; idx++)                                    // :326-333
          sum = mul_add(EX(bytes[idx]), C(1ULL << (24 - 8 * idx)), EX(sum), shl(sub(H[wi], 24 - 8 * idx, 8 * (idx + 1)), 24 - 8 * idx));
        assert_equal(rebind(out_h[wi], H[wi]), sum);                         // :334-338
      }
    }
    end_unit(); end_group();
    commit_class(1 + d, dig);
    P_->digests.push_back(dp);
    P_->handles.push_back(hd);
  }

  // ======================================================================================
  // finalize: chunk + de-duplicate the cells of every unit type, build tables, job classes, layout
  // ======================================================================================
  // normalised form of a symbolic value: small plain values come from the byte table instead of a Barrett reduction
  Sym normalise(const Sym& s0) const {
    Sym s = s0;
    if (s.kind == KIND_GENERIC && !s.neg && s.shl == 0 && s.w <= 8) { s.kind = KIND_TABLE; s.table = T_BYTE; s.tbl_off = 0; }
    if (s.kind == KIND_TABLE && s.w == 0) { s.slot = 0; s.sh = 0; s.shl = 0; s.neg = 0; }
    if (s.kind == KIND_SIGNED) { s.sh = 0; s.w = 64; s.shl = 0; s.neg = 0; }
    return s;
  }
  uint32_t table_index(const Sym& s) const {
    uint32_t tbl = 0;
    switch (s.table) {
      case T_CONST: tbl = s.tbl_off; break;
      case T_BYTE: tbl = P_->tb_byte + s.tbl_off; break;
      case T_SBYTE: tbl = P_->tb_sbyte + s.tbl_off; break;
      case T_INV: tbl = P_->tb_inv + s.tbl_off; break;
    }
    if (s.table == T_SBYTE && s.w > cfg_.limb_bits) fail("spread-table index wider than a limb");
    if (tbl > 0xffff) fail("static table too large");
    return tbl;
  }
  std::map<uint32_t, uint32_t> resident_slot_;   // const table index -> fixed scratch slot
  bool is_resident(const Sym& s) const { return s.kind == KIND_TABLE && s.w == 0 && resident_slot_.count(table_index(s)); }
  // a spread-column cell: the dense cell (even dst) is a limb-wide extract whose slot / shift the kernel also uses for the table-row
  // multiplicities; the spread cell is its table image (num_bits_lookup <= 8) or the 32-bit spread slot (num_bits_lookup = 16)
  bool limb_cell_ok(const Sym& s, uint32_t dst) const {
    if ((dst & 1u) == 0) return (s.kind == KIND_TABLE && s.table == T_BYTE && s.w == cfg_.limb_bits) || (s.kind == KIND_GENERIC && !s.neg && s.shl == 0 && s.w == cfg_.limb_bits);
    return (s.kind == KIND_TABLE && s.table == T_SBYTE && s.w == cfg_.limb_bits) || (cfg_.limb_bits == 16 && s.kind == KIND_GENERIC && !s.neg && s.shl == 0 && s.w == 32);
  }
  // sort class of a fill entry: table copies, then <= 32-bit Barrett, then the full 64-bit / signed path
  static int fill_class(const Sym& s) {
    if (s.kind == KIND_TABLE) return 0;
    if (s.kind == KIND_GENERIC && (uint32_t)s.w + s.shl <= 32) return 1;
    return 2;
  }
  static uint64_t sym_key(const Sym& s) {
    return (uint64_t)s.kind | ((uint64_t)s.neg << 2) | ((uint64_t)s.slot << 3) | ((uint64_t)s.sh << 11) | ((uint64_t)s.w << 17) |
           ((uint64_t)s.shl << 24) | ((uint64_t)s.table << 29) | ((uint64_t)s.tbl_off << 32);
  }

  // Cuts one unit's cell stream into chunks of at most cfg_.max_fill distinct values.
  // (position of a unit's first gate cell inside its output column) mod 8, over every occurrence of the unit type in
  // an instance: the copy loop aligns its lanes to 256-byte groups of the output, so these are the only ways the
  // cells of a chunk can be grouped into quarter-warps.
  std::map<std::string, std::set<uint32_t>> align_;
  std::set<uint32_t> cur_align_;
  uint64_t stat_cost_greedy_ = 0, stat_cost_final_ = 0, stat_cost_ideal_ = 0, stat_norm_ = 1;   // shared-memory wavefronts of the unit type being chunked
  void compute_alignments() {
    Plan& P = *P_;
    auto residue = [&](uint32_t gidx) {
      size_t c = 0;
      while (c + 1 < P.breaks.size() && P.breaks[c + 1] <= gidx) c++;
      return (gidx - P.breaks[c]) & 7u;
    };
    for (size_t ci = 0; ci < class_recs_.size(); ci++) {
      const ClassRec& c = class_recs_[ci];
      std::vector<uint32_t> origins;
      if (ci == 0) {
        for (const DigestPlace& dp : P.digests)
          for (uint32_t j = 0; j < dp.n_blocks; j++) origins.push_back(dp.blk_gate_base + j * dp.blk_gate_stride);
      } else {
        origins.push_back(0);
      }
      for (const GroupRec& g : c.groups)
        for (uint32_t o : origins)
          for (uint32_t u = 0; u < g.count; u++) align_[g.type].insert(residue(o + g.gate_base + u * g.gate_stride));
    }
  }

  void build_chunks(const UnitRec& u, UnitType* ut) {
    // pass 1: greedy, to learn how many chunks the distinct-value limit forces; pass 2: the same number of chunks with
    // balanced cell counts (multiples of 32 gate cells)
    Plan& P = *P_;
    const size_t f0 = P.fill.size(), c0 = P.cells.size(), k0 = P.chunks.size();
    build_chunks_pass(u, ut, 0xffffffffu);
    const uint32_t n = ut->n_chunks;
    if (n > 1) {
      P.fill.resize(f0); P.cells.resize(c0); P.chunks.resize(k0);
      uint32_t cap = ((ut->gate_len + n - 1) / n + 31) / 32 * 32;
      build_chunks_pass(u, ut, cap);
    }
  }
  void build_chunks_pass(const UnitRec& u, UnitType* ut, uint32_t max_gate_cells) {
    Plan& P = *P_;
    ut->chunk_off = (uint32_t)P.chunks.size();
    struct Pending { uint8_t kind; Sym s; uint32_t dst; };
    std::vector<Pending> cur;
    std::map<uint64_t, Sym> distinct;
    uint32_t n_gate = 0, n_lk = 0, n_limb = 0, gate_in_chunk = 0;
    auto flush = [&]() {
      if (cur.empty()) return;
      // spread-column cells: group them by output column (dense_0.., spread_0..) so that consecutive lanes store to
      // consecutive rows of one column (the limb entries keep their slots in `cur`, only their order changes)
      {
        const uint32_t nc = cfg_.spread_cols;
        std::vector<size_t> where;
        std::vector<Pending> limbs;
        for (size_t i2 = 0; i2 < cur.size(); i2++) if (cur[i2].kind == EV_LIMB) { where.push_back(i2); limbs.push_back(cur[i2]); }
        std::stable_sort(limbs.begin(), limbs.end(), [&](const Pending& a, const Pending& b) {
          return (a.dst & 1u) * nc + (a.dst >> 1) % nc < (b.dst & 1u) * nc + (b.dst >> 1) % nc;
        });
        for (size_t i2 = 0; i2 < where.size(); i2++) cur[where[i2]] = limbs[i2];
      }
      // order the distinct values: TABLE | GENERIC32 | GENERIC64, stable by first use
      std::vector<Sym> order;
      std::map<uint64_t, uint32_t> index;
      for (int cls = 0; cls < 3; cls++)
        for (auto& pc : cur) {
          if (fill_class(pc.s) != cls) continue;
          uint64_t k = sym_key(pc.s);
          if (index.count(k)) continue;
          index[k] = (uint32_t)order.size();
          order.push_back(pc.s);
        }
      // ---- scratch slot of every distinct value, chosen to avoid shared-memory bank conflicts in the copy loops ----
      // A 128-bit shared load is served one quarter-warp (8 lanes x 16 B) at a time: two lanes of a quarter conflict
      // when they read different slots with the same (slot mod 8).  Greedy colouring of the co-occurrence graph;
      // resident constants have fixed slots [0, n_resident).
      const uint32_t nd = (uint32_t)order.size();
      std::vector<std::map<uint32_t, uint32_t>> adj(nd);
      for (int kind = 0; kind < 3; kind++) {
        std::vector<uint32_t> seq;
        for (auto& pc : cur) if (pc.kind == kind) seq.push_back(index.at(sym_key(pc.s)));
        // the gate copy loop aligns its lanes to 256-byte groups of the output at run time, so a quarter-warp holds the
        // cells whose (position mod 32) lie in the same group of 8: enumerate the possible alignments of this chunk.
        // Lookup / limb loops start at cell 0: fixed quarters.
        if (kind == EV_GATE) {
          uint32_t first_dst = 0xffffffffu;
          for (auto& pc : cur) if (pc.kind == EV_GATE) first_dst = std::min(first_dst, pc.dst);
          for (uint32_t a : cur_align_) {
            const uint32_t r = (a + first_dst) & 7u;   // position mod 8 of seq[0]
            for (size_t i0 = 0; i0 < seq.size(); i0++)
              for (size_t i1 = i0 + 1; i1 < seq.size() && (i1 + r) / 8 == (i0 + r) / 8; i1++)
                if (seq[i0] != seq[i1]) { adj[seq[i0]][seq[i1]]++; adj[seq[i1]][seq[i0]]++; }
          }
        } else {
          for (size_t q = 0; q < seq.size(); q += 8) {
            size_t qe = std::min(seq.size(), q + 8);
            for (size_t a = q; a < qe; a++)
              for (size_t b = a + 1; b < qe; b++)
                if (seq[a] != seq[b]) { adj[seq[a]][seq[b]] += (uint32_t)cur_align_.size(); adj[seq[b]][seq[a]] += (uint32_t)cur_align_.size(); }
          }
        }
      }
      const uint32_t n_res = (uint32_t)P.resident.size();
      std::vector<int> residue(nd, -1);
      std::vector<uint32_t> loc(nd, 0);
      std::vector<uint8_t> resident(nd, 0);
      // free slots per residue class: all slots >= n_res
      std::vector<std::vector<uint32_t>> free_slots(8);
      for (uint32_t sl = cfg_.max_fill; sl-- > n_res;) free_slots[sl % 8].push_back(sl);   // back() = smallest free slot
      uint32_t cap_left[8];
      for (int r = 0; r < 8; r++) cap_left[r] = (uint32_t)free_slots[r].size();
      uint32_t n_dyn = 0;
      for (uint32_t i2 = 0; i2 < nd; i2++) {
        if (is_resident(order[i2])) { resident[i2] = 1; loc[i2] = resident_slot_.at(table_index(order[i2])); residue[i2] = (int)(loc[i2] % 8); }
        else n_dyn++;
      }
      if (n_dyn + n_res > cfg_.max_fill) fail("chunk has too many distinct values");
      std::vector<uint32_t> by_weight;
      std::vector<uint64_t> wsum(nd, 0);
      for (uint32_t i2 = 0; i2 < nd; i2++) { if (!resident[i2]) by_weight.push_back(i2); for (auto& kv : adj[i2]) wsum[i2] += kv.second; }
      std::stable_sort(by_weight.begin(), by_weight.end(), [&](uint32_t a, uint32_t b) { return wsum[a] > wsum[b]; });
      for (uint32_t vi : by_weight) {
        uint64_t cost[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (auto& kv : adj[vi]) if (residue[kv.first] >= 0) cost[residue[kv.first]] += kv.second;
        int best = -1;
        for (int r = 0; r < 8; r++)
          if (cap_left[r] && (best < 0 || cost[r] < cost[best] || (cost[r] == cost[best] && cap_left[r] > cap_left[best]))) best = r;
        if (best < 0) fail("scratch colouring out of space");
        residue[vi] = best;
        cap_left[best]--;
      }
      // ---- local search on the exact cost: shared-memory wavefronts of one execution of the chunk ----
      // A quarter-warp access costs max over the 8 bank groups of the number of DISTINCT slots it touches there
      // (tools/lsu_probe.cu: conflicts inside a quarter serialise even when the warp as a whole is balanced).  Reads:
      // every quarter of the three copy loops (per possible alignment of the chunk in its output column).  Writes: the
      // fill loops store 8 consecutive fill entries per quarter; with the round-robin order emitted below a class of n
      // values costs max(ceil(n / 8), largest residue class), so the classes are balanced here as well.
      {
        struct Quarter { std::vector<uint32_t> vs; uint32_t w; };
        std::vector<Quarter> quarters;
        auto add_quarter = [&](std::vector<uint32_t> vs, uint32_t w) {
          std::sort(vs.begin(), vs.end());
          vs.erase(std::unique(vs.begin(), vs.end()), vs.end());
          if (vs.size() > 1) quarters.push_back(Quarter{vs, w});
        };
        const uint32_t n_al = (uint32_t)cur_align_.size();
        for (int kind = 0; kind < 3; kind++) {
          std::vector<uint32_t> seq;
          uint32_t first_dst = 0xffffffffu;
          for (auto& pc : cur) if (pc.kind == kind) { seq.push_back(index.at(sym_key(pc.s))); first_dst = std::min(first_dst, pc.dst); }
          if (seq.empty()) continue;
          // every copy loop aligns its lanes to the 256-byte groups of the output at run time: a quarter holds the cells
          // whose position falls into the same group of 8; enumerate the alignments this chunk can have
          std::map<uint32_t, uint32_t> shifts;   // shift -> number of alignments that produce it
          if (kind == EV_GATE) for (uint32_t a : cur_align_) shifts[(a + first_dst) & 7u]++;
          else if (kind == EV_LK) for (uint32_t sh = 0; sh < 8; sh++) shifts[sh] = n_al;   // lookup stream: any alignment, equally likely
          else shifts[0] = n_al * 8u;                                                       // limb loop: lanes start at cell 0
          for (auto& sw : shifts) {
            std::vector<uint32_t> q;
            for (size_t i0 = 0; i0 < seq.size(); i0++) {
              if (i0 && (i0 + sw.first) % 8 == 0) { add_quarter(q, sw.second * (kind == EV_GATE ? 8u : 1u)); q.clear(); }
              q.push_back(seq[i0]);
            }
            add_quarter(q, sw.second * (kind == EV_GATE ? 8u : 1u));
          }
        }
        std::vector<std::vector<uint32_t>> memb(nd);
        for (uint32_t q = 0; q < quarters.size(); q++) for (uint32_t v : quarters[q].vs) memb[v].push_back(q);
        auto qcost = [&](const Quarter& q) {
          uint32_t c8[8] = {0, 0, 0, 0, 0, 0, 0, 0}, m = 0;
          for (uint32_t v : q.vs) m = std::max(m, ++c8[residue[v]]);
          return m * q.w;
        };
        // fill classes for the write cost: 0 = table copies, 1 = Barrett (32- and 64-bit entries share one loop)
        auto wclass = [&](uint32_t v) { return fill_class(order[v]) == 0 ? 0 : 1; };
        uint32_t ccount[2][8] = {{0}}, ctotal[2] = {0, 0};
        for (uint32_t v = 0; v < nd; v++) if (!resident[v]) { ccount[wclass(v)][residue[v]]++; ctotal[wclass(v)]++; }
        auto fcost = [&]() {
          uint32_t t = 0;
          for (int c = 0; c < 2; c++) {
            uint32_t m = (ctotal[c] + 7) / 8;
            for (int r = 0; r < 8; r++) m = std::max(m, ccount[c][r]);
            t += m;
          }
          return t * n_al * 8u;
        };
        auto local_cost = [&](uint32_t v, uint32_t u) {   // cost of the quarters touching v (and u, if any), each counted once
          uint64_t t = fcost();
          for (uint32_t q : memb[v]) t += qcost(quarters[q]);
          if (u != ~0u)
            for (uint32_t q : memb[u]) if (!std::binary_search(quarters[q].vs.begin(), quarters[q].vs.end(), v)) t += qcost(quarters[q]);
          return t;
        };
        uint64_t total0 = fcost();
        for (auto& q : quarters) total0 += qcost(q);
        uint64_t total = total0;
        std::vector<uint32_t> dyn;
        for (uint32_t v = 0; v < nd; v++) if (!resident[v]) dyn.push_back(v);
        for (int sweep = 0; sweep < 12; sweep++) {
          bool improved = false;
          for (uint32_t v : dyn) {
            const int r0 = residue[v];
            const int cv = wclass(v);
            int64_t best_gain = 0; int best_r = -1; uint32_t best_u = ~0u;
            for (int r = 0; r < 8; r++) {
              if (r == r0 || !cap_left[r]) continue;
              const uint64_t before = local_cost(v, ~0u);
              residue[v] = r; ccount[cv][r0]--; ccount[cv][r]++;
              const uint64_t after = local_cost(v, ~0u);
              residue[v] = r0; ccount[cv][r0]++; ccount[cv][r]--;
              const int64_t gain = (int64_t)before - (int64_t)after;
              if (gain > best_gain) { best_gain = gain; best_r = r; best_u = ~0u; }
            }
            for (uint32_t u : dyn) {
              const int r = residue[u];
              if (r == r0) continue;
              const int cu = wclass(u);
              const uint64_t before = local_cost(v, u);
              residue[v] = r; residue[u] = r0; ccount[cv][r0]--; ccount[cv][r]++; ccount[cu][r]--; ccount[cu][r0]++;
              const uint64_t after = local_cost(v, u);
              residue[v] = r0; residue[u] = r; ccount[cv][r0]++; ccount[cv][r]--; ccount[cu][r]++; ccount[cu][r0]--;
              const int64_t gain = (int64_t)before - (int64_t)after;
              if (gain > best_gain) { best_gain = gain; best_r = r; best_u = u; }
            }
            if (best_r >= 0) {
              if (best_u == ~0u) { cap_left[r0]++; cap_left[best_r]--; }
              else { residue[best_u] = r0; const int cu = wclass(best_u); ccount[cu][best_r]--; ccount[cu][r0]++; }
              residue[v] = best_r; ccount[cv][r0]--; ccount[cv][best_r]++;
              total -= (uint64_t)best_gain;
              improved = true;
            }
          }
          if (!improved) break;
        }
        uint64_t ideal = 0;
        for (auto& q : quarters) ideal += q.w;
        ideal += (uint64_t)n_al * 8u * ((ctotal[0] + 7) / 8 + (ctotal[1] + 7) / 8);
        stat_cost_greedy_ += total0; stat_cost_final_ += total; stat_cost_ideal_ += ideal; stat_norm_ = n_al * 8u;
      }
      for (uint32_t vi = 0; vi < nd; vi++) {
        if (resident[vi]) continue;
        if (free_slots[residue[vi]].empty()) fail("scratch colouring out of space");
        loc[vi] = free_slots[residue[vi]].back();
        free_slots[residue[vi]].pop_back();
      }
      // gate-checksum weights of every distinct value, and how many lookup-column cells carry it
      std::vector<uint32_t> cnt(nd, 0), sumdst(nd, 0), lkcnt(nd, 0);
      uint32_t dmin = 0xffff, dmax = 0;
      for (auto& pc : cur) {
        const uint32_t vi = index.at(sym_key(pc.s));
        if (pc.kind == EV_GATE) {
          cnt[vi]++; sumdst[vi] += pc.dst;
          dmin = std::min(dmin, pc.dst); dmax = std::max(dmax, pc.dst);
        } else if (pc.kind == EV_LK) {
          // the fused multiplicity count reads the raw value of a looked-up cell from its fill entry: a byte-table value or a
          // plain (shifted) extract -- the only kinds the reference ever range-checks
          const Sym& sy = order[vi];
          const bool ok = (sy.kind == KIND_TABLE && sy.table == T_BYTE) || (sy.kind == KIND_GENERIC && !sy.neg);
          if (!ok || resident[vi]) fail("a looked-up cell holds a constant, a negated or a signed value");
          lkcnt[vi]++;
        }
      }
      for (uint32_t i2 = 0; i2 < nd; i2++) if (cnt[i2] > 0xffff || lkcnt[i2] > 0xffff) fail("chunk too large for the fill-entry counters");
      Chunk c{};
      c.fill_off = (uint32_t)P.fill.size();
      c.gate_dst_min = (uint16_t)dmin; c.gate_dst_max = (uint16_t)dmax;
      for (uint32_t i2 = 0; i2 < nd; i2++)
        if (resident[i2] && cnt[i2]) {
          const uint32_t* x = reinterpret_cast<const uint32_t*>(P.mont_table[table_index(order[i2])].l);
          uint32_t h = 0;
          for (int k = 0; k < 8; k++) h += x[k] * kCkM[k];
          c.res_a += (uint64_t)h * (2ull * sumdst[i2]);
          c.res_b += (uint64_t)h * (uint64_t)cnt[i2];
        }
      // emit the fill list class by class, each class sorted by scratch slot (conflict-free scratch writes); resident
      // constants need no fill entry but their gate-checksum weight is folded into one "virtual" entry per constant
      for (int cls = 0; cls < 3; cls++) {
        std::vector<uint32_t> ids;
        for (uint32_t i2 = 0; i2 < nd; i2++) if (fill_class(order[i2]) == cls) ids.push_back(i2);
        // order: round-robin over the 8 bank-group residues of the scratch slots, so that the 8 lanes of a quarter-warp
        // write (and the fill loop reads) different bank groups
        {
          std::vector<std::vector<uint32_t>> by_res(8);
          std::stable_sort(ids.begin(), ids.end(), [&](uint32_t a, uint32_t b) { return loc[a] < loc[b]; });
          for (uint32_t i2 : ids) by_res[loc[i2] % 8].push_back(i2);
          std::vector<uint32_t> inter;
          for (size_t round = 0; inter.size() < ids.size(); round++)
            for (int r = 0; r < 8; r++)
              if (round < by_res[r].size()) inter.push_back(by_res[r][round]);
          ids.swap(inter);
        }
        for (uint32_t i2 : ids) {
          const Sym& sy = order[i2];
          if (resident[i2]) continue;
          if (cls == 0) c.n_fill_table++;
          if (cls == 1) c.n_fill32++;
          c.n_fill++;
          TmplEntry te = tmpl_pack(loc[i2], sy.kind == KIND_TABLE ? table_index(sy) : 0, sy.slot, sy.sh, sy.w, sy.shl, sy.kind, sy.neg);
          P.fill.push_back(FillEntry{te.lo, te.hi, cnt[i2] | (lkcnt[i2] << 16), sumdst[i2]});
        }
      }
      for (int kind = 0; kind < 3; kind++) {
        uint32_t off = (uint32_t)P.cells.size(), n = 0;
        for (auto& pc : cur) {
          if (pc.kind != kind) continue;
          const uint32_t sl = loc[index.at(sym_key(pc.s))];
          if (kind == EV_LIMB) {
            // src (8) | dst (10) | slot (8) | sh (6): where the limb's raw value sits (dense: the extract itself; spread: its table index)
            if (sl > 0xff || pc.dst > 0x3ff || !limb_cell_ok(pc.s, pc.dst)) fail("spread-column cell does not fit its descriptor");
            P.cells.push_back(CellEntry{sl | (pc.dst << 8) | ((uint32_t)pc.s.slot << 18) | ((uint32_t)pc.s.sh << 26)});
          } else {
            P.cells.push_back(CellEntry{sl | (pc.dst << 16)});
          }
          n++;
        }
        if (kind == EV_GATE) { c.gate_off = off; c.gate_len = (uint16_t)n; }
        if (kind == EV_LK) { c.lk_off = off; c.lk_len = (uint16_t)n; }
        if (kind == EV_LIMB) { c.limb_off = off; c.limb_len = (uint16_t)n; }
      }
      P.chunks.push_back(c);
      cur.clear(); distinct.clear(); gate_in_chunk = 0;
    };
    // greedy: close the chunk at a multiple of 32 gate cells once the next 32-cell group could overflow the scratch table
    size_t i = 0;
    while (i < u.ev.size()) {
      // next group: events up to and including the 32nd gate cell from here (plus the lookup / limb events in between)
      size_t j = i; uint32_t g = 0;
      while (j < u.ev.size() && !(g == 32 && u.ev[j].kind == EV_GATE)) { if (u.ev[j].kind == EV_GATE) g++; j++; }
      std::map<uint64_t, Sym> trial = distinct;
      for (size_t k = i; k < j; k++) {
        Sym sy = normalise(u.ev[k].s);
        trial[sym_key(sy)] = sy;
      }
      auto scratch_need = [&](const std::map<uint64_t, Sym>& m) {
        size_t n = P.resident.size();
        for (auto& kv : m) if (!is_resident(kv.second)) n++;
        return n;
      };
      if ((scratch_need(trial) > cfg_.max_fill || gate_in_chunk + g > max_gate_cells) && !cur.empty()) { flush(); continue; }
      if (scratch_need(trial) > cfg_.max_fill) fail("a 32-cell group has more distinct values than max_fill");
      for (size_t k = i; k < j; k++) {
        Sym sy = normalise(u.ev[k].s);
        uint32_t dst = (u.ev[k].kind == EV_GATE) ? n_gate++ : (u.ev[k].kind == EV_LK) ? n_lk++ : n_limb++;
        if (dst > 0xffff) fail("unit too large");
        cur.push_back(Pending{u.ev[k].kind, sy, dst});
        if (u.ev[k].kind == EV_GATE) gate_in_chunk++;
      }
      distinct.swap(trial);
      i = j;
    }
    flush();
    ut->n_chunks = (uint32_t)P.chunks.size() - ut->chunk_off;
    ut->gate_len = n_gate; ut->lk_len = n_lk; ut->limb_len = n_limb;
    if (n_gate != u.gate.size() || n_lk != u.lk.size() || n_limb != u.limb.size()) fail("event list out of sync");
  }

  // cost estimate of one work item (for the heaviest-first ordering)
  uint32_t chunk_cost(const Chunk& c) const {
    return 3u * c.n_fill_table + 12u * (c.n_fill - c.n_fill_table) + c.gate_len + c.lk_len + c.limb_len + 32u;
  }

  // appends a JobClass made of `groups` (already with final counts / bases / input maps)
  // appends a JobClass made of `groups` (final per-instance counts / bases / input maps); one job covers `batch`
  // consecutive circuit instances: unit instance u' of a group belongs to instance u' / per_inst
  void add_class(const std::vector<UnitGroup>& groups_in, uint32_t n_trace_words, uint32_t batch) {
    Plan& P = *P_;
    JobClass jc{};
    jc.group_off = (uint32_t)P.groups.size(); jc.n_groups = (uint32_t)groups_in.size();
    jc.batch = batch;
    if (groups_in.size() > 255) fail("too many groups in a job class");
    if (batch == 0 || batch > H2SHA_MAX_JOB_BATCH) fail("bad job batch");
    std::vector<UnitGroup> groups = groups_in;
    uint32_t slot_base = 0;
    for (UnitGroup& g : groups) {
      g.per_inst = g.count;
      g.count = g.per_inst * batch;
      g.slot_base = slot_base;
      slot_base += g.count * (P.types[g.type].n_slots | 1u);
      P.groups.push_back(g);   // g.dict_base was set by the caller (relative to the job's dictionary base)
    }
    jc.n_slots_total = slot_base;
    P.max_slots = std::max(P.max_slots, slot_base);
    // phase-1 warp tasks, longest program first
    jc.task_off = (uint32_t)P.tasks.size();
    std::vector<std::pair<uint32_t, WarpTask>> ts;
    for (uint32_t gi = 0; gi < groups.size(); gi++)
      for (uint32_t first = 0; first < groups[gi].count; first += 32) ts.push_back({P.types[groups[gi].type].prog_len, WarpTask{gi, first}});
    std::stable_sort(ts.begin(), ts.end(), [](const auto& x, const auto& y) { return x.first > y.first; });
    for (auto& t : ts) P.tasks.push_back(t.second);
    jc.n_tasks = (uint32_t)ts.size();
    // phase-2 items, heaviest first
    jc.item_off = (uint32_t)P.items.size();
    std::vector<std::pair<uint32_t, std::pair<ItemDesc, uint32_t>>> its;
    for (uint32_t gi = 0; gi < groups.size(); gi++) {
      const UnitGroup& g = groups[gi];
      const UnitType& ut = P.types[g.type];
      for (uint32_t u = 0; u < g.count; u++)
        for (uint32_t c = 0; c < ut.n_chunks; c++) {
          ItemDesc d{};
          const uint32_t slot_off = g.slot_base + u * (ut.n_slots | 1u);
          const uint32_t inst_off = u / g.per_inst, uu = u % g.per_inst;
          if (slot_off > 0xffff || ut.chunk_off + c > 0x7ff || inst_off > 31) fail("item descriptor overflow (job class too large)");
          d.gate_rel = g.gate_base + uu * g.gate_stride;
          d.lk_rel = g.lk_base + uu * g.lk_stride;
          d.limb_rel = g.limb_base + uu * g.limb_stride;
          d.slot_chunk = slot_off | ((ut.chunk_off + c) << 16) | (inst_off << 27);
          uint32_t dict_rel = g.dict_base + uu * ut.dict_len;
          for (uint32_t c2 = 0; c2 < c; c2++) dict_rel += P.chunks[ut.chunk_off + c2].n_fill;
          its.push_back({chunk_cost(P.chunks[ut.chunk_off + c]), {d, dict_rel}});
        }
    }
    std::stable_sort(its.begin(), its.end(), [](const auto& x, const auto& y) { return x.first > y.first; });
    for (auto& it : its) { P.items.push_back(it.second.first); P.item_dict.push_back(it.second.second); }
    jc.n_items = (uint32_t)its.size();
    jc.n_trace_words = n_trace_words;
    P.max_trace_words = std::max(P.max_trace_words, n_trace_words * batch);
    P.classes.push_back(jc);
  }

  UnitGroup make_group(const GroupRec& g, uint32_t first, uint32_t count) const {
    UnitGroup ug{};
    ug.type = type_idx_.at(g.type); ug.count = count;
    ug.gate_base = g.gate_base + first * g.gate_stride; ug.gate_stride = g.gate_stride;
    ug.lk_base = g.lk_base + first * g.lk_stride; ug.lk_stride = g.lk_stride;
    ug.limb_base = g.limb_base + first * g.limb_stride; ug.limb_stride = g.limb_stride;
    ug.dict_base = g.dict_base + first * P_->types[ug.type].dict_len;
    for (size_t i = 0; i < g.in.size(); i++) {
      ug.in[i] = g.in[i];
      if (ug.in[i].base >= 0) ug.in[i].base += g.in[i].stride * (int32_t)first;
      else ug.in[i].stride = (int32_t)first;  // instance-index input: value = stride + u
    }
    return ug;
  }

  // which dictionary entry (or resident constant) every cell of an instance copies: what the host-side expander of the compact
  // hand-off needs, derived from the same fill / cell lists the kernel walks
  void build_compact_map() {
    Plan& P = *P_;
    const uint32_t kUnset = 0xffffffffu;
    P.map_gate.assign(n_gate_, kUnset); P.map_lookup.assign(n_lk_, kUnset); P.map_dense.assign(n_limb_, kUnset); P.map_spread.assign(n_limb_, kUnset);
    auto map_unit = [&](const UnitType& ut, uint32_t gate0, uint32_t lk0, uint32_t limb0, uint32_t dict0) {
      uint32_t doff = dict0;
      std::vector<uint32_t> ent(std::max<uint32_t>(cfg_.max_fill, 1));
      for (uint32_t c = 0; c < ut.n_chunks; c++) {
        const Chunk& ch = P.chunks[ut.chunk_off + c];
        std::fill(ent.begin(), ent.end(), kUnset);
        for (uint32_t sl = 0; sl < P.resident.size(); sl++) ent[sl] = 0x80000000u | P.resident[sl];
        for (uint32_t i = 0; i < ch.n_fill; i++) ent[H2SHA_TE_DST(P.fill[ch.fill_off + i])] = doff + i;
        for (uint32_t i = 0; i < ch.gate_len; i++) { const CellEntry ce = P.cells[ch.gate_off + i]; P.map_gate[gate0 + H2SHA_CE_DST(ce)] = ent[H2SHA_CE_SRC(ce)]; }
        for (uint32_t i = 0; i < ch.lk_len; i++) { const CellEntry ce = P.cells[ch.lk_off + i]; P.map_lookup[lk0 + H2SHA_CE_DST(ce)] = ent[H2SHA_CE_SRC(ce)]; }
        for (uint32_t i = 0; i < ch.limb_len; i++) {
          const CellEntry ce = P.cells[ch.limb_off + i];
          const uint32_t n = limb0 + (H2SHA_LE_DST(ce) >> 1);
          ((H2SHA_LE_DST(ce) & 1u) ? P.map_spread : P.map_dense)[n] = ent[H2SHA_LE_SRC(ce)];
        }
        doff += ch.n_fill;
      }
    };
    auto map_class = [&](const ClassRec& c, uint32_t g0, uint32_t l0, uint32_t m0, uint32_t dict0) {
      for (const GroupRec& g : c.groups) {
        const UnitType& ut = P.types[type_idx_.at(g.type)];
        for (uint32_t u = 0; u < g.count; u++)
          map_unit(ut, g0 + g.gate_base + u * g.gate_stride, l0 + g.lk_base + u * g.lk_stride, m0 + g.limb_base + u * g.limb_stride, dict0 + g.dict_base + u * ut.dict_len);
      }
    };
    for (size_t d = 0; d < P.digests.size(); d++) {
      const DigestPlace& dp = P.digests[d];
      map_class(class_recs_[1 + d], 0, 0, 0, dp.dict_base);
      for (uint32_t j = 0; j < dp.n_blocks; j++)
        map_class(class_recs_[0], dp.blk_gate_base + j * dp.blk_gate_stride, dp.blk_lk_base + j * dp.blk_lk_stride, dp.blk_limb_base + j * dp.blk_limb_stride,
                  dp.dict_base + dp.dict_dig_len + j * dp.dict_blk_len);
    }
    for (auto* m : {&P.map_gate, &P.map_lookup, &P.map_dense, &P.map_spread})
      for (uint32_t v : *m) if (v == kUnset) fail("compact map: a cell has no dictionary entry");
  }

  void finalize() {
    Plan& P = *P_;
    P.cfg = cfg_;
    P.n_gate = n_gate_; P.n_lookup = n_lk_; P.n_limb = n_limb_;
    // ---- Montgomery table ----
    P.tb_byte = (uint32_t)consts_.size();
    P.tb_sbyte = P.tb_byte + 256;
    const uint32_t n_sbyte = cfg_.limb_bits <= 8 ? (1u << cfg_.limb_bits) : 0u;   // 16-bit limbs use no spread table (see spread_limb)
    P.tb_inv = P.tb_sbyte + n_sbyte;
    P.inv_bias = inv_bias_;
    for (auto& c : consts_) P.mont_table.push_back(fr::to_mont(c));
    for (uint32_t i = 0; i < 256; i++) P.mont_table.push_back(fr::to_mont(fr::from_u64(i)));
    for (uint32_t i = 0; i < n_sbyte; i++) {
      uint64_t sp = 0;
      for (int b = 0; b < 8; b++) sp |= (uint64_t)((i >> b) & 1) << (2 * b);
      P.mont_table.push_back(fr::to_mont(fr::from_u64(sp)));
    }
    for (int64_t dv = -(int64_t)inv_bias_; dv <= (int64_t)inv_bias_; dv++) {
      U256 v = fr::from_i64(dv);
      P.mont_table.push_back(fr::to_mont(dv == 0 ? fr::from_u64(1) : fr::inv(v)));
    }
    // ---- constants kept resident in every warp's scratch: the most used ones, weighted by instances per block ----
    {
      std::map<uint32_t, uint64_t> use;   // const table index -> weighted use count
      std::map<std::string, uint64_t> weight;
      for (const GroupRec& g : class_recs_[0].groups) weight[g.type] += g.count;
      for (auto& kv : type_idx_) {
        const uint64_t w = weight.count(kv.first) ? weight[kv.first] : 1;
        for (const Event& ev : type_recs_[kv.second].ev) {
          Sym sy = normalise(ev.s);
          if (sy.kind == KIND_TABLE && sy.w == 0) use[table_index(sy)] += w;
        }
      }
      std::vector<std::pair<uint64_t, uint32_t>> byuse;
      for (auto& kv : use) byuse.push_back({kv.second, kv.first});
      std::sort(byuse.begin(), byuse.end(), [](const auto& a, const auto& b) { return a.first > b.first || (a.first == b.first && a.second < b.second); });
      const uint32_t nres = std::min<uint32_t>({cfg_.resident_consts, (uint32_t)byuse.size(), cfg_.max_fill / 2});
      for (uint32_t i = 0; i < nres; i++) { resident_slot_[byuse[i].second] = i; P.resident.push_back(byuse[i].second); }
    }
    compute_alignments();
    // ---- unit types ----
    for (auto& kv : type_idx_) { if (P.type_names.size() <= kv.second) P.type_names.resize(kv.second + 1); P.type_names[kv.second] = kv.first; }
    for (size_t t = 0; t < type_recs_.size(); t++) {
      const UnitRec& u = type_recs_[t];
      UnitType ut{};
      cur_align_ = align_[P.type_names[t]];
      if (cur_align_.empty()) cur_align_.insert(0);
      ut.n_in = (uint32_t)u.in.size(); ut.n_slots = u.n_slots;
      ut.prog_off = (uint32_t)P.prog.size(); ut.prog_len = (uint32_t)u.prog.size();
      P.prog.insert(P.prog.end(), u.prog.begin(), u.prog.end());
      stat_cost_greedy_ = stat_cost_final_ = stat_cost_ideal_ = 0;
      build_chunks(u, &ut);
      for (uint32_t c = 0; c < ut.n_chunks; c++) ut.dict_len += P.chunks[ut.chunk_off + c].n_fill;
      if (getenv("H2SHA_PLAN_STATS"))   // multi-chunk types run the chunking twice (see build_chunks): their numbers are doubled
        fprintf(stderr, "[plan] %-8s chunks %2u gate %4u lk %3u limb %3u | quarter-warp scratch accesses per unit: conflict-free %.1f greedy %.1f searched %.1f\n",
                P.type_names[t].c_str(), ut.n_chunks, ut.gate_len, ut.lk_len, ut.limb_len, (double)stat_cost_ideal_ / stat_norm_,
                (double)stat_cost_greedy_ / stat_norm_, (double)stat_cost_final_ / stat_norm_);
      P.types.push_back(ut);
    }
    // ---- compact hand-off: dictionary ranges.  Per digest: its prologue / epilogue units, then its compressions ----
    {
      std::vector<uint32_t> class_len(class_recs_.size(), 0);
      for (size_t ci = 0; ci < class_recs_.size(); ci++)
        for (GroupRec& g : class_recs_[ci].groups) {
          g.dict_base = class_len[ci];
          class_len[ci] += g.count * P.types[type_idx_.at(g.type)].dict_len;
        }
      uint32_t base = 0;
      for (size_t d = 0; d < P.digests.size(); d++) {
        P.digests[d].dict_base = base;
        P.digests[d].dict_dig_len = class_len[1 + d];
        P.digests[d].dict_blk_len = class_len[0];
        base += class_len[1 + d] + P.digests[d].n_blocks * class_len[0];
      }
      P.dict_cells = base;
    }
    // ---- job classes: the block job is split into `block_parts` parts of roughly equal cell count ----
    P.max_slots = 0;
    {
      const ClassRec& c = class_recs_[0];
      uint64_t total = 0;
      for (const GroupRec& g : c.groups) total += (uint64_t)g.count * P.types[type_idx_.at(g.type)].gate_len;
      const uint32_t parts = std::max(1u, cfg_.block_parts);
      // atoms: runs of <= 32 instances of one group (one phase-1 warp task each); greedy packing into `parts` bins.  Twelve parts or
      // more ask for latency rather than throughput (one digest at a time, BASELINE config 1): the atoms shrink to 8 instances so that a
      // compression really is cut into that many jobs for that many SMs -- the slot VM's latency per task is the same at 8 lanes as at 32,
      // so this costs phase-1 throughput and is not for batches.
      struct Atom { const GroupRec* g; uint32_t first, count; uint64_t cells; };
      std::vector<Atom> atoms;
      const uint32_t atom_len = parts >= 12 ? 8u : 32u;
      for (const GroupRec& g : c.groups)
        for (uint32_t first = 0; first < g.count; first += atom_len) {
          uint32_t cnt = std::min(atom_len, g.count - first);
          atoms.push_back(Atom{&g, first, cnt, (uint64_t)cnt * P.types[type_idx_.at(g.type)].gate_len});
        }
      std::vector<std::vector<UnitGroup>> part_groups(1);
      uint64_t acc = 0;
      auto push_atom = [&](const Atom& a) {
        auto& pg = part_groups.back();
        // merge with the previous sub-group when it continues the same group
        if (!pg.empty() && pg.back().type == type_idx_.at(a.g->type) &&
            pg.back().gate_base + pg.back().count * pg.back().gate_stride == a.g->gate_base + a.first * a.g->gate_stride && a.g->gate_stride &&
            pg.back().count + a.count <= 0xfff) {
          pg.back().count += a.count;
        } else {
          pg.push_back(make_group(*a.g, a.first, a.count));
        }
      };
      for (const Atom& a : atoms) {
        const uint64_t target = total * part_groups.size() / parts;   // cumulative target at the end of the current part
        const bool can_close = part_groups.size() < parts && !part_groups.back().empty();
        const uint64_t over = acc + a.cells > target ? acc + a.cells - target : target - acc - a.cells;
        const uint64_t under = target > acc ? target - acc : acc - target;
        if (can_close && under < over) part_groups.emplace_back();
        push_atom(a);
        acc += a.cells;
      }
      while (!part_groups.empty() && part_groups.back().empty()) part_groups.pop_back();
      P.n_block_parts = (uint32_t)part_groups.size();
      for (auto& pg : part_groups) add_class(pg, (uint32_t)TR_BLOCK_WORDS_WITH_K, 1);
    }
    const uint32_t block_slots = P.max_slots;
    for (size_t ci = 1; ci < class_recs_.size(); ci++) {
      std::vector<UnitGroup> gs;
      uint32_t slots_one = 0;
      for (const GroupRec& g : class_recs_[ci].groups) {
        gs.push_back(make_group(g, 0, g.count));
        slots_one += g.count * (P.types[gs.back().type].n_slots | 1u);
      }
      // batch as many instances per digest job as fit in the stage a block job needs anyway (slots and item encoding)
      uint32_t batch = cfg_.digest_batch ? cfg_.digest_batch : H2SHA_MAX_JOB_BATCH;
      batch = std::min<uint32_t>(batch, H2SHA_MAX_JOB_BATCH);
      while (batch > 1 && (slots_one * batch > std::max(block_slots, slots_one) || slots_one * batch > 0xffff)) batch--;
      P.digests[ci - 1].job_class = (uint32_t)P.classes.size();
      // very long digests (> 64 blocks): the prologue/epilogue units need more slots than a shared-memory stage should hold;
      // cut the job into parts of whole warp tasks (<= 32 unit instances of one group), like the block job
      const uint32_t kSplitAbove = 5300, kPartSlots = 2800;
      if (slots_one <= kSplitAbove) {
        add_class(gs, P.digests[ci - 1].trace_words, batch);
        P.classes.back().digest = (uint32_t)(ci - 1);
      } else {
        const uint32_t n_parts = (slots_one + kPartSlots - 1) / kPartSlots;
        const uint32_t target = (slots_one + n_parts - 1) / n_parts;
        std::vector<UnitGroup> part;
        uint32_t part_slots = 0;
        auto flush = [&]() {
          if (part.empty()) return;
          add_class(part, P.digests[ci - 1].trace_words, 1);
          P.classes.back().digest = (uint32_t)(ci - 1);
          part.clear(); part_slots = 0;
        };
        for (const GroupRec& g : class_recs_[ci].groups) {
          const uint32_t per_unit = P.types[type_idx_.at(g.type)].n_slots | 1u;
          for (uint32_t first = 0; first < g.count; first += 32) {
            const uint32_t cnt = std::min(32u, g.count - first);
            if (part_slots && part_slots + cnt * per_unit > target) flush();
            part.push_back(make_group(g, first, cnt));
            part_slots += cnt * per_unit;
          }
        }
        flush();
      }
    }
    if (cfg_.record_compact_map) build_compact_map();
    // ---- layout ----
    auto up8 = [](uint32_t x) { return (x + 7u) & ~7u; };   // column strides are multiples of 8 cells (256 B)
    P.n_gate_cols = (uint32_t)P.breaks.size();
    uint32_t rows = 0;
    for (size_t c = 0; c < P.breaks.size(); c++) {
      uint32_t e = (c + 1 < P.breaks.size()) ? P.breaks[c + 1] : n_gate_;
      rows = std::max(rows, e - P.breaks[c]);
    }
    P.gate_col_rows = up8(rows);
    const LookupGeom G = lookup_geom(P);
    P.n_lookup_cols = G.range_cols_needed();
    P.lookup_col_rows = up8(G.max_range_used());
    P.spread_rows = up8(G.max_spread_used());
    compute_zero_ranges(P_);
  }
};

}  // namespace


void compute_zero_ranges(Plan* plan) {
  Plan& P = *plan;
  const uint32_t n_gate_ = P.n_gate;
  const LookupGeom G = lookup_geom(P);
  P.zero_ranges.clear();
  // cells of the column-major buffers nobody assigns (column tails, stride padding)
    for (size_t c = 0; c < P.breaks.size(); c++) {
      uint32_t e = (c + 1 < P.breaks.size()) ? P.breaks[c + 1] : n_gate_;
      uint32_t used = e - P.breaks[c];
      if (used < P.gate_col_rows) P.zero_ranges.push_back(ZeroRange{BUF_GATE, (uint32_t)c * P.gate_col_rows + used, P.gate_col_rows - used});
    }
    for (uint32_t c = 0; c < P.n_lookup_cols; c++) {
      uint32_t used = G.range_used(c);
      if (used < P.lookup_col_rows) P.zero_ranges.push_back(ZeroRange{BUF_LOOKUP, c * P.lookup_col_rows + used, P.lookup_col_rows - used});
    }
    for (uint32_t c = 0; c < 2 * G.spread_cols; c++) {
      uint32_t used = G.spread_used(c % G.spread_cols);
      if (used < P.spread_rows) P.zero_ranges.push_back(ZeroRange{BUF_SPREAD, c * P.spread_rows + used, P.spread_rows - used});
    }
}

bool build_plan(const Config& cfg, Plan* out, std::string* err) {
  *out = Plan();
  try {
    Builder b(cfg, out);
    b.run();
  } catch (const std::exception& e) {
    if (err) *err = e.what();
    return false;
  }
  return true;
}

}  // namespace h2sha
