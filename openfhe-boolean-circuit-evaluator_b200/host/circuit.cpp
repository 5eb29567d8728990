// circuit.cpp -- level-synchronous circuit evaluator behind the reference's Circuit API.
//
// Replaces Circuit::{ReadFile,Reset,SetInput,Clock} + _CircuitManager/_ExecuteGates
// (src/circuit.cpp:102-817 in /root/reference).  The reference's dataflow manager fires gate g in wave
// 1 + max(wave of producers), i.e. ASAP levelisation (SURVEY 3.3); here the levels are computed once,
// and each bootstrap (sub-)level is ONE batched launch of the blind-rotation and key-switch kernels
// instead of one OpenMP task per gate.  XOR is the reference's composite OR(AND(a,!b), AND(!a,b))
// (src/gate.cpp:198-202): two ANDs at level L, the OR at level L+1.  NOT costs no bootstrap and is folded
// into the consumer's operand flags; NOT outputs are only materialised where a ciphertext is needed
// (circuit outputs, verify mode).
//
// Multi-GPU: every level's gate list is block-partitioned over the ranks, keys and the wire slab are
// replicated, and the level's output rows are exchanged -- by the key-switch kernel itself, which stores every output into every rank's
// slab over NVLink (setup_peer_exchange), or with one in-place ncclAllGather where the slabs cannot be mapped (SURVEY 8(e)).
#include "../csrc/engine.hpp"
#include "netlist.hpp"
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <queue>

using namespace bfhe;

namespace {

// ---- minimal NCCL binding, resolved at run time so that CPU-only use needs no NCCL ----
struct Id128 { char b[128]; }; // ncclUniqueId is passed by value
struct NcclApi {
  void *h = nullptr;
  int (*GetUniqueId)(void *) = nullptr;
  int (*CommInitRank)(void **, int, Id128, int) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
  int (*Broadcast)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
bool load_nccl() {
  if (g_nccl.h) return true;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) { set_error(std::string("cannot load NCCL: ") + dlerror()); return false; }
  g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(h, "ncclGetUniqueId");
  g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(h, "ncclCommInitRank");
  g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(h, "ncclAllGather");
  g_nccl.Broadcast = (decltype(g_nccl.Broadcast))dlsym(h, "ncclBroadcast");
  g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(h, "ncclCommDestroy");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.Broadcast || !g_nccl.CommDestroy) {
    set_error("NCCL symbols missing");
    return false;
  }
  g_nccl.h = h;
  return true;
}
constexpr int NCCL_UINT32 = 3, NCCL_FLOAT32 = 7;

struct NotOp { uint32_t in_row, out_row, copy; }; // out = copy ? in : EvalNOT(in)
struct Level {
  std::vector<bfhe_gate> gates; // out rows are first_row + index
  uint32_t first_row = 0;
  std::vector<NotOp> nots;      // materialised after this level
  bool sharded = true;          // world > 1: block-partitioned over the ranks + exchange; false: every rank computes the whole level
};
// launch costs (ms) of one blind rotation + key switch per kernel form; measured once per context by probe_costs(), else these
// B200 defaults.  In sharded runs the ranks agree on the element-wise maximum, so that every rank builds the same schedule.
// exchange: what a sharded level pays on top of its kernels -- the key switch's peer stores, one flag round trip over NVLink and one
// tiny wait launch (~0.015 ms), or one ncclAllGather (~0.05 ms, BFHE_EXCHANGE=nccl).  The plan is made before the slabs exist, so the
// peer-store figure is assumed unless NCCL was asked for; should the mapping fail later, the plan is merely a little optimistic.
struct FormCosts {
  double cl4 = 1.05, cl2 = 1.55, lat = 2.36, thr = 5.85, exchange = exchange_default();
  bool measured = false;
  static double exchange_default() { const char *m = std::getenv("BFHE_EXCHANGE"); return m && std::strcmp(m, "nccl") == 0 ? 0.05 : 0.015; }
};
inline bool is_single(GateKind k) {
  return k == GateKind::AND || k == GateKind::OR || k == GateKind::NAND || k == GateKind::NOR || k == GateKind::XOR_FAST || k == GateKind::XNOR_FAST;
}
inline bool is_boot(GateKind k) { return is_single(k) || k == GateKind::XOR; }
inline uint32_t op_of(GateKind k) {
  switch (k) {
  case GateKind::AND: return BFHE_AND;
  case GateKind::OR: return BFHE_OR;
  case GateKind::NAND: return BFHE_NAND;
  case GateKind::NOR: return BFHE_NOR;
  case GateKind::XOR_FAST: return BFHE_XOR_FAST;
  default: return BFHE_XNOR_FAST;
  }
}

} // namespace

struct bfhe_circuit {
  bfhe_ctx *ctx = nullptr;
  Netlist nl;      // the netlist that is planned and evaluated (LUTs / XNOR lowered)
  Netlist nl_file; // as read
  bool loaded = false;
  bool plaintext = false, encrypted = false, verify = false;
  bool planned_verify = false; // the verify setting the current plan was built for
  int rank = 0, world = 1;
  void *comm = nullptr;

  // plan
  bool planned = false;
  std::vector<uint32_t> topo;        // gate indices in dependency order
  std::vector<uint32_t> wire_row;    // slab row holding the wire (possibly of its un-negated source)
  std::vector<uint8_t> wire_neg;     // wire = NOT^neg(row)
  std::vector<uint32_t> wire_level;
  std::vector<Level> levels;         // levels[0] = Bootstrap of the fresh input encryptions
  std::vector<uint32_t> level_rpr;   // rows per rank
  uint32_t total_rows = 0, fresh_base = 0, n_in = 0;
  std::vector<uint32_t> in_wire_of_bit; // concatenated input bit -> wire
  std::vector<uint32_t> out_wire;       // output bit -> wire
  uint32_t n_bootstraps = 0, max_width = 0, asap_levels = 0; // of the ASAP schedule (what the reference's manager produces)
  uint32_t wave_cap = 0;             // > 0: pack ready gates into waves of at most this many bootstraps (build_plan pass 1b)
  int wave_cap_req = -1;             // requested: -1 = one gate per SM and rank when a device is attached, 0 = ASAP levels, > 0 explicit
  int shard_min_req = -1;            // world > 1: levels narrower than this run redundantly on every rank; -1 = cost model (device) / 0
  FormCosts costs;
  // DFF state (clocked circuits): Q wires read slab rows [state_base, +n_dff); after the last level  tmp[i] = D_i,  state[i] = tmp[i]
  uint32_t n_dff = 0, state_base = 0, dff_tmp_base = 0, dff_fresh_base = 0;
  std::vector<uint32_t> dff_gate;    // netlist gate ids of the DFFs, in file order
  std::vector<NotOp> dff_ops;        // n_dff ops into tmp, then n_dff copies into the state rows
  std::vector<uint8_t> plain_state;
  bool state_init_pending = true;
  uint64_t clocks = 0;

  // device state
  uint32_t *slab = nullptr;
  DevGate *d_desc = nullptr;             // my slice of every level, concatenated
  std::vector<size_t> desc_off;          // per level
  std::vector<uint32_t> my_count;        // per level
  const u32 **d_not_in = nullptr;    // low bit of an input pointer set: plain copy instead of EvalNOT
  u32 **d_not_out = nullptr;
  std::vector<size_t> not_off;       // per level; the last two entries delimit the DFF update batches
  u32 *d_ext = nullptr;
  size_t ext_cap = 0;
  bool dev_ready = false;
  cudaGraphExec_t graph = nullptr;
  bool use_graph = true;
  // multi-GPU exchange by direct stores into the peers' slabs (PeerX, csrc/common.hpp); falls back to ncclAllGather when the slabs
  // cannot be mapped (no peer access) or BFHE_EXCHANGE=nccl
  bool peer_ok = false;
  std::vector<void *> peer_slab_map, peer_flag_map; // cudaIpcOpenMemHandle results (null for the own rank)
  u32 **d_peer_slabs = nullptr, **d_peer_flags = nullptr;
  u32 *x_flags = nullptr, *x_counter = nullptr, *x_epoch = nullptr, *x_err = nullptr; // one allocation: flags[32] | counter | epoch | err
  uint32_t x_per_epoch = 1;
  std::vector<int> shard_index; // level -> index among the sharded levels (-1: not exchanged)

  // values
  std::vector<uint8_t> in_bits_set, plain_wire;
  bool has_input = false, done = false;
  bool ct_input = false;          // the input came as ciphertexts (bfhe_circuit_set_input_ct): there are no input bits
  u32 *d_egress = nullptr;        // clock_ct into host memory: the output rows are staged here
  double device_ms = 0, host_ms = 0;
  uint64_t verify_mismatches = 0, verify_checked = 0;
};

static void free_device(bfhe_circuit *c) {
  if (c->ctx && c->ctx->device >= 0) {
    cudaSetDevice(c->ctx->device);
    cudaStreamSynchronize(c->ctx->stream);
    if (c->graph) cudaGraphExecDestroy(c->graph);
    for (void *m : c->peer_slab_map) if (m) cudaIpcCloseMemHandle(m);
    for (void *m : c->peer_flag_map) if (m) cudaIpcCloseMemHandle(m);
    cudaFree(c->d_peer_slabs); cudaFree(c->d_peer_flags); cudaFree(c->x_flags);
    cudaFree(c->slab); cudaFree(c->d_desc); cudaFree(c->d_not_in); cudaFree(c->d_not_out); cudaFree(c->d_ext);
    cudaFree(c->d_egress);
  }
  c->peer_slab_map.clear(); c->peer_flag_map.clear();
  c->d_peer_slabs = nullptr; c->d_peer_flags = nullptr; c->x_flags = c->x_counter = c->x_epoch = c->x_err = nullptr;
  c->peer_ok = false;
  c->graph = nullptr; c->slab = nullptr; c->d_desc = nullptr; c->d_not_in = nullptr; c->d_not_out = nullptr; c->d_ext = nullptr;
  c->d_egress = nullptr;
  c->dev_ready = false;
}

// ---------------------------------------------------------------------------------------------
// planning
// ---------------------------------------------------------------------------------------------
static int build_plan_cap(bfhe_circuit *c, uint32_t cap);
static bool cluster_forms_available(const bfhe_ctx *x) { return x && x->v2.d_tw2 && x->p.method == BFHE_GINX; } // 2-CTA form (GINX)
static bool clx_form_available(const bfhe_ctx *x) { return x && x->v2.d_twx; }                                   // 4-CTA form (GINX and AP)

struct FormCaps { int sms = 0, cl2 = 0, cl4 = 0; };
// cost (ms) of one wave of n bootstraps on ONE GPU: 4-CTA cluster form up to `cl4` gates, 2-CTA cluster form up to `cl2`, else the
// cheaper of one-gate-per-SM waves and four-gates-per-SM waves (key switch included in the measured figures)
static double wave_cost_ms(const FormCosts &k, const FormCaps &f, long n) {
  if (n <= 0) return 0;
  if (n <= f.cl4) return k.cl4;
  if (n <= f.cl2) return k.cl2;
  const double lat = (double)((n + f.sms - 1) / f.sms) * k.lat, thr = (double)((n + 4 * f.sms - 1) / (4 * f.sms)) * k.thr;
  return lat < thr ? lat : thr;
}
// world > 1: a level is sharded only when that is cheaper than every rank computing all of it (SURVEY 8(e): "skipping the shard
// entirely for levels narrower than a threshold"): sharding a 30-gate wave over 8 GPUs does not reach a faster kernel form, it only
// adds the exchange.  Every rank evaluates the same deterministic rule on the same (agreed) costs.
static bool level_shards(const bfhe_circuit *c, const FormCaps &f, long n) {
  if (c->world <= 1) return false;
  if (c->shard_min_req >= 0) return n >= c->shard_min_req;
  if (f.sms <= 0) return true;
  const long per = (n + c->world - 1) / c->world;
  return wave_cost_ms(c->costs, f, per) + c->costs.exchange < wave_cost_ms(c->costs, f, n);
}
static FormCaps form_caps(const bfhe_circuit *c) {
  FormCaps f;
  if (!c->ctx || c->ctx->device < 0) return f;
  if (cudaDeviceGetAttribute(&f.sms, cudaDevAttrMultiProcessorCount, c->ctx->device) != cudaSuccess || f.sms <= 0) { f.sms = 0; return f; }
  // The schedule must be the same on every rank, so the cluster-form capacities come from the SM count alone, not from this
  // device's cudaOccupancyMaxActiveClusters (which differs between GPUs of one box: 74 and 63 two-CTA clusters were both seen on
  // 148-SM B200s): 5/12 of the SMs for one gate on two SMs, 2/9 for one gate on four.  A wave that a particular GPU cannot keep
  // co-resident in the planned form simply runs in the next form there (launch_blind_rotate checks the real limit).
  f.cl2 = cluster_forms_available(c->ctx) ? f.sms * 5 / 12 : 0;
  f.cl4 = clx_form_available(c->ctx) ? f.sms * 2 / 9 : 0;
  return f;
}
static double plan_cost_ms(const bfhe_circuit *c, const FormCaps &f) {
  double t = 0;
  for (size_t L = 0; L < c->levels.size(); L++) {
    const long n = (long)c->levels[L].gates.size();
    if (n == 0) continue;
    t += c->levels[L].sharded ? wave_cost_ms(c->costs, f, c->level_rpr[L]) + c->costs.exchange : wave_cost_ms(c->costs, f, n);
  }
  return t;
}

// wave_cap_req = -1 with a device attached: try the candidate wave capacities (ASAP levels, one 4-CTA or 2-CTA cluster-form wave, one
// one-gate-per-SM wave -- each also times the number of ranks) and keep the cheapest plan under plan_cost_ms.  Depth-bound circuits
// (SHA-256, MD5) end up on the cluster form, work-bound ones (AES, multipliers) on full one-gate-per-SM waves.
static int build_plan(bfhe_circuit *c) {
  if (c->wave_cap_req >= 0 || !c->ctx || c->ctx->device < 0) return build_plan_cap(c, c->wave_cap_req > 0 ? (uint32_t)c->wave_cap_req : 0);
  const FormCaps f = form_caps(c);
  if (f.sms <= 0) return build_plan_cap(c, 0);
  std::vector<uint32_t> cands = {0u};
  for (uint32_t base : {(uint32_t)f.sms, (uint32_t)f.cl2, (uint32_t)f.cl4}) {
    if (!base) continue;
    cands.push_back(base);
    if (c->world > 1) cands.push_back(base * (uint32_t)c->world);
  }
  uint32_t best = 0;
  double best_t = 0;
  for (size_t k = 0; k < cands.size(); k++) {
    int rc = build_plan_cap(c, cands[k]);
    if (rc) return rc;
    const double t = plan_cost_ms(c, f);
    if (k == 0 || t < best_t) { best = cands[k]; best_t = t; }
  }
  return build_plan_cap(c, best);
}

static int build_plan_cap(bfhe_circuit *c, uint32_t cap) {
  const Netlist &nl = c->nl;
  c->wave_cap = cap;
  c->topo.clear();
  const uint32_t NW = nl.n_wires, NG = (uint32_t)nl.gates.size();
  const uint32_t NONE = 0xffffffffu;
  std::vector<uint32_t> producer(NW, NONE);
  c->dff_gate.clear();
  for (uint32_t i = 0; i < NG; i++) {
    const NetGate &g = nl.gates[i];
    if (g.kind == GateKind::OUTPUT) continue;
    if (g.kind == GateKind::LUT3 || g.kind == GateKind::LUT4 || g.kind == GateKind::XNOR) { set_error("internal: netlist not lowered"); return BFHE_ERR_STATE; }
    if (g.out >= NW) { set_error("wire id out of range"); return BFHE_ERR_FORMAT; }
    if (producer[g.out] != NONE) { set_error("wire driven twice"); return BFHE_ERR_FORMAT; }
    producer[g.out] = i;
    if (g.kind == GateKind::DFF) c->dff_gate.push_back(i);
  }
  c->n_dff = (uint32_t)c->dff_gate.size();
  // dependency order (the reference needs none: its manager is dataflow-driven; files are ordered anyway).  A DFF's Q output is a
  // source like an input (it holds the state of the previous clock); its D input is a sink like an output.
  c->topo.reserve(NG);
  {
    std::vector<uint8_t> state(NG, 0);
    std::vector<uint32_t> stack;
    auto deps = [&](const NetGate &g, uint32_t d[2]) -> int {
      switch (g.kind) {
      case GateKind::INPUT: case GateKind::DFF: return 0;
      case GateKind::OUTPUT: case GateKind::NOT: d[0] = g.in0; return 1;
      default: d[0] = g.in0; d[1] = g.in1; return 2;
      }
    };
    for (uint32_t s = 0; s < NG; s++) {
      if (state[s]) continue;
      stack.push_back(s);
      while (!stack.empty()) {
        uint32_t gi = stack.back();
        if (state[gi] == 2) { stack.pop_back(); continue; }
        uint32_t d[2];
        int nd = deps(nl.gates[gi], d);
        bool ready = true;
        for (int k = 0; k < nd; k++) {
          if (d[k] >= NW || producer[d[k]] == NONE) { set_error("gate reads an undriven wire"); return BFHE_ERR_FORMAT; }
          uint32_t p = producer[d[k]];
          if (state[p] == 1) { set_error("combinational loop in netlist"); return BFHE_ERR_FORMAT; }
          if (state[p] == 0) { ready = false; stack.push_back(p); }
        }
        if (!ready) { state[gi] = 1; continue; }
        state[gi] = 2;
        c->topo.push_back(gi);
        stack.pop_back();
      }
    }
  }
  for (uint32_t gi : c->dff_gate)
    if (nl.gates[gi].in0 >= NW || producer[nl.gates[gi].in0] == NONE) { set_error("DFF reads an undriven wire"); return BFHE_ERR_FORMAT; }
  // which wires need a ciphertext of their own even though they are a NOT of something
  std::vector<uint8_t> feeds_output(NW, 0);
  for (const NetGate &g : nl.gates)
    if (g.kind == GateKind::OUTPUT) feeds_output[g.in0] = 1;

  c->n_in = 0;
  for (auto b : nl.in_bits) c->n_in += b;
  std::vector<uint32_t> bus_base(nl.in_bits.size() + 1, 0);
  for (size_t b = 0; b < nl.in_bits.size(); b++) bus_base[b + 1] = bus_base[b] + nl.in_bits[b];
  c->in_wire_of_bit.assign(c->n_in, NONE);
  c->out_wire.assign(nl.out_bits, NONE);
  c->wire_row.assign(NW, NONE);
  c->wire_neg.assign(NW, 0);
  c->wire_level.assign(NW, 0);

  // pass 1a: ASAP levels (the wave structure of the reference's manager, SURVEY 3.3): level of a gate = 1 + max(level of its
  // producers); NOT costs nothing; XOR = two ANDs at L and the OR at L + 1.
  std::vector<uint32_t> lvl1(NG, NONE), lvl2(NG, NONE); // bootstrap level of a gate's (first) bootstrap / of XOR's closing OR
  for (uint32_t gi : c->topo) {
    const NetGate &g = nl.gates[gi];
    if (g.kind == GateKind::INPUT || g.kind == GateKind::DFF) c->wire_level[g.out] = 0;
    else if (g.kind == GateKind::NOT) c->wire_level[g.out] = c->wire_level[g.in0];
    else if (is_boot(g.kind)) {
      lvl1[gi] = 1 + std::max(c->wire_level[g.in0], c->wire_level[g.in1]);
      if (g.kind == GateKind::XOR) lvl2[gi] = lvl1[gi] + 1;
      c->wire_level[g.out] = g.kind == GateKind::XOR ? lvl2[gi] : lvl1[gi];
    }
  }
  { // the reference-shaped statistics (SURVEY App. A) always describe the ASAP schedule
    std::vector<uint32_t> width(1, 0);
    c->n_bootstraps = 0;
    for (uint32_t gi = 0; gi < NG; gi++) {
      if (lvl1[gi] == NONE) continue;
      const bool x = nl.gates[gi].kind == GateKind::XOR;
      if (width.size() <= lvl1[gi] + (x ? 1u : 0u)) width.resize(lvl1[gi] + (x ? 2 : 1), 0);
      width[lvl1[gi]] += x ? 2 : 1;
      if (x) width[lvl2[gi]] += 1;
      c->n_bootstraps += x ? 3 : 1;
    }
    c->asap_levels = (uint32_t)width.size() - 1;
    c->max_width = 0;
    for (size_t L = 1; L < width.size(); L++) c->max_width = std::max(c->max_width, width[L]);
  }
  // pass 1b (wave_cap > 0): list scheduling into waves of at most wave_cap bootstraps.  An ASAP level of 196 gates costs
  // two launches of the one-gate-per-SM kernel on 148 SMs although the second is a third full; packing ready gates by
  // longest remaining path fills the waves (AES-128: 420 ASAP levels, 82 172 bootstraps -> ~560 full waves instead of ~790
  // launches' worth).  Gate outputs do not depend on the schedule, so ciphertexts stay bit-identical.
  if (c->wave_cap > 0) {
    // units: U1 = the gate's first bootstrap(s) (weight 2 for XOR's AND pair), U2 = XOR's OR.  unit id = 2*gi (+1)
    std::vector<uint32_t> wire_unit(NW, NONE);
    std::vector<uint32_t> indeg(2 * (size_t)NG, 0), height(2 * (size_t)NG, 0);
    std::vector<std::vector<uint32_t>> succ(2 * (size_t)NG);
    for (uint32_t gi : c->topo) {
      const NetGate &g = nl.gates[gi];
      if (g.kind == GateKind::NOT) { wire_unit[g.out] = wire_unit[g.in0]; continue; }
      if (lvl1[gi] == NONE) continue;
      const uint32_t u1 = 2 * gi, u2 = 2 * gi + 1;
      const uint32_t pa = wire_unit[g.in0], pb = wire_unit[g.in1];
      if (pa != NONE) { succ[pa].push_back(u1); indeg[u1]++; }
      if (pb != NONE && pb != pa) { succ[pb].push_back(u1); indeg[u1]++; }
      if (g.kind == GateKind::XOR) { succ[u1].push_back(u2); indeg[u2]++; wire_unit[g.out] = u2; }
      else wire_unit[g.out] = u1;
    }
    for (size_t k = c->topo.size(); k-- > 0;) { // longest path to a sink, in waves
      const uint32_t gi = c->topo[k];
      if (lvl1[gi] == NONE) continue;
      for (uint32_t u : {2 * gi + 1, 2 * gi}) {
        if (u == 2 * gi + 1 && nl.gates[gi].kind != GateKind::XOR) continue;
        uint32_t h = 0;
        for (uint32_t v : succ[u]) h = std::max(h, height[v]);
        height[u] = h + 1;
      }
    }
    auto weight = [&](uint32_t u) { return (u & 1) == 0 && nl.gates[u >> 1].kind == GateKind::XOR ? 2u : 1u; };
    auto worse = [&](uint32_t a, uint32_t b) { return height[a] != height[b] ? height[a] < height[b] : a > b; };
    std::priority_queue<uint32_t, std::vector<uint32_t>, decltype(worse)> ready(worse);
    uint64_t ready_weight = 0;
    for (uint32_t gi : c->topo) {
      if (lvl1[gi] == NONE) continue;
      if (indeg[2 * gi] == 0) { ready.push(2 * gi); ready_weight += weight(2 * gi); }
    }
    std::vector<uint32_t> wave_of(2 * (size_t)NG, NONE), next, held;
    // a wave must be able to hold the heaviest unit (XOR's AND pair, weight 2): with a smaller capacity nothing could ever be scheduled
    const uint32_t cap1 = std::max(c->wave_cap, 2u), cap4 = 4 * cap1; // one-gate-per-SM wave / four-gates-per-SM wave
    for (uint32_t W = 1; !ready.empty(); W++) {
      // plenty of independent work (at least two 4-gates-per-SM waves): use whole throughput-kernel waves, else one latency wave
      uint32_t cap = ready_weight >= 2 * (uint64_t)cap4 ? (uint32_t)(ready_weight / cap4) * cap4 : cap1;
      uint32_t used = 0;
      next.clear(); held.clear();
      while (!ready.empty() && used < cap) {
        const uint32_t u = ready.top();
        ready.pop();
        const uint32_t wt = weight(u);
        if (used + wt > cap) { held.push_back(u); if (held.size() > 8) break; continue; }
        used += wt;
        ready_weight -= wt;
        wave_of[u] = W;
        for (uint32_t v : succ[u]) if (--indeg[v] == 0) next.push_back(v);
      }
      for (uint32_t u : held) ready.push(u);
      for (uint32_t v : next) { ready.push(v); ready_weight += weight(v); }
    }
    for (uint32_t gi : c->topo) {
      const NetGate &g = nl.gates[gi];
      if (g.kind == GateKind::INPUT || g.kind == GateKind::DFF) c->wire_level[g.out] = 0;
      else if (g.kind == GateKind::NOT) c->wire_level[g.out] = c->wire_level[g.in0];
      else if (is_boot(g.kind)) {
        lvl1[gi] = wave_of[2 * gi];
        if (g.kind == GateKind::XOR) lvl2[gi] = wave_of[2 * gi + 1];
        c->wire_level[g.out] = g.kind == GateKind::XOR ? lvl2[gi] : lvl1[gi];
      }
    }
  }

  // pass 1c: placement.  Rows are assigned afterwards, so gates carry (level, index) first.
  std::vector<std::vector<uint32_t>> lvl_gates(1); // netlist gate ids per bootstrap level (XOR appears at its two levels)
  struct Slot { uint32_t level, index; };
  std::vector<Slot> wire_slot(NW, Slot{NONE, NONE}); // for bootstrapped wires
  std::vector<Slot> xor_t1(NG, Slot{NONE, NONE});
  auto ensure_level = [&](uint32_t L) { if (lvl_gates.size() <= L) lvl_gates.resize(L + 1); };
  // A NOT is free (an operand flag of its consumers).  A wire that needs a ciphertext of its own -- circuit outputs, and in verify mode
  // every wire -- is materialised from its BASE: the bootstrapped (or input / state) row it is a NOT^k of.  NOT^even aliases the base
  // row, NOT^odd becomes ONE EvalNOT of the base row after the base's level, so no materialised NOT ever reads another one (a chain
  // NOT(NOT(x)) inside one batched launch would race, and Bristol's EQW is lowered to exactly that pair).
  std::vector<uint32_t> base_wire(NW, NONE);
  std::vector<uint8_t> base_neg(NW, 0);
  std::vector<std::vector<uint32_t>> lvl_nots(1); // wires materialised after each level
  std::vector<uint32_t> mat_of_base(NW, NONE);    // base wire -> the wire already materialising NOT(base)
  uint32_t dff_idx = 0;
  std::vector<uint32_t> dff_index_of_gate(NG, NONE);
  for (uint32_t gi : c->dff_gate) dff_index_of_gate[gi] = dff_idx++;
  for (uint32_t gi : c->topo) {
    const NetGate &g = nl.gates[gi];
    if (g.kind == GateKind::INPUT) {
      if (g.in0 >= nl.in_bits.size() || g.in1 >= nl.in_bits[g.in0]) { set_error("LOAD out of range"); return BFHE_ERR_FORMAT; }
      uint32_t bit = bus_base[g.in0] + g.in1;
      if (c->in_wire_of_bit[bit] != NONE) { set_error("input bit loaded twice"); return BFHE_ERR_FORMAT; }
      c->in_wire_of_bit[bit] = g.out;
      wire_slot[g.out] = Slot{0, bit};
      base_wire[g.out] = g.out;
    } else if (g.kind == GateKind::DFF) {
      base_wire[g.out] = g.out; // row assigned below (state block)
    } else if (g.kind == GateKind::NOT) {
      base_wire[g.out] = base_wire[g.in0];
      base_neg[g.out] = base_neg[g.in0] ^ 1;
      if ((c->verify || feeds_output[g.out]) && base_neg[g.out] && mat_of_base[base_wire[g.out]] == NONE) {
        const uint32_t L = c->wire_level[g.in0];
        if (lvl_nots.size() <= L) lvl_nots.resize(L + 1);
        lvl_nots[L].push_back(g.out);
        mat_of_base[base_wire[g.out]] = g.out;
      }
    } else if (is_boot(g.kind)) {
      const uint32_t L = lvl1[gi];
      ensure_level(g.kind == GateKind::XOR ? lvl2[gi] : L);
      if (g.kind == GateKind::XOR) {
        xor_t1[gi] = Slot{L, (uint32_t)lvl_gates[L].size()};
        lvl_gates[L].push_back(gi);      // AND(a,!b)
        lvl_gates[L].push_back(gi);      // AND(!a,b)
        wire_slot[g.out] = Slot{lvl2[gi], (uint32_t)lvl_gates[lvl2[gi]].size()};
        lvl_gates[lvl2[gi]].push_back(gi);  // OR
      } else {
        wire_slot[g.out] = Slot{L, (uint32_t)lvl_gates[L].size()};
        lvl_gates[L].push_back(gi);
      }
      base_wire[g.out] = g.out;
    } else if (g.kind == GateKind::OUTPUT) {
      if (g.out >= nl.out_bits) { set_error("STORE out of range"); return BFHE_ERR_FORMAT; }
      c->out_wire[g.out] = g.in0;
    }
  }
  for (uint32_t b = 0; b < c->n_in; b++)
    if (c->in_wire_of_bit[b] == NONE) { set_error("input bit " + std::to_string(b) + " is never loaded"); return BFHE_ERR_FORMAT; }
  for (uint32_t b = 0; b < nl.out_bits; b++)
    if (c->out_wire[b] == NONE) { set_error("output bit " + std::to_string(b) + " is never stored"); return BFHE_ERR_FORMAT; }

  // pass 2: rows.  level block = [bootstrap outputs, padded to world * rows_per_rank][materialised NOTs]
  if (lvl_nots.size() < lvl_gates.size()) lvl_nots.resize(lvl_gates.size());
  if (lvl_gates.size() < lvl_nots.size()) lvl_gates.resize(lvl_nots.size());
  const uint32_t NL = (uint32_t)lvl_gates.size();
  const FormCaps fcaps = form_caps(c);
  c->levels.assign(NL, Level());
  c->level_rpr.assign(NL, 0);
  std::vector<uint32_t> first(NL, 0);
  uint32_t row = 0;
  std::vector<std::vector<uint32_t>> not_rows(NL);
  for (uint32_t L = 0; L < NL; L++) {
    const uint32_t cnt = (L == 0) ? c->n_in : (uint32_t)lvl_gates[L].size();
    const uint32_t rpr = (cnt + c->world - 1) / c->world;
    first[L] = row;
    c->level_rpr[L] = rpr;
    c->levels[L].sharded = level_shards(c, fcaps, cnt);
    row += rpr * c->world;
    not_rows[L].resize(lvl_nots[L].size());
    for (auto &r : not_rows[L]) r = row++;
  }
  c->state_base = row;      row += c->n_dff;
  c->dff_tmp_base = row;    row += c->n_dff;
  c->fresh_base = row;      row += c->n_in;
  c->dff_fresh_base = row;  row += c->n_dff;
  c->total_rows = row;
  // base rows, then wire -> (row, neg) in dependency order
  std::vector<uint32_t> base_row(NW, NONE);
  for (uint32_t gi : c->topo) {
    const NetGate &g = nl.gates[gi];
    if (g.kind == GateKind::INPUT || is_boot(g.kind)) base_row[g.out] = first[wire_slot[g.out].level] + wire_slot[g.out].index;
    else if (g.kind == GateKind::DFF) base_row[g.out] = c->state_base + dff_index_of_gate[gi];
  }
  std::vector<uint32_t> mat_row(NW, NONE); // base wire -> row holding NOT(base)
  for (uint32_t L = 0; L < NL; L++)
    for (size_t k = 0; k < lvl_nots[L].size(); k++) mat_row[base_wire[lvl_nots[L][k]]] = not_rows[L][k];
  for (uint32_t gi : c->topo) {
    const NetGate &g = nl.gates[gi];
    if (g.kind == GateKind::OUTPUT) continue;
    const uint32_t b = base_wire[g.out];
    if (g.kind == GateKind::NOT && base_neg[g.out] && mat_row[b] != NONE && (c->verify || feeds_output[g.out])) {
      c->wire_row[g.out] = mat_row[b]; // owns (or shares) the materialised NOT(base)
      c->wire_neg[g.out] = 0;
    } else {
      c->wire_row[g.out] = base_row[b];
      c->wire_neg[g.out] = base_neg[g.out];
    }
  }
  // gate descriptors
  for (uint32_t L = 0; L < NL; L++) {
    Level &lv = c->levels[L];
    lv.first_row = first[L];
    if (L == 0) {
      for (uint32_t b = 0; b < c->n_in; b++) lv.gates.push_back(bfhe_gate{BFHE_BOOTSTRAP, c->fresh_base + b, c->fresh_base + b, b});
    } else {
      for (uint32_t idx = 0; idx < lvl_gates[L].size(); idx++) {
        const uint32_t gi = lvl_gates[L][idx];
        const NetGate &g = nl.gates[gi];
        const uint32_t out = first[L] + idx;
        const uint32_t ra = c->wire_row[g.in0], rb = c->wire_row[g.in1];
        const uint32_t fa = c->wire_neg[g.in0] ? BFHE_NEG0 : 0, fb = c->wire_neg[g.in1] ? BFHE_NEG1 : 0;
        if (g.kind == GateKind::XOR) {
          const Slot t1 = xor_t1[gi];
          if (t1.level == L && idx - t1.index < 2) { // the two ANDs
            if (idx == t1.index) lv.gates.push_back(bfhe_gate{BFHE_AND | fa | (fb ^ BFHE_NEG1), ra, rb, out});
            else lv.gates.push_back(bfhe_gate{BFHE_AND | (fa ^ BFHE_NEG0) | fb, ra, rb, out});
          } else {
            lv.gates.push_back(bfhe_gate{BFHE_OR, first[t1.level] + t1.index, first[t1.level] + t1.index + 1, out});
          }
        } else {
          lv.gates.push_back(bfhe_gate{op_of(g.kind) | fa | fb, ra, rb, out});
        }
        const bfhe_gate &d = lv.gates.back();
        if (d.in0 == d.in1 && (((d.op & BFHE_NEG0) != 0) == ((d.op & BFHE_NEG1) != 0))) {
          // OpenFHE throws for EvalBinGate(ct, ct); the reference's catch re-encrypts both inputs with the
          // secret key (src/gate.cpp:134-152).  A server-side evaluator has no secret key: reject at load.
          set_error("gate with both inputs on the same wire (EvalBinGate requires independent ciphertexts)");
          return BFHE_ERR_ALIAS;
        }
      }
    }
    for (size_t k = 0; k < lvl_nots[L].size(); k++) lv.nots.push_back(NotOp{base_row[base_wire[lvl_nots[L][k]]], not_rows[L][k], 0});
  }
  // DFF: after the last level  scratch[i] = D_i (copy or EvalNOT of the row D reads);  at the start of the next clock  state[i] = scratch[i].
  c->dff_ops.clear();
  for (uint32_t i = 0; i < c->n_dff; i++) {
    const uint32_t d = nl.gates[c->dff_gate[i]].in0;
    c->dff_ops.push_back(NotOp{c->wire_row[d], c->dff_tmp_base + i, c->wire_neg[d] ? 0u : 1u});
  }
  for (uint32_t i = 0; i < c->n_dff; i++) c->dff_ops.push_back(NotOp{c->dff_tmp_base + i, c->state_base + i, 1u});
  c->planned = true;
  return BFHE_OK;
}

// ---------------------------------------------------------------------------------------------
// device plan
// ---------------------------------------------------------------------------------------------
static void my_slice(const bfhe_circuit *c, uint32_t L, int rank, uint32_t *begin, uint32_t *count) {
  const uint32_t cnt = (uint32_t)c->levels[L].gates.size(), rpr = c->level_rpr[L];
  if (!c->levels[L].sharded) { *begin = 0; *count = cnt; return; } // every rank computes the whole level, no exchange
  const uint32_t b = std::min(cnt, rpr * (uint32_t)rank), e = std::min(cnt, rpr * (uint32_t)(rank + 1));
  *begin = b;
  *count = e - b;
}

// Start-up probe: the cost of one wave (blind rotation + key switch) in each kernel form on THIS device with THIS key set, measured
// once per context on a scratch slab of random ciphertext rows.  Replaces hard-coded launch costs in the wave-packing cost model.
static int probe_costs(bfhe_circuit *c) {
  bfhe_ctx *x = c->ctx;
  if (!x->form_cost_measured) {
    const FormCaps f = form_caps(c);
    const size_t st = x->p.ct_stride, N = x->p.N;
    const int nmax = 4 * f.sms;
    u32 *slab = nullptr, *ext = nullptr;
    DevGate *dg = nullptr;
    BFHE_CUDA(cudaMalloc(&slab, (size_t)(2 + nmax) * st * 4));
    BFHE_CUDA(cudaMalloc(&ext, (size_t)nmax * (N + 4) * 4));
    BFHE_CUDA(cudaMalloc(&dg, (size_t)nmax * sizeof(DevGate)));
    std::vector<u32> rows(2 * st);
    u64 lcg = 0x9E3779B97F4A7C15ull; // any fixed non-trivial rows: the kernels' work does not depend on the values (zeros would let the
    for (auto &v : rows) { lcg = lcg * 6364136223846793005ull + 1442695040888963407ull; v = (u32)(lcg >> 40) % x->p.q; } // latency form skip steps)
    std::vector<DevGate> hg(nmax);
    for (int i = 0; i < nmax; i++) hg[i] = DevGate{slab, slab + st, slab + (size_t)(2 + i) * st, BFHE_NAND, 0};
    BFHE_CUDA(cudaMemcpy(slab, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice));
    BFHE_CUDA(cudaMemcpy(dg, hg.data(), hg.size() * sizeof(DevGate), cudaMemcpyHostToDevice));
    cudaEvent_t e0, e1;
    BFHE_CUDA(cudaEventCreate(&e0));
    BFHE_CUDA(cudaEventCreate(&e1));
    const int force[4] = {128, 32, 8, 4};
    const int count[4] = {std::min(f.cl4, clx_fast_gates()), std::min(f.cl2, cl2_max_gates()), f.sms, 4 * f.sms};
    const double dflt[4] = {FormCosts().cl4, FormCosts().cl2, FormCosts().lat, FormCosts().thr};
    for (int k = 0; k < 4; k++) {
      x->form_cost_ms[k] = dflt[k];
      if (count[k] <= 0 || (k == 0 && !clx_form_available(x)) || (k == 1 && !cluster_forms_available(x))) continue;
      float best = 0;
      for (int rep = 0; rep < 3; rep++) { // first repetition warms the key into L2
        BFHE_CUDA(cudaEventRecord(e0, x->stream));
        int rc = launch_blind_rotate(x->P, x->p.method == BFHE_AP, dg, count[k], x->d_bk, x->d_twl, x->d_psiM, ext, nullptr, force[k], x->stream, nullptr, &x->v2);
        if (rc) return cuda_fail((cudaError_t)rc, "probe: blind_rotate launch");
        rc = launch_keyswitch(x->P, ext, dg, count[k], x->d_ksk, x->ksk_elem_bytes, x->stream);
        if (rc) return cuda_fail((cudaError_t)rc, "probe: keyswitch launch");
        BFHE_CUDA(cudaEventRecord(e1, x->stream));
        BFHE_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep == 1 || (rep == 2 && ms < best)) best = ms;
      }
      x->form_cost_ms[k] = best;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(slab); cudaFree(ext); cudaFree(dg);
    x->form_cost_measured = true;
  }
  float v[4] = {(float)x->form_cost_ms[0], (float)x->form_cost_ms[1], (float)x->form_cost_ms[2], (float)x->form_cost_ms[3]};
  if (c->world > 1 && c->comm) { // every rank must plan with the same numbers: element-wise maximum over the ranks
    float *d = nullptr;
    BFHE_CUDA(cudaMalloc(&d, (size_t)c->world * 4 * sizeof(float)));
    BFHE_CUDA(cudaMemcpyAsync(d + 4 * c->rank, v, sizeof v, cudaMemcpyHostToDevice, x->stream));
    int nrc = g_nccl.AllGather(d + 4 * c->rank, d, 4, NCCL_FLOAT32, c->comm, x->stream);
    if (nrc) { cudaFree(d); set_error("ncclAllGather (probe) failed"); return BFHE_ERR_NCCL; }
    std::vector<float> all((size_t)c->world * 4);
    BFHE_CUDA(cudaMemcpyAsync(all.data(), d, all.size() * sizeof(float), cudaMemcpyDeviceToHost, x->stream));
    BFHE_CUDA(cudaStreamSynchronize(x->stream));
    cudaFree(d);
    for (int r = 0; r < c->world; r++)
      for (int k = 0; k < 4; k++) v[k] = std::max(v[k], all[(size_t)r * 4 + k]);
  }
  c->costs.cl4 = v[0]; c->costs.cl2 = v[1]; c->costs.lat = v[2]; c->costs.thr = v[3];
  c->costs.measured = true;
  return BFHE_OK;
}

// Map every peer's wire slab and flag array into this process (CUDA IPC) so that the key switch can store its outputs into all slabs
// directly.  The 64-byte handles travel through one ncclAllGather, which is also the barrier that orders "flags initialised" before
// "anybody signals".  Every rank takes the same decision (the allgathered record carries an ok byte): peer stores or ncclAllGather.
static int setup_peer_exchange(bfhe_circuit *c) {
  bfhe_ctx *x = c->ctx;
  const int W = c->world;
  c->shard_index.assign(c->levels.size(), -1);
  uint32_t S = 0;
  for (size_t L = 0; L < c->levels.size(); L++)
    if (c->level_rpr[L] && c->levels[L].sharded) c->shard_index[L] = (int)S++;
  c->x_per_epoch = S + 1;
  if (W <= 1 || W > 32 || !c->comm) return BFHE_OK;
  const char *mode = std::getenv("BFHE_EXCHANGE");
  struct Rec { cudaIpcMemHandle_t slab, flags; uint32_t ok; uint32_t pad[3]; };
  static_assert(sizeof(Rec) % 16 == 0, "record size");
  Rec mine{};
  BFHE_CUDA(cudaMalloc(&c->x_flags, 64 * sizeof(u32)));
  c->x_counter = c->x_flags + 32; c->x_epoch = c->x_flags + 33; c->x_err = c->x_flags + 34;
  {
    std::vector<u32> init(64, 0);
    for (int r = 0; r < 32; r++) init[r] = c->x_per_epoch; // = value(epoch 0, end-of-Clock): the first Clock's opening wait passes
    BFHE_CUDA(cudaMemcpy(c->x_flags, init.data(), init.size() * sizeof(u32), cudaMemcpyHostToDevice));
  }
  mine.ok = !(mode && std::strcmp(mode, "nccl") == 0) && cudaIpcGetMemHandle(&mine.slab, c->slab) == cudaSuccess &&
            cudaIpcGetMemHandle(&mine.flags, c->x_flags) == cudaSuccess;
  cudaGetLastError();
  Rec *d = nullptr;
  BFHE_CUDA(cudaMalloc(&d, (size_t)W * sizeof(Rec)));
  BFHE_CUDA(cudaMemcpyAsync(d + c->rank, &mine, sizeof(Rec), cudaMemcpyHostToDevice, x->stream));
  int nrc = g_nccl.AllGather(d + c->rank, d, sizeof(Rec) / 4, NCCL_UINT32, c->comm, x->stream);
  if (nrc) { cudaFree(d); set_error("ncclAllGather (IPC handles) failed"); return BFHE_ERR_NCCL; }
  std::vector<Rec> all(W);
  BFHE_CUDA(cudaMemcpyAsync(all.data(), d, (size_t)W * sizeof(Rec), cudaMemcpyDeviceToHost, x->stream));
  BFHE_CUDA(cudaStreamSynchronize(x->stream));
  bool ok = true;
  for (int r = 0; r < W; r++) ok = ok && all[r].ok;
  std::vector<u32 *> slabs(W, nullptr), flags(W, nullptr);
  c->peer_slab_map.assign(W, nullptr); c->peer_flag_map.assign(W, nullptr);
  uint32_t opened = ok ? 1 : 0;
  for (int r = 0; r < W && opened; r++) {
    if (r == c->rank) { slabs[r] = c->slab; flags[r] = c->x_flags; continue; }
    if (cudaIpcOpenMemHandle(&c->peer_slab_map[r], all[r].slab, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
        cudaIpcOpenMemHandle(&c->peer_flag_map[r], all[r].flags, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); opened = 0; break; }
    slabs[r] = (u32 *)c->peer_slab_map[r]; flags[r] = (u32 *)c->peer_flag_map[r];
  }
  // second round: did EVERY rank manage to open every mapping?  (also the barrier after which signalling may start)
  uint32_t *dflag = reinterpret_cast<uint32_t *>(d);
  BFHE_CUDA(cudaMemcpyAsync(dflag + c->rank, &opened, sizeof(uint32_t), cudaMemcpyHostToDevice, x->stream));
  nrc = g_nccl.AllGather(dflag + c->rank, dflag, 1, NCCL_UINT32, c->comm, x->stream);
  if (nrc) { cudaFree(d); set_error("ncclAllGather (IPC status) failed"); return BFHE_ERR_NCCL; }
  std::vector<uint32_t> st(W);
  BFHE_CUDA(cudaMemcpyAsync(st.data(), dflag, (size_t)W * sizeof(uint32_t), cudaMemcpyDeviceToHost, x->stream));
  BFHE_CUDA(cudaStreamSynchronize(x->stream));
  cudaFree(d);
  for (int r = 0; r < W; r++) ok = ok && st[r];
  if (!ok) return BFHE_OK; // ncclAllGather path
  BFHE_CUDA(cudaMalloc(&c->d_peer_slabs, (size_t)W * sizeof(u32 *)));
  BFHE_CUDA(cudaMalloc(&c->d_peer_flags, (size_t)W * sizeof(u32 *)));
  BFHE_CUDA(cudaMemcpy(c->d_peer_slabs, slabs.data(), (size_t)W * sizeof(u32 *), cudaMemcpyHostToDevice));
  BFHE_CUDA(cudaMemcpy(c->d_peer_flags, flags.data(), (size_t)W * sizeof(u32 *), cudaMemcpyHostToDevice));
  c->peer_ok = true;
  return BFHE_OK;
}
static PeerX peer_x(const bfhe_circuit *c, uint32_t index) {
  PeerX px;
  px.slabs = c->d_peer_slabs; px.local_base = c->slab; px.flags = c->d_peer_flags; px.counter = c->x_counter; px.epoch = c->x_epoch;
  px.world = (u32)c->world; px.rank = (u32)c->rank; px.index = index; px.per_epoch = c->x_per_epoch;
  return px;
}

static int upload_plan(bfhe_circuit *c) {
  bfhe_ctx *x = c->ctx;
  if (x->device < 0) { set_error("no CUDA device attached (this engine has no CPU fallback)"); return BFHE_ERR_CUDA; }
  if (c->world > 1 && !c->comm) { set_error("sharded evaluation needs an NCCL communicator: pass the unique id to bfhe_circuit_set_sharding"); return BFHE_ERR_STATE; }
  BFHE_CUDA(cudaSetDevice(x->device));
  int rc = ensure_device_keys(x);
  if (rc) return rc;
  rc = blind_rotate_set_attrs(); // function attributes must not be set under stream capture
  if (rc) return cuda_fail((cudaError_t)rc, "cudaFuncSetAttribute");
  free_device(c);
  if (c->wave_cap_req < 0 && !c->costs.measured) { // cost model: measure the launch forms once, then plan with the measured numbers
    rc = probe_costs(c);
    if (rc) return rc;
    rc = build_plan(c);
    if (rc) return rc;
  }
  const size_t st = x->p.ct_stride;
  // one row past the plan holds the status word of a ciphertext SetInput, next to the fresh rows so that one broadcast carries both
  BFHE_CUDA(cudaMalloc(&c->slab, (size_t)(c->total_rows + 1) * st * 4));
  BFHE_CUDA(cudaMemset(c->slab, 0, (size_t)(c->total_rows + 1) * st * 4));
  std::vector<DevGate> desc;
  std::vector<const u32 *> nin;
  std::vector<u32 *> nout;
  c->desc_off.clear(); c->my_count.clear(); c->not_off.clear();
  auto push_not = [&](const NotOp &o) { // the copy flag travels in the low bit of the (16-byte aligned) input pointer
    nin.push_back(reinterpret_cast<const u32 *>(reinterpret_cast<uintptr_t>(c->slab + (size_t)o.in_row * st) | (o.copy ? 1u : 0u)));
    nout.push_back(c->slab + (size_t)o.out_row * st);
  };
  uint32_t widest = std::max(1u, c->n_dff);
  for (uint32_t L = 0; L < c->levels.size(); L++) {
    uint32_t b, n;
    my_slice(c, L, c->rank, &b, &n);
    c->desc_off.push_back(desc.size());
    c->my_count.push_back(n);
    widest = std::max(widest, n);
    for (uint32_t i = b; i < b + n; i++) {
      const bfhe_gate &g = c->levels[L].gates[i];
      desc.push_back(DevGate{c->slab + (size_t)g.in0 * st, c->slab + (size_t)g.in1 * st, c->slab + (size_t)g.out * st, g.op, 0});
    }
    c->not_off.push_back(nin.size());
    for (const NotOp &o : c->levels[L].nots) push_not(o);
  }
  c->not_off.push_back(nin.size());
  for (uint32_t i = 0; i < c->n_dff; i++) push_not(c->dff_ops[i]);           // batch 1: tmp[i] = D_i
  c->not_off.push_back(nin.size());
  for (uint32_t i = 0; i < c->n_dff; i++) push_not(c->dff_ops[c->n_dff + i]); // batch 2: state[i] = tmp[i]
  c->not_off.push_back(nin.size());
  BFHE_CUDA(cudaMalloc(&c->d_desc, std::max<size_t>(desc.size(), 1) * sizeof(DevGate)));
  BFHE_CUDA(cudaMemcpy(c->d_desc, desc.data(), desc.size() * sizeof(DevGate), cudaMemcpyHostToDevice));
  BFHE_CUDA(cudaMalloc(&c->d_not_in, std::max<size_t>(nin.size(), 1) * sizeof(void *)));
  BFHE_CUDA(cudaMalloc(&c->d_not_out, std::max<size_t>(nin.size(), 1) * sizeof(void *)));
  BFHE_CUDA(cudaMemcpy(c->d_not_in, nin.data(), nin.size() * sizeof(void *), cudaMemcpyHostToDevice));
  BFHE_CUDA(cudaMemcpy(c->d_not_out, nout.data(), nout.size() * sizeof(void *), cudaMemcpyHostToDevice));
  c->ext_cap = widest;
  BFHE_CUDA(cudaMalloc(&c->d_ext, (size_t)widest * (x->p.N + 4) * 4));
  rc = setup_peer_exchange(c);
  if (rc) return rc;
  c->dev_ready = true;
  return BFHE_OK;
}

// enqueue every level on the stream (directly, or under stream capture)
static int enqueue_levels(bfhe_circuit *c) {
  bfhe_ctx *x = c->ctx;
  const size_t st = x->p.ct_stride;
  const size_t NLv = c->levels.size();
  const bool px_on = c->world > 1 && c->peer_ok;
  if (px_on) { // new epoch; nobody stores into a peer's slab before that peer has finished its previous Clock (its end-of-Clock signal)
    int rc = launch_peer_epoch_bump(c->x_epoch, x->stream);
    if (!rc) rc = launch_peer_wait(c->x_flags, c->x_epoch, (u32)c->world, (u32)c->rank, -1, c->x_per_epoch, c->x_err, x->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "peer exchange launch");
  }
  if (c->n_dff) { // clocked circuits: the state rows take the values latched at the end of the previous clock (or the power-up values)
    int rc = launch_eval_not(x->P, c->d_not_in + c->not_off[NLv + 1], c->d_not_out + c->not_off[NLv + 1], (int)c->n_dff, x->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "DFF state launch");
  }
  for (uint32_t L = 0; L < c->levels.size(); L++) {
    const uint32_t n = c->my_count[L];
    if (n) {
      int rc = launch_blind_rotate(x->P, x->p.method == BFHE_AP, c->d_desc + c->desc_off[L], (int)n, x->d_bk, x->d_twl, x->d_psiM,
                                   c->d_ext, nullptr, x->force_g, x->stream, nullptr, &x->v2);
      if (rc) return cuda_fail((cudaError_t)rc, "blind_rotate launch");
      const bool xl = px_on && c->shard_index[L] >= 0;
      const PeerX px = xl ? peer_x(c, (uint32_t)c->shard_index[L]) : PeerX();
      rc = launch_keyswitch(x->P, c->d_ext, c->d_desc + c->desc_off[L], (int)n, x->d_ksk, x->ksk_elem_bytes, x->stream, xl ? &px : nullptr);
      if (rc) return cuda_fail((cudaError_t)rc, "keyswitch launch");
    }
    if (px_on && c->shard_index[L] >= 0) { // outputs were stored into every slab by the key switch: wait for the peers' flags of this level
      int rc = 0;
      if (!n) rc = launch_peer_signal(peer_x(c, (uint32_t)c->shard_index[L]), x->stream); // nothing of this level is mine: only say so
      if (!rc) rc = launch_peer_wait(c->x_flags, c->x_epoch, (u32)c->world, (u32)c->rank, c->shard_index[L], c->x_per_epoch, c->x_err, x->stream);
      if (rc) return cuda_fail((cudaError_t)rc, "peer exchange launch");
    } else if (c->world > 1 && c->level_rpr[L] && c->levels[L].sharded) {
      u32 *base = c->slab + (size_t)c->levels[L].first_row * st;
      const size_t cnt = (size_t)c->level_rpr[L] * st;
      int nrc = g_nccl.AllGather(base + (size_t)c->rank * cnt, base, cnt, NCCL_UINT32, c->comm, x->stream);
      if (nrc) { set_error(std::string("ncclAllGather: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(nrc) : "?")); return BFHE_ERR_NCCL; }
    }
    const size_t nn = c->not_off[L + 1] - c->not_off[L];
    if (nn) {
      int rc = launch_eval_not(x->P, c->d_not_in + c->not_off[L], c->d_not_out + c->not_off[L], (int)nn, x->stream);
      if (rc) return cuda_fail((cudaError_t)rc, "eval_not launch");
    }
  }
  if (c->n_dff) { // latch: scratch[i] = D_i (the state rows keep this clock's Q until the next clock starts, so outputs and verify
                  // mode read consistent values, and a D that is another flip-flop's Q sees the old state)
    int rc = launch_eval_not(x->P, c->d_not_in + c->not_off[NLv], c->d_not_out + c->not_off[NLv], (int)c->n_dff, x->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "DFF latch launch");
  }
  if (px_on) { // end-of-Clock signal: this rank no longer reads its slab, the peers may start storing the next Clock's rows
    int rc = launch_peer_signal(peer_x(c, c->x_per_epoch - 1), x->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "peer exchange launch");
  }
  return BFHE_OK;
}

// ---------------------------------------------------------------------------------------------
// plaintext evaluation (the reference's plaintext_flag path of Gate::Evaluate, src/gate.cpp:86-190)
// ---------------------------------------------------------------------------------------------
static void eval_plain(bfhe_circuit *c) {
  const Netlist &nl = c->nl;
  c->plain_wire.assign(nl.n_wires, 0);
  std::vector<uint32_t> bus_base(nl.in_bits.size() + 1, 0);
  for (size_t b = 0; b < nl.in_bits.size(); b++) bus_base[b + 1] = bus_base[b] + nl.in_bits[b];
  if (c->plain_state.size() != c->n_dff) c->plain_state.assign(c->n_dff, 0); // flip-flops power up at 0
  for (uint32_t i = 0; i < c->n_dff; i++) c->plain_wire[nl.gates[c->dff_gate[i]].out] = c->plain_state[i];
  for (uint32_t gi : c->topo) {
    const NetGate &g = nl.gates[gi];
    auto &w = c->plain_wire;
    switch (g.kind) {
    case GateKind::INPUT: w[g.out] = c->in_bits_set[bus_base[g.in0] + g.in1] & 1; break;
    case GateKind::NOT: w[g.out] = !w[g.in0]; break;
    case GateKind::AND: w[g.out] = w[g.in0] && w[g.in1]; break;
    case GateKind::OR: w[g.out] = w[g.in0] || w[g.in1]; break;
    case GateKind::NAND: w[g.out] = !(w[g.in0] && w[g.in1]); break;
    case GateKind::NOR: w[g.out] = !(w[g.in0] || w[g.in1]); break;
    case GateKind::XOR: case GateKind::XOR_FAST: w[g.out] = w[g.in0] ^ w[g.in1]; break;
    case GateKind::XNOR_FAST: w[g.out] = !(w[g.in0] ^ w[g.in1]); break;
    default: break; // OUTPUT; DFF: Q was set from the state above
    }
  }
  for (uint32_t i = 0; i < c->n_dff; i++) c->plain_state[i] = c->plain_wire[nl.gates[c->dff_gate[i]].in0]; // state := D
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" bfhe_circuit *bfhe_circuit_create(bfhe_ctx *ctx) {
  if (!ctx) { set_error("null context"); return nullptr; }
  bfhe_circuit *c = new bfhe_circuit();
  c->ctx = ctx;
  return c;
}
extern "C" void bfhe_circuit_destroy(bfhe_circuit *c) {
  if (!c) return;
  free_device(c);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  delete c;
}
// any change of the netlist, the schedule or the sharding drops the device state AND the pending input: the next
// SetInput uploads the new plan (Clock without it fails with BFHE_ERR_STATE instead of touching freed buffers)
static int replan(bfhe_circuit *c) {
  free_device(c);
  c->has_input = false;
  c->done = false;
  return build_plan(c);
}
static int after_load(bfhe_circuit *c, std::string err) {
  if (err.empty()) { // composite XNOR = XOR + free NOT (what EvalBinGate(XNOR) computes); LUT3 / LUT4 -> 2-input gates
    Netlist &nl = c->nl;
    if (nl.wire_reg.size() != nl.n_wires) { nl.wire_reg.resize(nl.n_wires); for (uint32_t i = 0; i < nl.n_wires; i++) nl.wire_reg[i] = i; }
    c->nl_file = nl; // dumpNetList / dumpGates / get_netlist describe the file, the plan the lowered netlist
    err = lower_luts(nl);
  }
  if (!err.empty()) { set_error(err); c->loaded = false; return BFHE_ERR_FORMAT; }
  c->loaded = true;
  c->planned = false;
  c->plain_state.clear();
  c->state_init_pending = true;
  c->clocks = 0;
  return replan(c);
}
extern "C" int bfhe_circuit_read_file(bfhe_circuit *c, const char *path) {
  if (!c || !path) return BFHE_ERR_ARG;
  return after_load(c, parse_out_file(path, c->nl));
}
extern "C" int bfhe_circuit_read_bristol(bfhe_circuit *c, const char *path, int new_format) {
  if (!c || !path) return BFHE_ERR_ARG;
  return after_load(c, parse_bristol_file(path, new_format != 0, c->nl));
}
/* netlist straight from arrays: kind[i] in GateEnum order {INPUT, OUTPUT, NOT, AND, OR, XOR, DFF, LUT3, LUT4} (src/gate.h:51) followed by
 * {NAND, NOR, XNOR, XOR_FAST, XNOR_FAST}; INPUT: in0 = bus, in1 = bit, out = wire; OUTPUT: in0 = wire, out = output bit; DFF: in0 = D,
 * out = Q; LUT3 / LUT4: in0..in3 and the truth table (in2 / in3 / table may be NULL when no LUT is present); others: wires */
extern "C" int bfhe_circuit_load_netlist_ex(bfhe_circuit *c, const uint8_t *kind, const uint32_t *in0, const uint32_t *in1, const uint32_t *in2,
                                            const uint32_t *in3, const uint32_t *table, const uint32_t *out, size_t count, uint32_t n_wires,
                                            const uint32_t *in_bits, uint32_t n_in_buses, uint32_t out_bits) {
  if (!c || !kind || !in0 || !in1 || !out || !in_bits) return BFHE_ERR_ARG;
  Netlist nl;
  nl.n_wires = n_wires;
  nl.in_bits.assign(in_bits, in_bits + n_in_buses);
  nl.out_bits = out_bits;
  nl.gates.resize(count);
  for (size_t i = 0; i < count; i++) {
    if (kind[i] >= (uint8_t)GateKind::KIND_COUNT) return after_load(c, "unknown gate kind");
    NetGate &g = nl.gates[i];
    g.kind = (GateKind)kind[i]; g.in0 = in0[i]; g.in1 = in1[i]; g.out = out[i];
    if (g.kind == GateKind::LUT3 || g.kind == GateKind::LUT4) {
      if (!in2 || !table || (g.kind == GateKind::LUT4 && !in3)) return after_load(c, "LUT gate without in2 / in3 / table arrays");
      g.in2 = in2[i]; g.in3 = in3 ? in3[i] : 0; g.table = table[i];
      if (g.in0 >= n_wires || g.in1 >= n_wires || g.in2 >= n_wires || (g.kind == GateKind::LUT4 && g.in3 >= n_wires)) return after_load(c, "wire id out of range");
    }
    nl.count(g.kind);
  }
  c->nl = std::move(nl);
  return after_load(c, "");
}
extern "C" int bfhe_circuit_load_netlist(bfhe_circuit *c, const uint8_t *kind, const uint32_t *in0, const uint32_t *in1,
                                         const uint32_t *out, size_t count, uint32_t n_wires, const uint32_t *in_bits,
                                         uint32_t n_in_buses, uint32_t out_bits) {
  return bfhe_circuit_load_netlist_ex(c, kind, in0, in1, nullptr, nullptr, nullptr, out, count, n_wires, in_bits, n_in_buses, out_bits);
}
/* the netlist that is evaluated (LUTs and XNOR lowered to the 2-input gate set) */
extern "C" int bfhe_circuit_get_netlist(const bfhe_circuit *c, uint8_t *kind, uint32_t *in0, uint32_t *in1, uint32_t *out, size_t cap,
                                        uint32_t *count, uint32_t *n_wires) {
  if (!c || !c->loaded) return BFHE_ERR_STATE;
  if (count) *count = (uint32_t)c->nl.gates.size();
  if (n_wires) *n_wires = c->nl.n_wires;
  if (kind) {
    if (cap < c->nl.gates.size()) return BFHE_ERR_ARG;
    for (size_t i = 0; i < c->nl.gates.size(); i++) {
      kind[i] = (uint8_t)c->nl.gates[i].kind; in0[i] = c->nl.gates[i].in0; in1[i] = c->nl.gates[i].in1; out[i] = c->nl.gates[i].out;
    }
  }
  return BFHE_OK;
}
/* emit the reference's ".out" assembler text (what assemble_bristol writes, src/assemble.cpp:111-114,155-184,310-368,409-425) */
extern "C" int bfhe_circuit_write_out(const bfhe_circuit *c, const char *path) {
  if (!c || !c->loaded || !path) return BFHE_ERR_STATE;
  FILE *f = std::fopen(path, "w");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  const Netlist &nl = c->nl;
  std::fprintf(f, "# Max depth 0\n");
  for (size_t b = 0; b < 2; b++) std::fprintf(f, "# number input%zu bits %u\n", b + 1, b < nl.in_bits.size() ? nl.in_bits[b] : 0);
  std::fprintf(f, "# number output1 bits %u\n", nl.out_bits);
  for (const NetGate &g : nl.gates) {
    const char *two = nullptr;
    switch (g.kind) {
    case GateKind::INPUT: std::fprintf(f, "R%u = LOAD(In%u,%u)\n", g.out, g.in0 + 1, g.in1); break;
    case GateKind::OUTPUT: std::fprintf(f, "Out%u = STORE(R%u) ! depth = 0\n", g.out, g.in0); break;
    case GateKind::NOT: std::fprintf(f, "R%u = NOT(R%u) !depth = 0\n", g.out, g.in0); break;
    case GateKind::DFF: std::fprintf(f, "R%u = DFF(R%u) !depth = 0\n", g.out, g.in0); break;
    case GateKind::AND: two = "AND"; break;
    case GateKind::OR: two = "OR"; break;
    case GateKind::XOR: two = "XOR"; break;
    case GateKind::NAND: two = "NAND"; break;
    case GateKind::NOR: two = "NOR"; break;
    case GateKind::XOR_FAST: two = "XOR_FAST"; break;
    case GateKind::XNOR_FAST: two = "XNOR_FAST"; break;
    default: break;
    }
    if (two) std::fprintf(f, "R%u = %s(R%u, R%u) !depth = 0\n", g.out, two, g.in0, g.in1);
  }
  std::fprintf(f, "# Assembler statistics\n# max depth supported: 0\n# max depth required: 0\n# max tower jump: 0\n# %u registers used\n", nl.n_wires);
  std::fclose(f);
  return BFHE_OK;
}
/* Circuit::dumpNetList (what = 0) / dumpGates (what = 1) text, src/circuit.cpp:844-865.  Returns the length needed (without the
 * terminating 0) in *needed; copies at most cap - 1 characters. */
extern "C" int bfhe_circuit_dump_text(const bfhe_circuit *c, int what, char *buf, size_t cap, size_t *needed) {
  if (!c || !c->loaded) return BFHE_ERR_STATE;
  if (what != 0 && what != 1) return BFHE_ERR_ARG;
  const std::string s = what == 0 ? dump_netlist_text(c->nl_file) : dump_gates_text(c->nl_file);
  if (needed) *needed = s.size();
  if (buf && cap) {
    const size_t n = std::min(cap - 1, s.size());
    std::memcpy(buf, s.data(), n);
    buf[n] = 0;
  }
  return BFHE_OK;
}

extern "C" int bfhe_circuit_set_flags(bfhe_circuit *c, int plaintext, int encrypted, int verify) {
  if (!c) return BFHE_ERR_ARG;
  const bool v = verify != 0;
  // setVerify(true) forces both other modes on (src/circuit.cpp:833-840)
  c->plaintext = plaintext != 0 || v;
  c->encrypted = encrypted != 0 || v;
  // verify mode materialises every NOT output, which is a different row plan.  The reference harness toggles the flags on every
  // iteration (Reset clears them, src/circuit.cpp:378-381): the re-plan is deferred to the next SetInput, so off -> on toggles that
  // end where they started cost nothing.
  c->verify = v;
  return BFHE_OK;
}
extern "C" int bfhe_circuit_info(const bfhe_circuit *c, uint32_t *n_inputs, uint32_t *input_bits, uint32_t *n_output_bits,
                                 uint32_t *n_gates, uint32_t *n_bootstraps, uint32_t *n_levels, uint32_t *max_width) {
  if (!c || !c->loaded) return BFHE_ERR_STATE;
  if (n_inputs) *n_inputs = (uint32_t)c->nl.in_bits.size();
  if (input_bits)
    for (size_t i = 0; i < 8; i++) input_bits[i] = i < c->nl.in_bits.size() ? c->nl.in_bits[i] : 0;
  if (n_output_bits) *n_output_bits = c->nl.out_bits;
  const Netlist &f = c->nl_file;
  if (n_gates) *n_gates = f.n_and + f.n_or + f.n_xor + f.n_not + f.n_nand + f.n_nor + f.n_xnor + f.n_xor_fast + f.n_xnor_fast + f.n_dff + f.n_lut3 + f.n_lut4;
  if (n_bootstraps) *n_bootstraps = c->n_bootstraps;
  if (n_levels) *n_levels = c->asap_levels;
  if (max_width) *max_width = c->max_width;
  return BFHE_OK;
}
extern "C" int bfhe_circuit_dump_gate_count(const bfhe_circuit *c, uint32_t *in, uint32_t *out, uint32_t *and_, uint32_t *or_,
                                            uint32_t *xor_, uint32_t *not_) {
  if (!c || !c->loaded) return BFHE_ERR_STATE;
  if (in) *in = c->nl_file.n_input;
  if (out) *out = c->nl_file.n_output;
  if (and_) *and_ = c->nl_file.n_and;
  if (or_) *or_ = c->nl_file.n_or;
  if (xor_) *xor_ = c->nl_file.n_xor;
  if (not_) *not_ = c->nl_file.n_not;
  return BFHE_OK;
}
/* counts of the gate types beyond the reference's six: {DFF, LUT3, LUT4, NAND, NOR, XNOR, XOR_FAST, XNOR_FAST} */
extern "C" int bfhe_circuit_dump_gate_count_ex(const bfhe_circuit *c, uint32_t *counts8) {
  if (!c || !c->loaded || !counts8) return BFHE_ERR_STATE;
  const Netlist &f = c->nl_file;
  const uint32_t v[8] = {f.n_dff, f.n_lut3, f.n_lut4, f.n_nand, f.n_nor, f.n_xnor, f.n_xor_fast, f.n_xnor_fast};
  std::memcpy(counts8, v, sizeof v);
  return BFHE_OK;
}
extern "C" int bfhe_get_nccl_unique_id(void *out128) {
  if (!out128) return BFHE_ERR_ARG;
  if (!load_nccl()) return BFHE_ERR_NCCL;
  int rc = g_nccl.GetUniqueId(out128);
  if (rc) { set_error("ncclGetUniqueId failed"); return BFHE_ERR_NCCL; }
  return BFHE_OK;
}
extern "C" int bfhe_circuit_set_sharding(bfhe_circuit *c, int rank, int world, const void *id) {
  if (!c || world < 1 || rank < 0 || rank >= world) return BFHE_ERR_ARG;
  free_device(c); // graphs captured with the old communicator must go before it does
  if (c->comm && g_nccl.CommDestroy) { g_nccl.CommDestroy(c->comm); c->comm = nullptr; }
  c->rank = rank;
  c->world = world;
  c->costs.measured = false; // the ranks agree on the costs again
  if (world > 1 && id) { // id == NULL: plan only (tests of the partition on CPU)
    if (c->ctx->device < 0) { set_error("sharded evaluation needs a CUDA device"); return BFHE_ERR_CUDA; }
    if (!load_nccl()) return BFHE_ERR_NCCL;
    BFHE_CUDA(cudaSetDevice(c->ctx->device));
    Id128 uid;
    std::memcpy(uid.b, id, 128);
    int rc = g_nccl.CommInitRank(&c->comm, world, uid, rank);
    if (rc) { set_error(std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?")); return BFHE_ERR_NCCL; }
  }
  if (c->loaded) return replan(c);
  return BFHE_OK;
}
extern "C" int bfhe_circuit_set_wave_capacity(bfhe_circuit *c, int cap) {
  if (!c || cap < -1) return BFHE_ERR_ARG;
  if (cap == c->wave_cap_req) return BFHE_OK;
  c->wave_cap_req = cap;
  if (c->loaded) return replan(c);
  return BFHE_OK;
}
/* world > 1: levels with fewer than min_bootstraps bootstraps are computed redundantly on every rank (no exchange); 0 = shard every
 * level; -1 (default) = per level by the measured cost model when a device is attached, else shard every level */
extern "C" int bfhe_circuit_set_shard_threshold(bfhe_circuit *c, int min_bootstraps) {
  if (!c || min_bootstraps < -1) return BFHE_ERR_ARG;
  if (min_bootstraps == c->shard_min_req) return BFHE_OK;
  c->shard_min_req = min_bootstraps;
  if (c->loaded) return replan(c);
  return BFHE_OK;
}
/* the schedule the planner chose: wave capacity (0 = ASAP levels), number of levels incl. the input level, how many of them are sharded */
extern "C" int bfhe_circuit_exchange_mode(const bfhe_circuit *c) {
  if (!c) return BFHE_ERR_ARG;
  if (c->world <= 1) return 0;
  return c->dev_ready && c->peer_ok ? 2 : 1;
}
extern "C" int bfhe_circuit_get_schedule(const bfhe_circuit *c, uint32_t *wave_cap, uint32_t *n_levels, uint32_t *n_sharded, double *cost_ms4) {
  if (!c || !c->planned) return BFHE_ERR_STATE;
  if (wave_cap) *wave_cap = c->wave_cap;
  if (n_levels) *n_levels = (uint32_t)c->levels.size();
  uint32_t ns = 0;
  for (const Level &l : c->levels) ns += (c->world > 1 && l.sharded && !l.gates.empty()) ? 1 : 0;
  if (n_sharded) *n_sharded = ns;
  if (cost_ms4) { cost_ms4[0] = c->costs.cl4; cost_ms4[1] = c->costs.cl2; cost_ms4[2] = c->costs.lat; cost_ms4[3] = c->costs.thr; }
  return BFHE_OK;
}
extern "C" int bfhe_circuit_level_plan(const bfhe_circuit *c, uint32_t level, int rank, int world, bfhe_gate *out, size_t cap,
                                       uint32_t *count, uint32_t *first_row, uint32_t *rows_per_rank) {
  if (!c || !c->planned || level >= c->levels.size()) return BFHE_ERR_ARG;
  if (world != c->world) { set_error("plan was built for a different world size"); return BFHE_ERR_STATE; }
  uint32_t b, n;
  my_slice(c, level, rank, &b, &n);
  if (count) *count = n;
  if (first_row) *first_row = c->levels[level].first_row;
  if (rows_per_rank) *rows_per_rank = c->levels[level].sharded || c->world == 1 ? c->level_rpr[level] : 0; // 0: no exchange after this level
  if (out) {
    if (cap < n) return BFHE_ERR_ARG;
    std::memcpy(out, c->levels[level].gates.data() + b, n * sizeof(bfhe_gate));
  }
  return BFHE_OK;
}
extern "C" int bfhe_circuit_plan_misc(const bfhe_circuit *c, uint32_t *total_rows, uint32_t *fresh_base, uint32_t *n_levels_incl_input,
                                      uint32_t *out_rows /*[out_bits]*/, uint32_t *not_count, uint32_t level,
                                      uint32_t *not_pairs /*[2*not_count] in,out*/) {
  if (!c || !c->planned) return BFHE_ERR_STATE;
  if (total_rows) *total_rows = c->total_rows;
  if (fresh_base) *fresh_base = c->fresh_base;
  if (n_levels_incl_input) *n_levels_incl_input = (uint32_t)c->levels.size();
  if (out_rows)
    for (uint32_t b = 0; b < c->nl.out_bits; b++) out_rows[b] = c->wire_row[c->out_wire[b]] | (c->wire_neg[c->out_wire[b]] ? 0x80000000u : 0);
  if (level < c->levels.size()) {
    if (not_count) *not_count = (uint32_t)c->levels[level].nots.size();
    if (not_pairs)
      for (size_t k = 0; k < c->levels[level].nots.size(); k++) {
        not_pairs[2 * k] = c->levels[level].nots[k].in_row;
        not_pairs[2 * k + 1] = c->levels[level].nots[k].out_row;
      }
  }
  return BFHE_OK;
}
/* clocked circuits, for tests of the plan: n_dff, and per flip-flop {row D is read from | bit 31 = through EvalNOT, state row (Q),
 * scratch row, row of the fresh encryption of the power-up value 0 that the first clock bootstraps into the state row} */
extern "C" int bfhe_circuit_dff_plan(const bfhe_circuit *c, uint32_t *n_dff, uint32_t *quads, size_t cap_dffs) {
  if (!c || !c->planned) return BFHE_ERR_STATE;
  if (n_dff) *n_dff = c->n_dff;
  if (quads) {
    if (cap_dffs < c->n_dff) return BFHE_ERR_ARG;
    for (uint32_t i = 0; i < c->n_dff; i++) {
      quads[4 * i] = c->dff_ops[i].in_row | (c->dff_ops[i].copy ? 0 : 0x80000000u);
      quads[4 * i + 1] = c->state_base + i;
      quads[4 * i + 2] = c->dff_tmp_base + i;
      quads[4 * i + 3] = c->dff_fresh_base + i;
    }
  }
  return BFHE_OK;
}

extern "C" int bfhe_circuit_reset(bfhe_circuit *c) {
  if (!c || !c->loaded) return BFHE_ERR_STATE;
  // Circuit::Reset clears the mode flags as well (src/circuit.cpp:378-381); callers set them again afterwards,
  // exactly as the reference harnesses do (src/test_adder.cpp:228-233).  Flip-flops go back to their power-up state.
  c->has_input = false;
  c->done = false;
  c->device_ms = c->host_ms = 0;
  c->verify_mismatches = c->verify_checked = 0;
  c->plain_state.clear();
  c->state_init_pending = true;
  c->clocks = 0;
  return BFHE_OK;
}

// The common tail of SetInput on bits and on ciphertexts, once the fresh rows are enqueued on the launch stream: broadcast rank 0's
// rows [fresh_base, +bcast_words) where the ranks' rows may differ, bootstrap the flip-flops' power-up values into the latch rows,
// synchronise.  ct: the rows came from outside the program; the status word after the slab's last row holds the lowest row the
// ingest rejected (0xffffffff: none), and a rejected input leaves the circuit without input.
static int commit_input(bfhe_circuit *c, bool init_state, size_t bcast_words, bool ct) {
  bfhe_ctx *x = c->ctx;
  const size_t st = x->p.ct_stride;
  if (bcast_words) {
    u32 *fresh = c->slab + (size_t)c->fresh_base * st;
    int nrc = g_nccl.Broadcast(fresh, fresh, bcast_words, NCCL_UINT32, 0, c->comm, x->stream);
    if (nrc) { set_error(ct ? "ncclBroadcast of the input ciphertexts failed" : "ncclBroadcast of the fresh input encryptions failed"); return BFHE_ERR_NCCL; }
  }
  if (init_state) {
    std::vector<DevGate> init(c->n_dff);
    for (uint32_t i = 0; i < c->n_dff; i++) {
      const u32 *src = c->slab + (size_t)(c->dff_fresh_base + i) * st;
      init[i] = DevGate{src, src, c->slab + (size_t)(c->dff_tmp_base + i) * st, BFHE_BOOTSTRAP, 0}; // latched; the clock moves it into the state row
    }
    int rc = run_gate_list(x, init.data(), init.size(), nullptr);
    if (rc) return rc;
    c->state_init_pending = false;
  }
  u32 bad_row = 0xffffffffu;
  if (ct) BFHE_CUDA(cudaMemcpyAsync(&bad_row, c->slab + (size_t)c->total_rows * st, sizeof bad_row, cudaMemcpyDeviceToHost, x->stream));
  BFHE_CUDA(cudaStreamSynchronize(x->stream));
  if (bad_row != 0xffffffffu) {
    set_error("SetInput: input ciphertext row " + std::to_string(bad_row) + " has a word >= q");
    return BFHE_ERR_FORMAT;
  }
  c->has_input = true;
  return BFHE_OK;
}

extern "C" int bfhe_circuit_set_input(bfhe_circuit *c, const uint8_t *bits, size_t nbits, uint64_t seed) {
  if (!c || !c->loaded || !bits) return BFHE_ERR_STATE;
  if (c->planned_verify != c->verify || !c->planned) { // the deferred re-plan of set_flags
    c->planned_verify = c->verify;
    int rc = replan(c);
    if (rc) return rc;
  }
  if (nbits != c->n_in) { set_error("SetInput: expected " + std::to_string(c->n_in) + " bits, got " + std::to_string(nbits)); return BFHE_ERR_ARG; }
  c->in_bits_set.assign(bits, bits + nbits);
  c->ct_input = false;
  c->has_input = false;
  c->done = false;
  if (c->encrypted) {
    if (!c->dev_ready) {
      int rc = upload_plan(c);
      if (rc) return rc;
      c->state_init_pending = true; // a new slab has no flip-flop state
    }
    bfhe_ctx *x = c->ctx;
    std::lock_guard<std::mutex> lk(x->mtx);
    BFHE_CUDA(cudaSetDevice(x->device));
    const size_t st = x->p.ct_stride;
    // fresh encryptions on the host; the Bootstrap that Encrypt's BOOTSTRAPPED default applies (src/circuit.cpp:506) is level 0 of
    // the plan.  Every rank must hold the same rows: with an explicit seed they are deterministic; with seed 0 (OS entropy) rank 0
    // encrypts and the rows are broadcast.
    const bool init_state = c->state_init_pending && c->n_dff > 0;
    const size_t nfresh = (size_t)c->n_in + (init_state ? c->n_dff : 0);
    std::vector<u32> fresh(nfresh * st);
    if (c->world == 1 || seed != 0 || c->rank == 0) {
      int rc = bfhe_encrypt(x, bits, nbits, seed, fresh.data());
      if (rc) return rc;
      if (init_state) { // flip-flops power up at 0: Encrypt(0), bootstrapped into the state rows by commit_input
        std::vector<uint8_t> zeros(c->n_dff, 0);
        rc = bfhe_encrypt(x, zeros.data(), zeros.size(), seed ? seed ^ 0xD1FFull : 0, fresh.data() + (size_t)c->n_in * st);
        if (rc) return rc;
      }
    }
    // fresh_base .. fresh_base + n_in and dff_fresh_base .. are adjacent rows (build_plan_cap)
    BFHE_CUDA(cudaMemcpyAsync(c->slab + (size_t)c->fresh_base * st, fresh.data(), fresh.size() * 4, cudaMemcpyHostToDevice, x->stream));
    return commit_input(c, init_state, c->world > 1 && seed == 0 ? fresh.size() : 0, false);
  }
  c->has_input = true;
  return BFHE_OK;
}

extern "C" int bfhe_circuit_set_input_ct(bfhe_circuit *c, const uint32_t *cts, size_t nbits, int on_device) {
  if (!c) return BFHE_ERR_ARG;
  if (!c->loaded) { set_error("SetInput before a netlist was loaded"); return BFHE_ERR_STATE; }
  if (!c->encrypted || c->plaintext || c->verify) {
    set_error("SetInput on ciphertexts needs encrypted mode with plaintext and verify mode off (ciphertext inputs have no plaintext)");
    return BFHE_ERR_STATE;
  }
  if (c->planned_verify || !c->planned) {
    c->planned_verify = false;
    int rc = replan(c);
    if (rc) return rc;
  }
  if (nbits != c->n_in) { set_error("SetInput: expected " + std::to_string(c->n_in) + " ciphertexts, got " + std::to_string(nbits)); return BFHE_ERR_ARG; }
  const bool source = c->world == 1 || c->rank == 0; // sharded: rank 0's rows are used, the other ranks' buffers are not read
  if (source && !cts && nbits) { set_error("SetInput: null ciphertext buffer"); return BFHE_ERR_ARG; }
  c->in_bits_set.clear();
  c->ct_input = true;
  c->has_input = false;
  c->done = false;
  if (!c->dev_ready) {
    int rc = upload_plan(c);
    if (rc) return rc;
    c->state_init_pending = true;
  }
  bfhe_ctx *x = c->ctx;
  std::lock_guard<std::mutex> lk(x->mtx);
  BFHE_CUDA(cudaSetDevice(x->device));
  const size_t st = x->p.ct_stride;
  const bool init_state = c->state_init_pending && c->n_dff > 0;
  if (source) {
    if (on_device && nbits) {
      cudaPointerAttributes pa{};
      if (cudaPointerGetAttributes(&pa, cts) != cudaSuccess || (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) ||
          pa.device != x->device) {
        cudaGetLastError();
        set_error("SetInput: the ciphertext buffer is not memory of device " + std::to_string(x->device));
        return BFHE_ERR_ARG;
      }
    }
    u32 *fresh = c->slab + (size_t)c->fresh_base * st, *status = c->slab + (size_t)c->total_rows * st;
    if (nbits)
      BFHE_CUDA(cudaMemcpyAsync(fresh, cts, nbits * st * 4, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, x->stream));
    BFHE_CUDA(cudaMemsetAsync(status, 0xff, sizeof(u32), x->stream));
    int rc = launch_ct_ingest(x->P, fresh, (int)nbits, status, x->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "ct_ingest launch");
    // no secret key, no Encrypt(0): flip-flops power up from the trivial encryption of 0.  The rows may still hold a bit-path
    // SetInput's Encrypt(0).
    if (init_state) BFHE_CUDA(cudaMemsetAsync(c->slab + (size_t)c->dff_fresh_base * st, 0, (size_t)c->n_dff * st * 4, x->stream));
  }
  // sharded: the input rows, the flip-flops' fresh rows and the status word are adjacent (build_plan_cap, upload_plan)
  const size_t bcast = c->world > 1 ? ((size_t)c->n_in + c->n_dff) * st + 1 : 0;
  return commit_input(c, init_state, bcast, true);
}

// Circuit::Clock.  out_cts == nullptr: the outputs are decrypted into out_bits (cap bits); else they stay encrypted and go to out_cts
// (cap rows of ct_stride words, device memory when on_device)
static int clock_run(bfhe_circuit *c, uint8_t *out_bits, size_t cap, uint8_t *plain_out_bits, uint32_t *out_cts, int on_device) {
  if (!c || !c->planned) return BFHE_ERR_STATE;
  if (!c->has_input) { set_error("Clock before SetInput (or after a change of flags / schedule / sharding: call SetInput again)"); return BFHE_ERR_STATE; }
  // a combinational circuit is done after one clock (src/circuit.cpp:538-541); one with flip-flops is clocked again and again
  if (c->done && c->n_dff == 0) { set_error("done ckt clocked! should reset"); return BFHE_ERR_STATE; }
  if (c->encrypted && (!c->dev_ready || !c->slab)) { set_error("Clock: encrypted mode was switched on after SetInput; call SetInput again"); return BFHE_ERR_STATE; }
  if (c->encrypted && c->world > 1 && !c->comm) { set_error("Clock: sharded evaluation without an NCCL communicator"); return BFHE_ERR_STATE; }
  if (c->verify != c->planned_verify) { set_error("Clock: verify mode changed after SetInput; call SetInput again"); return BFHE_ERR_STATE; }
  if (c->plaintext && c->ct_input) { set_error("Clock: plaintext mode needs input bits; the input was set as ciphertexts"); return BFHE_ERR_STATE; }
  if (!out_cts && c->encrypted && !c->ctx->has_sk) { set_error("Clock: decrypting the outputs needs the secret key (clock_ct returns them encrypted)"); return BFHE_ERR_STATE; }
  const uint32_t nout = c->nl.out_bits;
  if (cap < nout) return BFHE_ERR_ARG;
  auto t0 = std::chrono::steady_clock::now();
  if (c->plaintext || c->verify) {
    eval_plain(c);
    uint8_t *dst = plain_out_bits ? plain_out_bits : (c->encrypted ? nullptr : out_bits);
    if (dst)
      for (uint32_t b = 0; b < nout; b++) dst[b] = c->plain_wire[c->out_wire[b]];
  }
  if (c->encrypted) {
    bfhe_ctx *x = c->ctx;
    std::lock_guard<std::mutex> lk(x->mtx);
    BFHE_CUDA(cudaSetDevice(x->device));
    const size_t st = x->p.ct_stride;
    if (out_cts && on_device && nout) {
      cudaPointerAttributes pa{};
      if (cudaPointerGetAttributes(&pa, out_cts) != cudaSuccess || (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) ||
          pa.device != x->device) {
        cudaGetLastError();
        set_error("Clock: the output buffer is not memory of device " + std::to_string(x->device));
        return BFHE_ERR_ARG;
      }
    }
    cudaEvent_t e0, e1;
    BFHE_CUDA(cudaEventCreate(&e0));
    BFHE_CUDA(cudaEventCreate(&e1));
    int rc = BFHE_OK;
    if (c->use_graph && !c->graph) { // one CUDA graph per circuit, sharded or not (NCCL collectives are capturable)
      if (c->world > 1 && !c->peer_ok) { // NCCL's lazy set-up (channels, buffers) must happen outside the capture: one eager exchange first
        int nrc = g_nccl.AllGather(c->slab + (size_t)c->rank * st, c->slab, st, NCCL_UINT32, c->comm, x->stream);
        if (nrc) { set_error("ncclAllGather warm-up failed"); return BFHE_ERR_NCCL; }
        BFHE_CUDA(cudaStreamSynchronize(x->stream));
        // rows 0 .. world-1 (level-0 outputs) were overwritten with copies of themselves per rank: level 0 rewrites them
      }
      cudaGraph_t g = nullptr;
      BFHE_CUDA(cudaStreamBeginCapture(x->stream, c->world > 1 && !c->peer_ok ? cudaStreamCaptureModeRelaxed : cudaStreamCaptureModeThreadLocal));
      rc = enqueue_levels(c);
      cudaError_t ce = cudaStreamEndCapture(x->stream, &g);
      if (rc) { if (g) cudaGraphDestroy(g); return rc; }
      if (ce != cudaSuccess) return cuda_fail(ce, "cudaStreamEndCapture");
      ce = cudaGraphInstantiate(&c->graph, g, 0);
      cudaGraphDestroy(g);
      if (ce != cudaSuccess) return cuda_fail(ce, "cudaGraphInstantiate");
    }
    BFHE_CUDA(cudaEventRecord(e0, x->stream));
    if (c->use_graph) {
      BFHE_CUDA(cudaGraphLaunch(c->graph, x->stream));
    } else {
      rc = enqueue_levels(c);
      if (rc) return rc;
    }
    BFHE_CUDA(cudaEventRecord(e1, x->stream));
    BFHE_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    c->device_ms += ms;
    if (c->world > 1 && c->peer_ok) { // a wait for a peer's flag timed out (the kernels do not hang: they record which peer and go on)
      u32 xe = 0;
      BFHE_CUDA(cudaMemcpy(&xe, c->x_err, sizeof xe, cudaMemcpyDeviceToHost));
      if (xe) { set_error("multi-GPU exchange: no signal from rank " + std::to_string(xe - 1) + " within the exchange timeout (rank lost, or the ranks disagree on the schedule)"); return BFHE_ERR_NCCL; }
    }
    if (out_cts) { // outputs stay encrypted: one launch copies every output row, through EvalNOT where the output reads its row negated
      u32 *dst = out_cts;
      if (!on_device) {
        if (!c->d_egress) BFHE_CUDA(cudaMalloc(&c->d_egress, std::max<size_t>(nout, 1) * st * 4));
        dst = c->d_egress;
      }
      BFHE_CUDA(cudaMemsetAsync(dst, 0, (size_t)nout * st * 4, x->stream)); // the kernel writes the ct_words, not the padding
      std::vector<const u32 *> in(nout);
      std::vector<u32 *> out(nout);
      for (uint32_t b = 0; b < nout; b++) {
        const uint32_t w = c->out_wire[b];
        in[b] = reinterpret_cast<const u32 *>(reinterpret_cast<uintptr_t>(c->slab + (size_t)c->wire_row[w] * st) | (c->wire_neg[w] ? 0u : 1u));
        out[b] = dst + (size_t)b * st;
      }
      rc = not_ptr_batch(x, in, out);
      if (rc) return rc;
      if (!on_device) BFHE_CUDA(cudaMemcpyAsync(out_cts, dst, (size_t)nout * st * 4, cudaMemcpyDeviceToHost, x->stream));
      BFHE_CUDA(cudaStreamSynchronize(x->stream));
    } else if (c->verify) { // OUTPUT gates: decrypt on the host (src/circuit.cpp:796-801)
      std::vector<u32> rows((size_t)c->total_rows * st);
      BFHE_CUDA(cudaMemcpy(rows.data(), c->slab, rows.size() * 4, cudaMemcpyDeviceToHost));
      std::vector<uint8_t> dec(c->total_rows);
      rc = bfhe_decrypt(x, rows.data(), c->total_rows, dec.data());
      if (rc) return rc;
      // gate-by-gate check of every wire that owns a ciphertext against the plaintext evaluation
      // (src/gate.cpp:113-120,153-160,174-181,206-213 -- reported, not "fixed")
      for (uint32_t w = 0; w < c->nl.n_wires; w++) {
        if (c->wire_row[w] == 0xffffffffu) continue;
        const uint8_t v = dec[c->wire_row[w]] ^ c->wire_neg[w];
        c->verify_checked++;
        if (v != c->plain_wire[w]) c->verify_mismatches++;
      }
      for (uint32_t b = 0; b < nout; b++) out_bits[b] = dec[c->wire_row[c->out_wire[b]]] ^ c->wire_neg[c->out_wire[b]];
    } else {
      std::vector<u32> orow((size_t)nout * st);
      for (uint32_t b = 0; b < nout; b++)
        BFHE_CUDA(cudaMemcpyAsync(orow.data() + (size_t)b * st, c->slab + (size_t)c->wire_row[c->out_wire[b]] * st, st * 4,
                                  cudaMemcpyDeviceToHost, x->stream));
      BFHE_CUDA(cudaStreamSynchronize(x->stream));
      std::vector<uint8_t> dec(nout);
      rc = bfhe_decrypt(x, orow.data(), nout, dec.data());
      if (rc) return rc;
      for (uint32_t b = 0; b < nout; b++) out_bits[b] = dec[b] ^ c->wire_neg[c->out_wire[b]];
    }
  }
  c->done = true;
  c->clocks++;
  c->host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return BFHE_OK;
}
extern "C" int bfhe_circuit_clock(bfhe_circuit *c, uint8_t *out_bits, size_t cap, uint8_t *plain_out_bits) {
  return clock_run(c, out_bits, cap, plain_out_bits, nullptr, 0);
}
extern "C" int bfhe_circuit_clock_ct(bfhe_circuit *c, uint32_t *out_cts, size_t cap_rows, int on_device) {
  if (!c || !out_cts) return BFHE_ERR_ARG;
  if (!c->encrypted || c->verify) { set_error("Clock on ciphertexts needs encrypted mode with verify mode off"); return BFHE_ERR_STATE; }
  return clock_run(c, nullptr, cap_rows, nullptr, out_cts, on_device);
}

extern "C" int bfhe_circuit_stats(const bfhe_circuit *c, double *device_ms, double *host_ms, uint64_t *verify_mismatches) {
  if (!c) return BFHE_ERR_ARG;
  if (device_ms) *device_ms = c->device_ms;
  if (host_ms) *host_ms = c->host_ms;
  if (verify_mismatches) *verify_mismatches = c->verify_mismatches;
  return BFHE_OK;
}
extern "C" int bfhe_circuit_use_graph(bfhe_circuit *c, int on) {
  if (!c) return BFHE_ERR_ARG;
  c->use_graph = on != 0;
  return BFHE_OK;
}
/* wire-level ciphertext access for parity tests: row of output bit b (host copy) */
extern "C" int bfhe_circuit_download_slab(bfhe_circuit *c, uint32_t *host, size_t rows_cap) {
  if (!c || !c->dev_ready) return BFHE_ERR_STATE;
  if (rows_cap < c->total_rows) return BFHE_ERR_ARG;
  BFHE_CUDA(cudaSetDevice(c->ctx->device));
  BFHE_CUDA(cudaMemcpy(host, c->slab, (size_t)c->total_rows * c->ctx->p.ct_stride * 4, cudaMemcpyDeviceToHost));
  return BFHE_OK;
}
