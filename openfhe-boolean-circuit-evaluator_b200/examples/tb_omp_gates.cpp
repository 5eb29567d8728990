// tb_omp_gates.cpp -- the reference's per-gate path over host/binfhecontext.h: _CircuitManager's ready-gate waves, each run as one OpenMP
// task per gate (src/circuit.cpp:593-710), each task evaluating its gate through lbcrypto::BinFHEContext as src/gate.cpp:84-214 does.
// Tasks that call EvalBinGate at the same time are combined into shared GPU waves by bfhe_eval_bingate_host.  The same fresh inputs
// then go through the level-synchronous evaluator (bfhe_circuit_set_input_ct / bfhe_circuit_clock_ct) on the same context, and the two
// paths' output ciphertexts are compared word for word.
//     usage: tb_omp_gates <circuit .out file> [-s TOY|STD128_OPT] [-m AP|GINX] [-k key seed] [-i input seed]
// Prints one "key value" line per figure; exit code 0 when both paths agree word for word and decrypt alike.
#include "../host/binfhecontext.h"
#include <chrono>
#include <cstdio>
#include <cstring>
#include <omp.h>
#include <random>

using namespace lbcrypto;

// netlist kinds of bfhe_circuit_get_netlist (include/bfhe.h)
enum { K_INPUT, K_OUTPUT, K_NOT, K_AND, K_OR, K_XOR, K_DFF, K_LUT3, K_LUT4, K_NAND, K_NOR };

static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int main(int argc, char **argv) {
  if (argc < 2) { std::fprintf(stderr, "usage: %s <circuit .out file> [-s set] [-m method] [-k key seed] [-i input seed]\n", argv[0]); return 2; }
  BINFHE_PARAMSET set = STD128_OPT;
  BINFHE_METHOD method = GINX;
  uint64_t key_seed = 1, input_seed = 7;
  for (int i = 2; i + 1 < argc; i += 2) {
    if (!std::strcmp(argv[i], "-s")) set = !std::strcmp(argv[i + 1], "TOY") ? TOY : STD128_OPT;
    else if (!std::strcmp(argv[i], "-m")) method = !std::strcmp(argv[i + 1], "AP") ? AP : GINX;
    else if (!std::strcmp(argv[i], "-k")) key_seed = std::strtoull(argv[i + 1], nullptr, 0);
    else if (!std::strcmp(argv[i], "-i")) input_seed = std::strtoull(argv[i + 1], nullptr, 0);
  }
  BinFHEContext cc;
  cc.GenerateBinFHEContext(set, method, 0);
  auto sk = cc.KeyGen(key_seed);
  cc.BTKeyGen(sk, key_seed + 1);
  bfhe_circuit *circ = bfhe_circuit_create(cc.raw());
  if (bfhe_circuit_read_file(circ, argv[1]) != BFHE_OK) { std::fprintf(stderr, "%s\n", bfhe_last_error()); return 1; }
  uint32_t count = 0, n_wires = 0, n_buses = 0, bus_bits[8], n_out = 0;
  bfhe_circuit_get_netlist(circ, nullptr, nullptr, nullptr, nullptr, 0, &count, &n_wires);
  std::vector<uint8_t> kind(count);
  std::vector<uint32_t> in0(count), in1(count), out(count);
  bfhe_circuit_get_netlist(circ, kind.data(), in0.data(), in1.data(), out.data(), count, &count, &n_wires);
  bfhe_circuit_info(circ, &n_buses, bus_bits, &n_out, nullptr, nullptr, nullptr, nullptr);
  std::vector<uint32_t> bus_base(n_buses + 1, 0);
  for (uint32_t b = 0; b < n_buses; b++) bus_base[b + 1] = bus_base[b] + bus_bits[b];
  const uint32_t n_in = bus_base[n_buses];
  size_t boots = n_in; // Encrypt's default output is BOOTSTRAPPED
  for (uint32_t g = 0; g < count; g++) {
    switch (kind[g]) {
    case K_INPUT: case K_OUTPUT: case K_NOT: break;
    case K_AND: case K_OR: case K_NAND: case K_NOR: boots += 1; break;
    case K_XOR: boots += 3; break;
    default: std::fprintf(stderr, "gate %u: kind %u is not one the reference's gate.cpp evaluates (AND, OR, NAND, NOR, NOT, XOR)\n", g, kind[g]); return 2;
    }
  }

  // fresh encryptions of seeded random bits, one per input bit (buses concatenated in SetInput's order)
  const size_t st = cc.params().ct_stride, words = cc.params().ct_words;
  std::vector<uint8_t> bits(n_in);
  std::mt19937_64 rng(input_seed);
  for (auto &b : bits) b = (uint8_t)(rng() & 1);
  std::vector<uint32_t> fresh((size_t)n_in * st);
  if (bfhe_encrypt(cc.raw(), bits.data(), n_in, input_seed, fresh.data()) != BFHE_OK) { std::fprintf(stderr, "%s\n", bfhe_last_error()); return 1; }
  auto row_ct = [&](const uint32_t *row) {
    auto ct = std::make_shared<LWECiphertextImpl>();
    ct->row.assign(row, row + st);
    return ct;
  };
  cc.Bootstrap(row_ct(fresh.data())); // warm-up: module load and first-launch costs stay out of the timed run

  // the reference's scheduler: ready-gate waves, one OpenMP task per gate
  std::vector<LWECiphertext> wire(n_wires);
  std::vector<char> done(count, 0), ready(n_wires, 0);
  std::vector<LWECiphertext> outs(n_out);
  bfhe_profile_read(cc.raw(), 0, nullptr, nullptr);
  bfhe_profile_read(cc.raw(), 1, nullptr, nullptr);
  bfhe_profile_enable(cc.raw(), 1);
  bool failed = false;
  const double t0 = now_ms();
  size_t n_waves = 0;
  for (size_t left = count;;) {
    std::vector<uint32_t> wave;
    for (uint32_t g = 0; g < count; g++) {
      if (done[g]) continue;
      const bool two = kind[g] != K_INPUT && kind[g] != K_OUTPUT && kind[g] != K_NOT;
      if (kind[g] == K_INPUT || (ready[in0[g]] && (!two || ready[in1[g]]))) wave.push_back(g);
    }
    if (wave.empty()) break;
#pragma omp parallel
#pragma omp single
    for (uint32_t g : wave) {
#pragma omp task firstprivate(g)
      {
        try {
          switch (kind[g]) {
          case K_INPUT: wire[out[g]] = cc.Bootstrap(row_ct(fresh.data() + (size_t)(bus_base[in0[g]] + in1[g]) * st)); break;
          case K_OUTPUT: outs[out[g]] = wire[in0[g]]; break;
          case K_NOT: wire[out[g]] = cc.EvalNOT(wire[in0[g]]); break;
          case K_AND: wire[out[g]] = cc.EvalBinGate(AND, wire[in0[g]], wire[in1[g]]); break;
          case K_OR: wire[out[g]] = cc.EvalBinGate(OR, wire[in0[g]], wire[in1[g]]); break;
          case K_NAND: wire[out[g]] = cc.EvalBinGate(NAND, wire[in0[g]], wire[in1[g]]); break;
          case K_NOR: wire[out[g]] = cc.EvalBinGate(NOR, wire[in0[g]], wire[in1[g]]); break;
          case K_XOR: { // src/gate.cpp:190-202: two NOTs, AND(a, !b), AND(!a, b), OR of the two
            const LWECiphertext &a = wire[in0[g]], &b = wire[in1[g]];
            auto na = cc.EvalNOT(a), nb = cc.EvalNOT(b);
            auto t1 = cc.EvalBinGate(AND, a, nb), t2 = cc.EvalBinGate(AND, na, b);
            wire[out[g]] = cc.EvalBinGate(OR, t1, t2);
            break;
          }
          }
        } catch (const std::exception &e) {
#pragma omp critical
          {
            std::fprintf(stderr, "gate %u: %s\n", g, e.what());
            failed = true;
          }
        }
      }
    }
    if (failed) return 1;
    for (uint32_t g : wave) {
      done[g] = 1;
      if (kind[g] != K_OUTPUT) ready[out[g]] = 1;
    }
    left -= wave.size();
    n_waves++;
    if (!left) break;
  }
  const double omp_ms = now_ms() - t0;
  bfhe_profile_enable(cc.raw(), 0);
  uint64_t br = 0, ks = 0;
  bfhe_profile_read(cc.raw(), 0, nullptr, &br);
  bfhe_profile_read(cc.raw(), 1, nullptr, &ks);
  for (uint32_t b = 0; b < n_out; b++)
    if (!outs[b]) { std::fprintf(stderr, "output bit %u never stored\n", b); return 1; }

  // the same fresh rows through the level-synchronous evaluator on the same context; the second Clock is the steady-state figure
  std::vector<uint32_t> clk((size_t)n_out * st);
  double clock_ms[2] = {0, 0};
  bfhe_circuit_reset(circ);
  bfhe_circuit_set_flags(circ, 0, 1, 0);
  for (int rep = 0; rep < 2; rep++) {
    if (bfhe_circuit_set_input_ct(circ, fresh.data(), n_in, 0) != BFHE_OK) { std::fprintf(stderr, "%s\n", bfhe_last_error()); return 1; }
    const double c0 = now_ms();
    if (bfhe_circuit_clock_ct(circ, clk.data(), n_out, 0) != BFHE_OK) { std::fprintf(stderr, "%s\n", bfhe_last_error()); return 1; }
    clock_ms[rep] = now_ms() - c0;
  }
  bool equal = true;
  std::vector<uint8_t> dec_omp(n_out), dec_clk(n_out);
  for (uint32_t b = 0; b < n_out; b++) {
    equal = equal && std::equal(outs[b]->row.begin(), outs[b]->row.begin() + words, clk.begin() + (size_t)b * st);
    bfhe_decrypt(cc.raw(), outs[b]->row.data(), 1, &dec_omp[b]);
  }
  bfhe_decrypt(cc.raw(), clk.data(), n_out, dec_clk.data());
  std::string in_s, out_s;
  for (auto b : bits) in_s += char('0' + b);
  for (auto b : dec_omp) out_s += char('0' + b);
  std::printf("threads %d\n", omp_get_max_threads());
  std::printf("gates %u\nbootstraps %zu\nwaves %zu\n", count, boots, n_waves);
  std::printf("inputs %s\n", in_s.c_str());
  std::printf("outputs %s\n", out_s.c_str());
  std::printf("decrypt_equal %d\n", dec_omp == dec_clk ? 1 : 0);
  std::printf("ct_equal %d\n", equal ? 1 : 0);
  std::printf("omp_wall_ms %.3f\n", omp_ms);
  std::printf("br_launches %llu\nks_launches %llu\n", (unsigned long long)br, (unsigned long long)ks);
  std::printf("bootstraps_per_launch %.2f\n", br ? (double)boots / br : 0.0);
  std::printf("clock_ms %.3f\nclock_first_ms %.3f\n", clock_ms[1], clock_ms[0]);
  bfhe_circuit_destroy(circ);
  return equal && dec_omp == dec_clk ? 0 : 1;
}
