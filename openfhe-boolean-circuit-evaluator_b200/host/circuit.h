// circuit.h -- the reference's Circuit / Gate / Wire public interface (src/circuit.h:46-114, src/gate.h:51-80,
// src/wire.h:45-73) over the level-synchronous GPU evaluator.  Same names, argument meaning and error behaviour, so
// the reference's harnesses (src/test_adder.cpp:155-156,228-233,265-270 ...) read unchanged:
//     Circuit circ(set, method); circ.ReadFile(f);
//     circ.Reset(); circ.setEncrypted(true); circ.setVerify(true); circ.SetInput(inputs); out = circ.Clock();
// Header-only; link with libbfhe_b200.so.
#pragma once
#include "binfhecontext.h"
#include <cstdlib>
#include <iostream>
#include <string>
#include <vector>

using NameList = std::vector<std::string>;
using CipherText = lbcrypto::LWECiphertext;
using Inputs = std::vector<std::vector<unsigned int>>;
using Outputs = std::vector<std::vector<unsigned int>>;

enum class GateEnum { INPUT, OUTPUT, NOT, AND, OR, XOR, DFF, LUT3, LUT4 };

// One gate of a wavefront.  In the reference a Gate is a heap of strings and shared_ptrs evaluated as one OpenMP
// task; here it is the 16-byte descriptor the batched kernels consume.
using Gate = bfhe_gate;

class GateEvalParams {
public:
  bool plaintext_flag = false, encrypted_flag = false, verify_flag = false;
  lbcrypto::BinFHEContext cc;
  lbcrypto::LWEPrivateKey sk;
};

// A wire is a row of the device slab (replaces Wire::ct, src/wire.h:72).
class Wire {
public:
  void setName(std::string n) { name = std::move(n); }
  std::string getName() const { return name; }
  void setValue(bool b) { value = b; }
  bool getValue() const { return value; }
  void setRow(uint32_t r) { row = r; }
  uint32_t getRow() const { return row; }

private:
  std::string name;
  bool value = false;
  uint32_t row = 0;
};

class Circuit {
public:
  // key_seed == 0 (default): keys and input encryptions from OS entropy; non-zero: reproducible, for tests only
  Circuit(lbcrypto::BINFHE_PARAMSET set, lbcrypto::BINFHE_METHOD method, int device = 0, uint64_t key_seed = 0) {
    // only TOY / STD128_OPT and AP / GINX, otherwise exit(-1), as src/circuit.cpp:69-86
    if (set != lbcrypto::TOY && set != lbcrypto::STD128_OPT) {
      std::cerr << "bad paramset" << std::endl;
      std::exit(-1);
    }
    if (method != lbcrypto::AP && method != lbcrypto::GINX) {
      std::cerr << "bad method" << std::endl;
      std::exit(-1);
    }
    cc.GenerateBinFHEContext(set, method, device); // src/circuit.cpp:88
    sk = cc.KeyGen(key_seed);                      // :90
    cc.BTKeyGen(sk, key_seed ? key_seed + 1 : 0);  // :91
    input_seed = key_seed ? key_seed + 2 : 0;
    gep.cc = cc;                                   // shares keys, :93-97
    gep.sk = sk;
    h = bfhe_circuit_create(cc.raw());
  }
  // evaluator over a context whose keys were imported (BinFHEContext::ImportKeys): no key generation, and the context may hold no
  // secret key.  Inputs and outputs are then ciphertexts: SetInput(ciphertexts) and ClockCiphertexts().
  explicit Circuit(const lbcrypto::BinFHEContext &context) : cc(context) {
    gep.cc = cc;
    h = bfhe_circuit_create(cc.raw());
  }
  ~Circuit() { bfhe_circuit_destroy(h); }
  Circuit(const Circuit &) = delete;
  Circuit &operator=(const Circuit &) = delete;

  bool ReadFile(std::string cktName) {
    std::cout << "Loading circuit description " << cktName << std::endl;
    return ok(bfhe_circuit_read_file(h, cktName.c_str()));
  }
  bool ReadBristol(std::string cktName, bool new_format = false) { return ok(bfhe_circuit_read_bristol(h, cktName.c_str(), new_format)); }
  void Reset() {
    plaintext_flag = encrypted_flag = verify_flag = false; // src/circuit.cpp:378-381
    push_flags();
    ok(bfhe_circuit_reset(h));
  }
  void SetInput(Inputs input, bool verbose = false) {
    std::vector<uint8_t> flat;
    for (auto &bus : input) {
      if (verbose) std::cout << "setting input size " << bus.size() << std::endl;
      for (auto b : bus) flat.push_back((uint8_t)b);
    }
    ok(bfhe_circuit_set_input(h, flat.data(), flat.size(), input_seed ? input_seed++ : 0));
  }
  // SetInput on ciphertexts (bfhe_circuit_set_input_ct): one ciphertext per input bit, buses in SetInput's order.  Needs encrypted
  // mode and evaluation keys only; throws std::runtime_error on failure (a ciphertext word >= q, wrong count, wrong mode).
  void SetInput(const std::vector<std::vector<lbcrypto::LWECiphertext>> &input) {
    const size_t st = cc.params().ct_stride;
    std::vector<uint32_t> rows;
    for (auto &bus : input)
      for (auto &ct : bus) {
        if (!ct || ct->row.size() != st) throw std::runtime_error("SetInput: ciphertext is not a row of ct_stride words");
        rows.insert(rows.end(), ct->row.begin(), ct->row.end());
      }
    check(bfhe_circuit_set_input_ct(h, rows.data(), rows.size() / st, 0));
  }
  // SetInput from a BFHECTS1 blob (BinFHEContext::EncryptCompact, buses concatenated in SetInput's order): the masks are generated on
  // the GPU.  Evaluation keys only; throws std::runtime_error on failure (a malformed blob, wrong count, wrong mode).
  void SetInputCompact(const std::vector<uint8_t> &blob) { check(bfhe_circuit_set_input_compact(h, blob.data(), blob.size())); }
  void setPlaintext(bool f) { plaintext_flag = f; push_flags(); }
  bool getPlaintext() const { return plaintext_flag; }
  void setEncrypted(bool f) { encrypted_flag = f; push_flags(); }
  bool getEncrypted() const { return encrypted_flag; }
  void setVerify(bool f) { // forces both other modes on, src/circuit.cpp:833-840
    verify_flag = f;
    if (f) plaintext_flag = encrypted_flag = true;
    push_flags();
  }
  bool getVerify() const { return verify_flag; }
  Outputs Clock() {
    uint32_t nout = 0;
    bfhe_circuit_info(h, nullptr, nullptr, &nout, nullptr, nullptr, nullptr, nullptr);
    std::vector<uint8_t> out(nout), pout(nout);
    if (!ok(bfhe_circuit_clock(h, out.data(), out.size(), pout.data()))) std::exit(-1); // "done ckt clocked! should reset"
    double dev = 0, host = 0;
    uint64_t bad = 0;
    bfhe_circuit_stats(h, &dev, &host, &bad);
    std::cout << std::endl << "### Total time " << (unsigned)host << " msec" << std::endl; // src/circuit.cpp:565-566
    if (verify_flag && bad) std::cerr << bad << " wire(s) failed gate-by-gate verification" << std::endl;
    Outputs o(1);
    const std::vector<uint8_t> &src = encrypted_flag ? out : pout;
    o[0].assign(src.begin(), src.end());
    plainOut.assign(1, std::vector<unsigned int>(pout.begin(), pout.end()));
    return o;
  }
  // Clock with the outputs left encrypted (bfhe_circuit_clock_ct): one ciphertext per output bit; needs no secret key
  std::vector<lbcrypto::LWECiphertext> ClockCiphertexts() {
    uint32_t nout = 0;
    bfhe_circuit_info(h, nullptr, nullptr, &nout, nullptr, nullptr, nullptr, nullptr);
    const size_t st = cc.params().ct_stride;
    std::vector<uint32_t> rows((size_t)nout * st);
    check(bfhe_circuit_clock_ct(h, rows.data(), nout, 0));
    std::vector<lbcrypto::LWECiphertext> out(nout);
    for (uint32_t b = 0; b < nout; b++) {
      out[b] = std::make_shared<lbcrypto::LWECiphertextImpl>();
      out[b]->row.assign(rows.begin() + (size_t)b * st, rows.begin() + (size_t)(b + 1) * st);
    }
    return out;
  }
  void dumpGateCount() {
    uint32_t i, o, a, r, x, n;
    bfhe_circuit_dump_gate_count(h, &i, &o, &a, &r, &x, &n);
    // the reference's wording and order, src/circuit.cpp:866-873
    std::cout << "Number of input gates " << i << std::endl << "Number of output gates " << o << std::endl << "Number of not gates " << n << std::endl
              << "Number of and gates " << a << std::endl << "Number of or gates " << r << std::endl << "Number of xor gates " << x << std::endl;
  }
  void dumpNetList() { std::cout << dump_text(0); } // src/circuit.cpp:844-855
  void dumpGates() { std::cout << dump_text(1); }   // src/circuit.cpp:856-865
  uint64_t verifyMismatches() const {
    uint64_t bad = 0;
    bfhe_circuit_stats(h, nullptr, nullptr, &bad);
    return bad;
  }
  bfhe_circuit *raw() { return h; }
  Outputs plainOut;

private:
  std::string dump_text(int what) {
    size_t need = 0;
    if (bfhe_circuit_dump_text(h, what, nullptr, 0, &need) != BFHE_OK) return std::string();
    std::string s(need + 1, '\0');
    bfhe_circuit_dump_text(h, what, &s[0], s.size(), &need);
    s.resize(need);
    return s;
  }
  static void check(int rc) {
    if (rc != BFHE_OK) throw std::runtime_error(bfhe_last_error());
  }
  bool ok(int rc) {
    if (rc != BFHE_OK) std::cerr << bfhe_last_error() << std::endl;
    return rc == BFHE_OK;
  }
  void push_flags() { bfhe_circuit_set_flags(h, plaintext_flag, encrypted_flag, verify_flag); }
  lbcrypto::BinFHEContext cc;
  lbcrypto::LWEPrivateKey sk;
  bool plaintext_flag = false, encrypted_flag = false, verify_flag = false;
  GateEvalParams gep;
  bfhe_circuit *h = nullptr;
  uint64_t input_seed = 0;
};
