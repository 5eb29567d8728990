// binfhecontext.h -- source-level shim with the exact lbcrypto names the reference uses, over the C ABI.
//
// The reference includes OpenFHE's "binfhecontext.h" (src/wire.h:39, src/utils.h:43) and touches only:
// GenerateBinFHEContext (src/circuit.cpp:88), KeyGen (:90), BTKeyGen (:91), Encrypt (:506), Decrypt (:800),
// EvalNOT (src/gate.cpp:112), EvalBinGate (src/gate.cpp:133), the enums BINFHE_PARAMSET / BINFHE_METHOD / BINGATE
// (src/utils.cpp:165-190, src/gate.cpp:133,172) and the types LWECiphertext / LWEPrivateKey / LWEPlaintext
// (src/wire.h:46, src/circuit.h:75-76, src/gate.cpp:71).  Pointing the reference's include path at this directory
// makes gate.cpp-style code compile against the B200 engine: every single-gate call is a batch of one.
// Header-only; link with libbfhe_b200.so.
#pragma once
#include "../../include/bfhe.h"
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace lbcrypto {

// same order as OpenFHE 1.0.x binfhe-constants.h, so integer values agree with include/bfhe.h
enum BINFHE_PARAMSET { TOY, MEDIUM, STD128_AP, STD128_APOPT, STD128, STD128_OPT, STD192, STD192_OPT, STD256, STD256_OPT };
enum BINFHE_METHOD { AP, GINX };
enum BINGATE { OR, AND, NOR, NAND, XOR_FAST, XNOR_FAST, XOR, XNOR };
enum BINFHE_OUTPUT { FRESH, BOOTSTRAPPED };

using LWEPlaintext = int64_t;

class config_error : public std::runtime_error {
public:
  explicit config_error(const std::string &m) : std::runtime_error(m) {}
};

class LWECiphertextImpl {
public:
  std::vector<uint32_t> row; // ct_stride words: a_0..a_{n-1}, b, padding
};
using LWECiphertext = std::shared_ptr<LWECiphertextImpl>;
using ConstLWECiphertext = std::shared_ptr<const LWECiphertextImpl>;

class LWEPrivateKeyImpl {}; // the secret key stays inside the engine context; this is a capability token
using LWEPrivateKey = std::shared_ptr<LWEPrivateKeyImpl>;
using ConstLWEPrivateKey = std::shared_ptr<const LWEPrivateKeyImpl>;

class BinFHEContext {
public:
  // copies share the key material, like gep.cc = cc in src/circuit.cpp:93-94
  void GenerateBinFHEContext(BINFHE_PARAMSET set, BINFHE_METHOD method = GINX, int device = 0) {
    bfhe_ctx *c = bfhe_create((int)set, (int)method, device);
    if (!c) throw config_error(bfhe_last_error());
    m_ctx.reset(c, bfhe_destroy);
    bfhe_get_params(c, &m_p);
  }
  // seed == 0 (default): keys, masks and noise are drawn from a ChaCha20 stream keyed with 256 bits of OS entropy, like OpenFHE's
  // self-seeding PRNG.  A non-zero seed gives reproducible (and therefore NOT confidential) material for tests and parity runs.
  LWEPrivateKey KeyGen(uint64_t seed = 0) const {
    check(bfhe_keygen(raw(), seed));
    return std::make_shared<LWEPrivateKeyImpl>();
  }
  void BTKeyGen(ConstLWEPrivateKey, uint64_t seed = 0) { check(bfhe_btkeygen(raw(), seed)); }
  // BTKeyGen with every public mask expanded from a fresh mask seed, so that ExportKeys(..., true) ships seed and bodies only
  void BTKeyGenCompact(ConstLWEPrivateKey, uint64_t seed = 0) { check(bfhe_btkeygen_compact(raw(), seed)); }
  LWECiphertext Encrypt(ConstLWEPrivateKey, const LWEPlaintext &m, BINFHE_OUTPUT output = BOOTSTRAPPED) const {
    auto ct = std::make_shared<LWECiphertextImpl>();
    ct->row.resize(m_p.ct_stride);
    uint8_t bit = (uint8_t)(m & 3);
    check(bfhe_encrypt(raw(), &bit, 1, next_seed(), ct->row.data()));
    if (output == FRESH || !m_bootstrap_inputs) return ct;
    return Bootstrap(ct); // OpenFHE's default output = BOOTSTRAPPED
  }
  void Decrypt(ConstLWEPrivateKey, ConstLWECiphertext ct, LWEPlaintext *result) const {
    uint8_t r = 0;
    check(bfhe_decrypt(raw(), ct->row.data(), 1, &r));
    *result = r;
  }
  LWECiphertext EvalNOT(ConstLWECiphertext ct) const { return one_gate(BFHE_BOOTSTRAP + 1, ct, ct); }
  LWECiphertext EvalBinGate(const BINGATE gate, ConstLWECiphertext ct1, ConstLWECiphertext ct2) const {
    if (ct1 == ct2) throw config_error("ERROR: Please only use independent ciphertexts as inputs.");
    return one_gate((uint32_t)gate, ct1, ct2);
  }
  LWECiphertext Bootstrap(ConstLWECiphertext ct) const { return one_gate(BFHE_BOOTSTRAP, ct, ct); }

  // the key blob of bfhe_export_keys (include/bfhe.h): without the secret key it is what an evaluator needs, and all it gets.
  // compact: the BFHEKEY2 blob of bfhe_export_keys_compact (keys from BTKeyGenCompact or a compact import only)
  std::vector<uint8_t> ExportKeys(bool include_sk, bool compact = false) const {
    std::vector<uint8_t> blob(compact ? bfhe_keyblob_compact_size(raw()) : bfhe_keyblob_size(raw()));
    check(compact ? bfhe_export_keys_compact(raw(), blob.data(), blob.size(), include_sk ? 1 : 0)
                  : bfhe_export_keys(raw(), blob.data(), blob.size(), include_sk ? 1 : 0));
    return blob;
  }
  // either blob
  void ImportKeys(const std::vector<uint8_t> &blob) { check(bfhe_import_keys(raw(), blob.data(), blob.size())); }

  bfhe_ctx *raw() const {
    if (!m_ctx) throw config_error("GenerateBinFHEContext has not been called");
    return m_ctx.get();
  }
  const bfhe_params &params() const { return m_p; }
  void SetBootstrapFreshEncryptions(bool on) { m_bootstrap_inputs = on; }
  void SetEncryptionSeed(uint64_t seed) { m_seed = seed; }

private:
  static void check(int rc) {
    if (rc == BFHE_ERR_ALIAS) throw config_error(bfhe_last_error());
    if (rc != BFHE_OK) throw std::runtime_error(bfhe_last_error());
  }
  // 0 = OS entropy for every encryption (default); SetEncryptionSeed(s != 0) = reproducible sequence for tests
  uint64_t next_seed() const {
    if (m_seed == 0) return 0;
    m_seed = m_seed * 6364136223846793005ull + 1442695040888963407ull;
    return m_seed ? m_seed : 1;
  }
  LWECiphertext one_gate(uint32_t op, ConstLWECiphertext a, ConstLWECiphertext b) const {
    const size_t st = m_p.ct_stride;
    auto out = std::make_shared<LWECiphertextImpl>();
    out->row.resize(st);
    if (op == BFHE_BOOTSTRAP + 1) { // EvalNOT: no bootstrap, device kernel on a 2-row slab
      uint32_t *slab = nullptr;
      check(bfhe_slab_alloc(raw(), 2, &slab));
      const uint32_t in = 0, o = 1;
      int rc = bfhe_slab_upload(raw(), slab, 0, a->row.data(), 1);
      if (!rc) rc = bfhe_eval_not_batch(raw(), slab, &in, &o, 1);
      if (!rc) rc = bfhe_slab_download(raw(), slab, 1, out->row.data(), 1);
      bfhe_slab_free(raw(), slab);
      check(rc);
      return out;
    }
    std::vector<uint32_t> in(2 * st);
    std::copy(a->row.begin(), a->row.end(), in.begin());
    std::copy(b->row.begin(), b->row.end(), in.begin() + st);
    bfhe_gate g{op, 0, op == BFHE_BOOTSTRAP ? 0u : 1u, 2};
    check(bfhe_eval_bingate_host(raw(), &g, 1, in.data(), 2, out->row.data(), 1));
    return out;
  }
  std::shared_ptr<bfhe_ctx> m_ctx;
  bfhe_params m_p{};
  bool m_bootstrap_inputs = true;
  mutable uint64_t m_seed = 0;
};

} // namespace lbcrypto
