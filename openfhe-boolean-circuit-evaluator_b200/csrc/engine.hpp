// engine.hpp -- internal definition of bfhe_ctx (the C ABI in include/bfhe.h only sees the opaque pointer).
#pragma once
#include "../../include/bfhe.h"
#include "common.hpp"
#include "hostmath.hpp"
#include <cuda_runtime.h>
#include <mutex>
#include <string>
#include <vector>

namespace bfhe {

void set_error(const std::string &msg);
int cuda_fail(cudaError_t e, const char *what);
#define BFHE_CUDA(call)                                                                                                \
  do {                                                                                                                 \
    cudaError_t _e = (call);                                                                                           \
    if (_e != cudaSuccess) return ::bfhe::cuda_fail(_e, #call);                                                        \
  } while (0)

struct ProfSpan {
  cudaEvent_t a, b;
  int kernel;
};

} // namespace bfhe

struct bfhe_ctx {
  bfhe_params p{};
  bfhe::DevConst P{};
  int device = -1;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  bfhe::u64 psi = 0;
  bfhe::HostNtt hntt;

  // host key material (canonical forms)
  std::vector<bfhe::i32> sk;
  std::vector<bfhe::i32> z; // RLWE key, only between keygen and btkeygen
  bool has_sk = false, has_bt = false;
  bool ofhe_have_bk = false, ofhe_have_ksk = false; // halves of the bootstrapping key imported from OpenFHE JSON (host/openfhe_json.cpp)
  std::vector<bfhe::u32> bk_coef;
  std::vector<bfhe::u8> ksk; // [N][baseKS][dKS][n+1], ksk_elem_bytes each
  // keys whose masks are the expansion of a public mask seed (bfhe_btkeygen_compact, BFHEKEY2 import).  A device context that imported
  // BFHEKEY2 keeps only the bodies here (bk_coef / ksk empty); the full forms are expanded on the host when an export asks for them.
  bool has_mask_seed = false;
  bfhe::MaskKey mask_seed{};
  std::vector<bfhe::u32> bk_body; // column-1 polynomials of bk_coef, BFHEKEY1 order
  std::vector<bfhe::u8> ksk_body; // [N][baseKS][dKS], ksk_elem_bytes each
  bfhe::u32 ksk_elem_bytes = 4;
  bfhe::u64 bk_words = 0, ksk_elems = 0;

  // device key material
  bfhe::u32 *d_bk = nullptr, *d_twl = nullptr, *d_psiM = nullptr;
  void *d_ksk = nullptr;
  bfhe::u32 *d_bk4 = nullptr, *d_tw2 = nullptr, *d_F = nullptr; // 2-CTA cluster kernel (kernels_v2.cu)
  bfhe::u32 *d_bkx = nullptr, *d_twx = nullptr; // slot-sliced cluster kernel (kernels_cl.cu)
  bfhe::u32 *d_bkf = nullptr; // GINX throughput kernel at the STD128_OPT shape: top digit folded into the key (kernels.cu bk_fold_kernel)
  bfhe::V2Bufs v2{};
  bool dev_keys = false;

  // per-call scratch
  static constexpr size_t CHUNK = 32768; // upper bound of gates per blind-rotation launch (buffer sizes)
  size_t chunk = CHUNK;                  // actual launch size: largest multiple of one full wave (4 gates x SM count) <= CHUNK
  bfhe::DevGate *d_gates = nullptr;      // CHUNK entries (buffer 0)
  bfhe::DevGate *d_gates_b = nullptr;    // buffer 1: key switch of chunk k overlaps blind rotation of chunk k+1
  bfhe::u32 *d_ext_b = nullptr;
  cudaStream_t ks_stream = nullptr;
  cudaEvent_t ev_br[2] = {nullptr, nullptr}, ev_ks[2] = {nullptr, nullptr};
  bfhe::DevGate *h_gates[2] = {nullptr, nullptr}; // pinned staging
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  int stage_next = 0;
  bfhe::u32 *d_ext = nullptr;            // CHUNK * (N+4)
  bfhe::u32 *d_tmp = nullptr;            // composite-gate temporaries
  size_t tmp_rows = 0;
  const bfhe::u32 **d_ptr_in = nullptr;  // EvalNOT pointer lists
  bfhe::u32 **d_ptr_out = nullptr;
  size_t ptr_cap = 0;
  bfhe::u32 *e2e_slab = nullptr;
  size_t e2e_rows = 0;
  int force_g = 0; // test hook: gates per CTA
  // measured cost (ms) of one wave (blind rotation + key switch) in the 4-CTA / 2-CTA cluster, one-gate-per-SM and four-gates-per-SM
  // forms on this device with this key set (host/circuit.cpp probe_costs)
  double form_cost_ms[4] = {0, 0, 0, 0};
  bool form_cost_measured = false;

  bool profiling = false;
  std::vector<bfhe::ProfSpan> spans;
  std::mutex mtx; // the reference calls EvalBinGate concurrently from OpenMP tasks (src/circuit.cpp:698-710)
};

namespace bfhe {
// run one list of single-bootstrap gates (device pointers already resolved) through blind rotation + key switch
int run_gate_list(bfhe_ctx *c, const DevGate *host_list, size_t count, u32 *acc_dbg_host);
int ensure_device_keys(bfhe_ctx *c);
// full coefficient-form BK / [N][baseKS][dKS][n+1] KSK of the context's keys: bk_coef / ksk, or expanded from the mask seed and the bodies
void host_full_bk(const bfhe_ctx *c, u32 *out);
void host_full_ksk(const bfhe_ctx *c, u8 *out);
// the keys stop being the expansion of a mask seed (some of them are replaced): full host forms, no seed, no bodies
void forget_mask_seed(bfhe_ctx *c);
// EvalNOT of in[i] into out[i] through the context's pointer buffers (low bit of in[i] set: plain copy); caller holds c->mtx
int not_ptr_batch(bfhe_ctx *c, const std::vector<const u32 *> &in, const std::vector<u32 *> &out);
} // namespace bfhe
