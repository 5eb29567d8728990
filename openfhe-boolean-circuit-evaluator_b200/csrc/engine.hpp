// engine.hpp -- internal definition of bfhe_ctx (the C ABI in include/bfhe.h only sees the opaque pointer).
#pragma once
#include "../../include/bfhe.h"
#include "common.hpp"
#include "hostmath.hpp"
#include <algorithm>
#include <condition_variable>
#include <cuda_runtime.h>
#include <deque>
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

// Owner of one device allocation (Pinned: page-locked host memory), released on destruction.  Allocate, reserve and release with the
// owning context's device current.
template <typename T, bool Pinned = false> class DevBuf {
public:
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept {
    if (this != &o) { reset(); p_ = o.p_; n_ = o.n_; o.p_ = nullptr; o.n_ = 0; }
    return *this;
  }
  ~DevBuf() { reset(); }
  // a fresh buffer of `count` elements; the old one is released first
  cudaError_t alloc(size_t count) {
    reset();
    void *p = nullptr;
    cudaError_t e = Pinned ? cudaMallocHost(&p, count * sizeof(T)) : cudaMalloc(&p, count * sizeof(T));
    if (e != cudaSuccess) return e;
    p_ = static_cast<T *>(p);
    n_ = count;
    return cudaSuccess;
  }
  // grow-only: a larger buffer once `stream` is done with the old one (work queued on it may still read or write it)
  cudaError_t reserve(size_t count, cudaStream_t stream) {
    if (count <= n_) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(stream);
    return e != cudaSuccess ? e : alloc(count);
  }
  void reset() {
    if (p_) Pinned ? cudaFreeHost(p_) : cudaFree(p_);
    p_ = nullptr;
    n_ = 0;
  }
  T *get() const { return p_; }
  size_t size() const { return n_; }

private:
  T *p_ = nullptr;
  size_t n_ = 0;
};

// dst := a device copy of src (at least one element, so that an empty list still has a valid address)
template <typename T> cudaError_t upload(DevBuf<T> &dst, const std::vector<T> &src) {
  cudaError_t e = dst.alloc(std::max<size_t>(src.size(), 1));
  return e != cudaSuccess ? e : cudaMemcpy(dst.get(), src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice);
}

// owner of a local cudaEvent_t (timing enabled)
struct DevEvent {
  cudaEvent_t e = nullptr;
  DevEvent() = default;
  DevEvent(const DevEvent &) = delete;
  DevEvent &operator=(const DevEvent &) = delete;
  ~DevEvent() { if (e) cudaEventDestroy(e); }
  cudaError_t create() { return cudaEventCreate(&e); }
};

// cost (ms) of one wave (blind rotation + key switch) in the kernel forms the circuit planner weighs: these B200 defaults, or measured once
// per context on its device with its key set (host/circuit.cpp probe_costs)
struct WaveCosts {
  double cl4 = 1.05, cl2 = 1.55, lat = 2.36, thr = 5.85;
};

struct ProfSpan {
  cudaEvent_t a, b;
  int kernel;
};

// one bfhe_eval_bingate_host call waiting to be combined with concurrent ones (engine.cu, "combining"); lives on the caller's stack
struct HostGateReq {
  const bfhe_gate *gates;
  size_t count;
  const u32 *in_host;
  size_t in_rows;
  u32 *out_host;
  size_t out_rows;
  enum { QUEUED, LEAD, DONE } state = QUEUED;
  int rc = BFHE_OK;
  std::string err;
  std::condition_variable cv;
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

  // device key material: tables made by bfhe_create, key copies by upload_keys; handed to the kernels as keys()
  bfhe::DevBuf<bfhe::u32> d_twl, d_psiM, d_tw2, d_F, d_twx;
  bfhe::DevBuf<bfhe::u32> d_bk, d_bkf, d_bk4, d_bkx;
  bfhe::DevBuf<bfhe::u8> d_ksk;
  bool dev_keys = false;
  bfhe::DevKeys keys() const {
    return {d_bk.get(), d_bkf.get(), d_bk4.get(), d_bkx.get(), d_twl.get(), d_psiM.get(), d_tw2.get(), d_F.get(), d_twx.get(), d_ksk.get(),
            (int)ksk_elem_bytes};
  }

  // per-call scratch
  static constexpr size_t CHUNK = 32768; // upper bound of gates per blind-rotation launch (buffer sizes)
  size_t chunk = CHUNK;                  // actual launch size: largest multiple of one full wave (4 gates x SM count) <= CHUNK
  bfhe::DevBuf<bfhe::DevGate> d_gates;   // CHUNK entries (buffer 0)
  bfhe::DevBuf<bfhe::DevGate> d_gates_b; // buffer 1: key switch of chunk k overlaps blind rotation of chunk k+1
  bfhe::DevBuf<bfhe::u32> d_ext, d_ext_b; // CHUNK * (N+4) each
  cudaStream_t ks_stream = nullptr;
  cudaEvent_t ev_br[2] = {nullptr, nullptr}, ev_ks[2] = {nullptr, nullptr};
  bfhe::DevBuf<bfhe::DevGate, true> h_gates[2]; // pinned staging
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  int stage_next = 0;
  bfhe::DevBuf<bfhe::u32> d_tmp;         // composite-gate temporaries; the bodies of a compact ciphertext blob (expand_ct_rows)
  bfhe::DevBuf<const bfhe::u32 *> d_ptr_in; // EvalNOT pointer lists
  bfhe::DevBuf<bfhe::u32 *> d_ptr_out;
  bfhe::DevBuf<bfhe::u32> e2e_slab;      // bfhe_eval_bingate_host staging
  int force_g = 0; // test hook: the bfhe::Form every launch uses (AUTO: the launch's own choice)
  bfhe::WaveCosts form_costs;
  bool form_cost_measured = false;

  bool profiling = false;
  std::vector<bfhe::ProfSpan> spans;
  std::mutex mtx; // the reference calls EvalBinGate concurrently from OpenMP tasks (src/circuit.cpp:698-710)

  // combining of concurrent bfhe_eval_bingate_host calls: at most one batch in flight; calls arriving meanwhile queue (FIFO) and the
  // front one leads the next batch.  q_mtx guards the queue only; the leader takes mtx for the device work.
  std::mutex q_mtx;
  std::deque<bfhe::HostGateReq *> q;
  bool q_busy = false; // a batch is in flight (a leader has been chosen)
  bool q_hold = false; // test hook bfhe_dbg_hold_batches: nothing launches
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
// a BFHECTS1 blob of compact fresh ciphertexts (include/bfhe.h) that passed every check of read_ct_blob; bodies points into the blob
struct CtBlob {
  MaskKey seed{};
  size_t count = 0;
  const u8 *bodies = nullptr; // count little-endian uint16, each below q
};
// the host checks of a BFHECTS1 blob against this context: BFHE_ERR_FORMAT naming what failed
int read_ct_blob(const bfhe_ctx *c, const void *blob, size_t len, CtBlob &out);
// enqueue on c->stream: the blob's count full rows into d_rows (device memory, ct_stride words per row, 16-byte aligned).  Caller holds
// c->mtx with the context's device current, and keeps `wide` (the bodies widened to u32, the copy's source) until the stream is past it.
int expand_ct_rows(bfhe_ctx *c, const CtBlob &b, u32 *d_rows, std::vector<u32> &wide);
// BFHE_ERR_ARG, "<what> is not memory of device d", unless p is device (or managed) memory of the context's device
int check_device_buffer(const bfhe_ctx *c, const void *p, const char *what);
} // namespace bfhe
