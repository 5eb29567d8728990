// engine.cu -- C-ABI implementation (include/bfhe.h): context, keys, host LWE, batch launches.
//
// Mirrors the lbcrypto::BinFHEContext surface the reference uses (src/circuit.cpp:88-91,506,800;
// src/gate.cpp:112,133,172).  Host side: parameters, key generation, fresh encryption, decryption
// (all one-off or per-I/O-bit work).  Device side: everything per gate.  There is no CPU fallback for
// EvalBinGate / Bootstrap / EvalNOT: without a CUDA device those calls fail with BFHE_ERR_CUDA.
#include "engine.hpp"
#include "device.cuh"
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <omp.h>

using namespace bfhe;

namespace bfhe {
static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
int cuda_fail(cudaError_t e, const char *what) {
  set_error(std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what);
  return BFHE_ERR_CUDA;
}
} // namespace bfhe

extern "C" const char *bfhe_last_error(void) { return g_err.c_str(); }

static constexpr double SIGMA = 3.19;
static const GaussTable &gauss_table() {
  static const GaussTable t(SIGMA);
  return t;
}
static int make_seed_key(uint64_t seed, SeedKey &key) {
  if (!SeedKey::make(seed, key)) { set_error("cannot read OS entropy (getrandom and /dev/urandom both failed)"); return BFHE_ERR_IO; }
  return BFHE_OK;
}

// ---- key blob header (documented in include/bfhe.h / DESIGN.md) ----
struct KeyBlobHeader {
  char magic[8];
  u32 version, paramset, method, n, N, q;
  u32 baseKS, dKS, baseG, dG, baseR, dR;
  u32 has_sk, ksk_elem_bytes;
  u64 Q, qKS, bk_words, ksk_elems;
  u64 reserved[4];
};
static size_t pad8(size_t x) { return (x + 7) & ~(size_t)7; }

// -------------------------------------------------------------------------------------------------
// context
// -------------------------------------------------------------------------------------------------
static u32 shoup32(u64 w, u64 Q) { return (u32)((w << 32) / Q); }

// the device side of a new context: the kernels' tables, the per-call buffers, the side stream and the events
static int init_device(bfhe_ctx *c) {
  const u32 N = c->p.N;
  const u64 Q = c->p.Q;
  const int ap = c->p.method == BFHE_AP;
  // per-lane twiddle tables of the narrow pass: [chunk][lane][4]; entry p = groups + gi is
  // psi^bitrev(groups*(32 + lane) + gi)  (see kernels.cu ct_pass)
  const u32 E = N / 32;
  std::vector<u32> tl(4 * (size_t)N, 0);
  for (u32 lane = 0; lane < 32; lane++)
    for (u32 pp = 1; pp < E; pp++) {
      u32 groups = 1;
      while (groups * 2 <= pp) groups *= 2;
      u32 gi = pp - groups, idx = groups * (32 + lane) + gi;
      size_t off = ((size_t)(pp / 4) * 32 + lane) * 4 + (pp % 4);
      tl[off] = c->hntt.tw[idx]; tl[N + off] = shoup32(c->hntt.tw[idx], Q);
      tl[2 * N + off] = c->hntt.itw[idx]; tl[3 * N + off] = shoup32(c->hntt.itw[idx], Q);
    }
  std::vector<u32> psiM(2 * (size_t)N);
  u64 cur = (1ull << 32) % Q; // Montgomery form of psi^0
  for (u32 k = 0; k < 2 * N; k++) { psiM[k] = (u32)cur; cur = mulmod64(cur, c->psi, Q); }
  BFHE_CUDA(upload(c->d_twl, tl));
  BFHE_CUDA(upload(c->d_psiM, psiM));
  BFHE_CUDA(c->d_gates.alloc(bfhe_ctx::CHUNK));
  BFHE_CUDA(c->d_ext.alloc(bfhe_ctx::CHUNK * (size_t)(N + 4)));
  BFHE_CUDA(c->d_gates_b.alloc(bfhe_ctx::CHUNK));
  BFHE_CUDA(c->d_ext_b.alloc(bfhe_ctx::CHUNK * (size_t)(N + 4)));
  BFHE_CUDA(cudaStreamCreateWithFlags(&c->ks_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    BFHE_CUDA(cudaEventCreateWithFlags(&c->ev_br[i], cudaEventDisableTiming));
    BFHE_CUDA(cudaEventCreateWithFlags(&c->ev_ks[i], cudaEventDisableTiming));
    BFHE_CUDA(c->h_gates[i].alloc(bfhe_ctx::CHUNK));
    BFHE_CUDA(cudaEventCreateWithFlags(&c->stage_ev[i], cudaEventDisableTiming));
  }
  if (form_supported(c->P, ap, Form::CL2)) { // tables of the 2-CTA cluster form (F is read by the GINX 4-CTA form too)
    std::vector<u32> t2(4 * (size_t)N), F(2 * (size_t)N);
    for (u32 k = 0; k < N; k++) { // natural order, last stage de-interleaved (kernels_v2.cu load_tw_narrow)
      u32 d = k;
      if (k >= N / 2) { const u32 i = k - N / 2, t = i >> 3, j = i & 7; d = N / 2 + (N / 4) * (j >> 2) + 4 * t + (j & 3); }
      t2[d] = c->hntt.tw[k]; t2[N + d] = shoup32(c->hntt.tw[k], Q);
      t2[2 * N + d] = c->hntt.itw[k]; t2[3 * N + d] = shoup32(c->hntt.itw[k], Q);
    }
    const u64 oneM = (1ull << 32) % Q;
    for (u32 k = 0; k < 2 * N; k++) // (psi^k - 1) in Montgomery form
      F[f_index(k)] = (u32)((psiM[k] + Q - oneM) % Q);
    BFHE_CUDA(upload(c->d_tw2, t2));
    BFHE_CUDA(upload(c->d_F, F));
  }
  if (form_supported(c->P, ap, Form::CL4)) { // per-rank twiddle blocks of the slot-sliced cluster kernel (layout: kernels_cl.cu TWF / TWI)
    // CTA k runs the sub-transform of block k (in-place positions 256 k + i, i < 256) as: pass A (lane holds i = lane + 32 m),
    // pass B (lane = 4 blk + q holds i = 32 blk + q + 4 m), pass C (lane holds i = 8 lane + j).  A stage with G groups uses tw[G + group],
    // group = position / (N / G) -- the table order of HostNtt (tw[k] = psi^bitrev(k)).  The inverse runs the five narrowest stages
    // as shuffles in the external-product threads (slot t = position t) and the three widest in pass-A layout.
    const size_t TWF = 8 + 2 * 256, TWI = 8 + 5 * 256, TWR = 2 * TWF + 2 * TWI;
    std::vector<u32> tx(clx_tw_words(), 0);
    for (u32 k = 0; k < 4; k++) {
      u32 *fw = tx.data() + (size_t)k * TWR, *fws = fw + TWF, *iw = fw + 2 * TWF, *iws = iw + TWI;
      auto putf = [&](size_t off, u32 idx) { fw[off] = c->hntt.tw[idx]; fws[off] = shoup32(c->hntt.tw[idx], Q); };
      auto puti = [&](size_t off, u32 idx) { iw[off] = c->hntt.itw[idx]; iws[off] = shoup32(c->hntt.itw[idx], Q); };
      putf(1, 4 + k); puti(1, 4 + k);
      for (u32 g = 0; g < 2; g++) { putf(2 + g, 8 + 2 * k + g); puti(2 + g, 8 + 2 * k + g); }
      for (u32 g = 0; g < 4; g++) { putf(4 + g, 16 + 4 * k + g); puti(4 + g, 16 + 4 * k + g); }
      for (u32 lane = 0; lane < 32; lane++) {
        const u32 blk = lane >> 2;
        auto at = [&](int s, u32 e) { return 8 + 256 * (size_t)s + ((size_t)(e >> 2) * 32 + lane) * 4 + (e & 3); }; // [chunk][lane][4]
        putf(at(0, 1), 32 + 8 * k + blk);
        for (u32 g = 0; g < 2; g++) putf(at(0, 2 + g), 64 + 16 * k + 2 * blk + g);
        for (u32 g = 0; g < 4; g++) putf(at(0, 4 + g), 128 + 32 * k + 4 * blk + g);
        for (u32 g = 0; g < 2; g++) putf(at(1, 2 + g), 256 + 64 * k + 2 * lane + g);
        for (u32 g = 0; g < 4; g++) putf(at(1, 4 + g), 512 + 128 * k + 4 * lane + g);
      }
      for (u32 s5 = 0; s5 < 5; s5++)
        for (u32 t = 0; t < 256; t++) puti(8 + 256 * (size_t)s5 + t, (512u >> s5) + ((256 * k + t) >> (s5 + 1)));
    }
    BFHE_CUDA(upload(c->d_twx, tx));
  }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
  c->chunk = std::max<size_t>(1, bfhe_ctx::CHUNK / (4 * (size_t)sms)) * 4 * (size_t)sms; // whole waves of 4-gate CTAs
  if (c->chunk > bfhe_ctx::CHUNK) c->chunk = bfhe_ctx::CHUNK;
  return BFHE_OK;
}

extern "C" bfhe_ctx *bfhe_create(int paramset, int method, int device) {
  bfhe_params p{};
  p.paramset = paramset;
  p.method = method;
  // GenerateBinFHEContext parameter table (OpenFHE 1.0.x binfhecontext.cpp; SURVEY App. C.1)
  if (paramset == BFHE_TOY) {
    p.n = 64; p.N = 512; p.q = 512; p.Q = previous_prime(first_prime(27, 1024), 1024); p.qKS = p.Q;
    p.baseKS = 25; p.baseG = 1u << 9; p.baseR = 23;
  } else if (paramset == BFHE_STD128_OPT) {
    p.n = 502; p.N = 1024; p.q = 1024; p.Q = previous_prime(first_prime(27, 2048), 2048); p.qKS = 1u << 14;
    p.baseKS = 1u << 7; p.baseG = 1u << 7; p.baseR = 32;
  } else {
    set_error("unsupported parameter set (the reference accepts only TOY and STD128_OPT, src/circuit.cpp:69-78)");
    return nullptr;
  }
  if (method != BFHE_AP && method != BFHE_GINX) {
    set_error("unsupported method (the reference accepts only AP and GINX, src/circuit.cpp:79-86)");
    return nullptr;
  }
  p.dKS = (u32)std::ceil(std::log((double)p.qKS) / std::log((double)p.baseKS));
  p.dG = (u32)std::ceil(std::log((double)p.Q) / std::log((double)p.baseG));
  p.dR = (u32)std::ceil(std::log((double)p.q) / std::log((double)p.baseR));
  p.ct_words = p.n + 1;
  p.ct_stride = (p.ct_words + 3) & ~3u;
  if (!(p.Q > (1ull << 26) && p.Q < (1ull << 27))) {
    set_error("ring modulus outside (2^26, 2^27): the lazy-reduction ranges of the kernels assume 32Q < 2^32");
    return nullptr;
  }
  if ((2 * p.N / p.q) % 2 != 0) {
    set_error("2N/q must be even (the monomial-factor table of the external product holds even exponents only)");
    return nullptr;
  }
  if (p.Q != SOLINAS_Q) {
    set_error("kernels are specialised for Q = 2^27 - 2^11 + 1");
    return nullptr;
  }
  bfhe_ctx *c = new bfhe_ctx();
  c->p = p;
  c->device = device;
  const u32 N = p.N;
  const u64 Q = p.Q;
  c->psi = min_primitive_root(2 * (u64)N, Q);
  c->hntt.init(N, (u32)Q, c->psi);
  DevConst &P = c->P;
  P.Q = (u32)Q; P.Q2 = 2 * (u32)Q;
  { // -Q^-1 mod 2^32 by Newton iteration
    u32 inv = (u32)Q;
    for (int i = 0; i < 5; i++) inv *= 2 - (u32)Q * inv;
    P.qinv_neg = 0u - inv;
  }
  P.oneM = (u32)((1ull << 32) % Q);
  P.Q8 = (u32)(Q / 8 + 1);
  P.n = p.n; P.N = N; P.q = p.q; P.factor = 2 * N / p.q;
  P.qKS = (u32)p.qKS; P.baseKS = p.baseKS; P.dKS = p.dKS;
  P.baseR = p.baseR; P.dR = p.dR; P.dG = p.dG; P.logBG = ilog2_ceil(p.baseG);
  P.ct_stride = p.ct_stride;
  u64 ninv = powmod64(N, Q - 2, Q);
  P.ninv = (u32)ninv; P.ninvs = shoup32(ninv, Q);
  u64 nM = mulmod64(ninv, (1ull << 32) % Q, Q);
  P.nM = (u32)nM; P.nMs = shoup32(nM, Q);
  const u32 q = p.q; // RingGSWCryptoParams gate constants
  P.gate_const[BFHE_OR] = 5 * (q >> 3); P.gate_const[BFHE_AND] = 7 * (q >> 3); P.gate_const[BFHE_NOR] = q >> 3;
  P.gate_const[BFHE_NAND] = 3 * (q >> 3); P.gate_const[BFHE_XOR_FAST] = 5 * (q >> 3); P.gate_const[BFHE_XNOR_FAST] = q >> 3;
  P.gate_const[BFHE_XOR] = P.gate_const[BFHE_XNOR] = 0; P.gate_const[BFHE_BOOTSTRAP] = 7 * (q >> 3);
  for (int k = 0; k < 32; k++) {
    P.tw[k] = c->hntt.tw[k]; P.tws[k] = shoup32(P.tw[k], Q);
    P.itw[k] = c->hntt.itw[k]; P.itws[k] = shoup32(P.itw[k], Q);
  }
  c->bk_words = (method == BFHE_GINX) ? (u64)p.n * 2 * (2 * p.dG) * 2 * N : (u64)p.n * (p.baseR - 1) * p.dR * (2 * p.dG) * 2 * N;
  c->ksk_elem_bytes = p.qKS <= 65536 ? 2 : 4;
  c->ksk_elems = (u64)N * p.baseKS * p.dKS * (p.n + 1);

  if (device >= 0) {
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
      cuda_fail(e, "bfhe_create: no usable CUDA device (this engine has no CPU fallback)");
      delete c;
      return nullptr;
    }
    c->stream = c->own_stream;
    if (init_device(c)) {
      bfhe_destroy(c);
      return nullptr;
    }
  }
  return c;
}

extern "C" void bfhe_destroy(bfhe_ctx *c) {
  if (!c) return;
  if (c->device >= 0) {
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto &s : c->spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
    for (int i = 0; i < 2; i++) {
      if (c->ev_br[i]) cudaEventDestroy(c->ev_br[i]);
      if (c->ev_ks[i]) cudaEventDestroy(c->ev_ks[i]);
      if (c->stage_ev[i]) cudaEventDestroy(c->stage_ev[i]);
    }
    if (c->ks_stream) cudaStreamDestroy(c->ks_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
  }
  delete c; // the buffers' owners release them, with the context's device current
}

extern "C" int bfhe_get_params(const bfhe_ctx *c, bfhe_params *out) {
  if (!c || !out) return BFHE_ERR_ARG;
  *out = c->p;
  return BFHE_OK;
}
extern "C" int bfhe_set_stream(bfhe_ctx *c, void *s, int use_own) {
  if (!c || c->device < 0) return BFHE_ERR_STATE;
  c->stream = use_own ? c->own_stream : (cudaStream_t)s; // s == NULL is the legacy default stream, as everywhere in CUDA
  return BFHE_OK;
}
extern "C" int bfhe_sync(bfhe_ctx *c) {
  if (!c || c->device < 0) { set_error("no device attached"); return BFHE_ERR_CUDA; }
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  return BFHE_OK;
}

// -------------------------------------------------------------------------------------------------
// key generation (host; one-off).  KeyGen: uniform ternary LWE key.  BTKeyGen: RLWE key z, KSK, BK.
// -------------------------------------------------------------------------------------------------
extern "C" int bfhe_keygen(bfhe_ctx *c, uint64_t seed) {
  if (!c) return BFHE_ERR_ARG;
  SeedKey key;
  if (int rc = make_seed_key(seed, key)) return rc;
  Rng r(key, 0x5EC2E7);
  c->sk.resize(c->p.n);
  for (auto &s : c->sk) s = r.ternary();
  c->has_sk = true;
  c->has_bt = false;
  c->dev_keys = false;
  c->has_mask_seed = false;
  return BFHE_OK;
}

static void ksk_put(bfhe_ctx *c, u64 idx, u32 v) {
  if (c->ksk_elem_bytes == 2) reinterpret_cast<u16 *>(c->ksk.data())[idx] = (u16)v;
  else reinterpret_cast<u32 *>(c->ksk.data())[idx] = v;
}
static u32 elem_get(const u8 *buf, size_t idx, u32 bytes) {
  return bytes == 2 ? reinterpret_cast<const u16 *>(buf)[idx] : reinterpret_cast<const u32 *>(buf)[idx];
}
static void elem_put(u8 *buf, size_t idx, u32 v, u32 bytes) {
  if (bytes == 2) reinterpret_cast<u16 *>(buf)[idx] = (u16)v;
  else reinterpret_cast<u32 *>(buf)[idx] = v;
}

// ---- mask expansion, host implementation (key_expand.cu is the device one; the rule is stated in include/bfhe.h) ----
// coefficients 0..count-1 of mask row `stream`: keystream words 4t..4t+3 as one little-endian 128-bit integer, mod m
template <typename F> static void expand_mask(const MaskKey &mask, u64 stream, u32 m, size_t count, F put) {
  SeedKey key;
  std::memcpy(key.k, mask.k, sizeof key.k);
  Rng r(key, stream);
  for (size_t t = 0; t < count; t++) {
    u128 v = r.next32();
    for (int w = 1; w < 4; w++) v |= (u128)r.next32() << (32 * w);
    put(t, (u32)(v % m));
  }
}
static size_t ksk_rows(const bfhe_ctx *c) { return (size_t)c->p.N * c->p.baseKS * c->p.dKS; }
static bool compact_only(const bfhe_ctx *c) { return c->bk_coef.empty() && !c->bk_body.empty(); }
void bfhe::host_full_bk(const bfhe_ctx *c, u32 *out) {
  if (!compact_only(c)) { std::memcpy(out, c->bk_coef.data(), c->bk_words * 4); return; }
  const size_t N = c->p.N;
#pragma omp parallel for schedule(static)
  for (i64 s = 0; s < (i64)(c->bk_words / (2 * N)); s++) {
    u32 *a = out + 2 * (size_t)s * N;
    expand_mask(c->mask_seed, BK_MASK_STREAM + (u64)s, (u32)c->p.Q, N, [&](size_t t, u32 v) { a[t] = v; });
    std::memcpy(a + N, c->bk_body.data() + (size_t)s * N, N * 4);
  }
}
void bfhe::host_full_ksk(const bfhe_ctx *c, u8 *out) {
  if (!compact_only(c)) { std::memcpy(out, c->ksk.data(), c->ksk_elems * c->ksk_elem_bytes); return; }
  const u32 n = c->p.n, eb = c->ksk_elem_bytes;
#pragma omp parallel for schedule(static)
  for (i64 r = 0; r < (i64)ksk_rows(c); r++) {
    const size_t base = (size_t)r * (n + 1);
    expand_mask(c->mask_seed, (u64)r, (u32)c->p.qKS, n, [&](size_t t, u32 v) { elem_put(out, base + t, v, eb); });
    elem_put(out, base + n, elem_get(c->ksk_body.data(), (size_t)r, eb), eb);
  }
}
static void clear_compact(bfhe_ctx *c) {
  c->has_mask_seed = false;
  std::vector<u32>().swap(c->bk_body);
  std::vector<u8>().swap(c->ksk_body);
}
void bfhe::forget_mask_seed(bfhe_ctx *c) {
  if (c->has_bt && compact_only(c)) {
    std::vector<u32> bk(c->bk_words);
    std::vector<u8> ksk(c->ksk_elems * c->ksk_elem_bytes);
    host_full_bk(c, bk.data());
    host_full_ksk(c, ksk.data());
    c->bk_coef.swap(bk);
    c->ksk.swap(ksk);
  }
  clear_compact(c);
}

// one RGSW ciphertext of sign * X^mm (or of 0) under z, coefficient form: rows (a, a*z + e) + m*G.
// mask != nullptr: every a is the expansion of mask row BK_MASK_STREAM + p0 + row, and an even row, whose message would otherwise sit in
// the public a, carries it in the body as -m*g^l*z instead (the same phase b - a*z = e - m*g^l*z)
static void rgsw_encrypt(const bfhe_ctx *c, const std::vector<u32> &z_eval, bool msg, u32 mm, int sign, const SeedKey &seed, u64 stream,
                         u32 *out, const MaskKey *mask = nullptr, u64 p0 = 0) {
  const u32 N = c->p.N, rows = 2 * c->p.dG;
  const u32 Q = (u32)c->p.Q;
  Rng r(seed, stream);
  std::vector<u32> tmp(N);
  u64 gpow = 1;
  for (u32 row = 0; row < rows; row++) {
    u32 *a = out + ((size_t)row * 2 + 0) * N, *b = out + ((size_t)row * 2 + 1) * N;
    if (mask) expand_mask(*mask, BK_MASK_STREAM + p0 + row, Q, N, [&](size_t t, u32 v) { a[t] = v; });
    else for (u32 j = 0; j < N; j++) a[j] = (u32)r.uniform(Q);
    std::copy(a, a + N, tmp.begin());
    c->hntt.fwd(tmp.data());
    for (u32 j = 0; j < N; j++) tmp[j] = (u32)((u64)tmp[j] * z_eval[j] % Q);
    c->hntt.inv(tmp.data());
    for (u32 j = 0; j < N; j++) {
      i64 e = gauss_table().sample(r);
      b[j] = (u32)(((i64)tmp[j] + e + Q) % Q);
    }
    if (msg && mask && !(row & 1)) { // b -= sign * g * X^mm * z  (negacyclic: X^N = -1)
      const i64 g = (i64)(gpow % Q);
      for (u32 j = 0; j < N; j++) {
        const i64 zj = j >= mm ? c->z[j - mm] : -(i64)c->z[j + N - mm];
        b[j] = (u32)((((i64)b[j] - sign * g * zj) % Q + Q) % Q);
      }
    } else if (msg) {
      u32 g = (u32)(gpow % Q);
      u32 *dst = (row & 1) ? b : a;
      dst[mm] = sign > 0 ? (u32)(((u64)dst[mm] + g) % Q) : (u32)(((u64)dst[mm] + Q - g) % Q);
    }
    if (row & 1) gpow *= c->p.baseG;
  }
}

// BTKeyGen; mask != nullptr: every mask is the expansion of that public seed (bfhe_btkeygen_compact)
static int btkeygen(bfhe_ctx *c, uint64_t seed64, const MaskKey *mask) {
  if (!c) return BFHE_ERR_ARG;
  if (!c->has_sk) { set_error("BTKeyGen before KeyGen"); return BFHE_ERR_STATE; }
  const bfhe_params &p = c->p;
  const u32 n = p.n, N = p.N;
  const u32 Q = (u32)p.Q;
  const u64 qKS = p.qKS;
  SeedKey seed;
  if (int rc = make_seed_key(seed64, seed)) return rc;
  Rng rz(seed, 0x2A11);
  c->z.resize(N);
  for (auto &v : c->z) v = rz.ternary();
  std::vector<u32> z_eval(N);
  for (u32 i = 0; i < N; i++) z_eval[i] = c->z[i] < 0 ? Q - 1 : (u32)c->z[i];
  c->hntt.fwd(z_eval.data());
  // key-switching key: KSK[i][j][k] = (a, <a,s> + e + z_i * j * B^k) mod qKS
  c->ksk.assign(c->ksk_elems * c->ksk_elem_bytes, 0);
  std::vector<u64> Bpow(p.dKS);
  { u64 b = 1; for (u32 k = 0; k < p.dKS; k++) { Bpow[k] = b; b *= p.baseKS; } }
#pragma omp parallel for schedule(static)
  for (i64 i = 0; i < (i64)N; i++) {
    Rng r(seed, 0x100000 + (u64)i);
    for (u32 j = 0; j < p.baseKS; j++)
      for (u32 k = 0; k < p.dKS; k++) {
        const u64 row = ((u64)i * p.baseKS + j) * p.dKS + k, base = row * (n + 1);
        i64 b = gauss_table().sample(r) + (i64)c->z[i] * (i64)((u64)j * Bpow[k] % qKS);
        if (mask) {
          expand_mask(*mask, row, (u32)qKS, n, [&](size_t t, u32 a) { ksk_put(c, base + t, a); b += (i64)a * c->sk[t]; });
        } else {
          for (u32 t = 0; t < n; t++) {
            u64 a = r.uniform(qKS);
            ksk_put(c, base + t, (u32)a);
            b += (i64)a * c->sk[t];
          }
        }
        b %= (i64)qKS;
        if (b < 0) b += qKS;
        ksk_put(c, base + n, (u32)b);
      }
  }
  // bootstrapping key
  c->bk_coef.assign(c->bk_words, 0);
  const size_t rw = (size_t)(2 * p.dG) * 2 * N;
  if (p.method == BFHE_GINX) { // ek[i] = (RGSW(s_i == 1), RGSW(s_i == -1))
#pragma omp parallel for schedule(dynamic, 4)
    for (i64 i = 0; i < (i64)n; i++) {
      rgsw_encrypt(c, z_eval, c->sk[i] == 1, 0, +1, seed, 0x200000 + 2 * (u64)i, c->bk_coef.data() + ((size_t)i * 2 + 0) * rw, mask,
                   ((u64)i * 2 + 0) * 2 * p.dG);
      rgsw_encrypt(c, z_eval, c->sk[i] == -1, 0, +1, seed, 0x200000 + 2 * (u64)i + 1, c->bk_coef.data() + ((size_t)i * 2 + 1) * rw, mask,
                   ((u64)i * 2 + 1) * 2 * p.dG);
    }
  } else { // ek[i][j][k] = RGSW(X^{(s_i * j * Br^k mod q) * 2N/q}), j in [1, Br)
    const i64 total = (i64)n * (p.baseR - 1) * p.dR;
#pragma omp parallel for schedule(dynamic, 16)
    for (i64 t = 0; t < total; t++) {
      const u32 k = (u32)(t % p.dR), j = (u32)((t / p.dR) % (p.baseR - 1)) + 1, i = (u32)(t / ((i64)p.dR * (p.baseR - 1)));
      i64 Br = 1;
      for (u32 kk = 0; kk < k; kk++) Br *= p.baseR;
      const i64 m = (i64)c->sk[i] * (i64)j * Br;
      i64 mm = (((m % (i64)p.q) + p.q) % p.q) * (2 * N / p.q);
      int sign = 1;
      if (mm >= (i64)N) { mm -= N; sign = -1; }
      rgsw_encrypt(c, z_eval, true, (u32)mm, sign, seed, 0x300000 + (u64)t, c->bk_coef.data() + (size_t)t * rw, mask, (u64)t * 2 * p.dG);
    }
  }
  c->z.clear();
  clear_compact(c);
  if (mask) { c->has_mask_seed = true; c->mask_seed = *mask; }
  c->has_bt = true;
  c->dev_keys = false;
  if (c->device >= 0) return ensure_device_keys(c);
  return BFHE_OK;
}

extern "C" int bfhe_btkeygen(bfhe_ctx *c, uint64_t seed64) { return btkeygen(c, seed64, nullptr); }

// a fresh public mask seed.  seed64 == 0: OS entropy, independent of the secret stream; else reproducible: 256 bits of stream `stream` of
// the secret SeedKey (ChaCha20 output reveals nothing about the key)
static int make_mask_seed(uint64_t seed64, u64 stream, MaskKey &mask) {
  if (seed64 == 0) {
    if (!SeedKey::os_entropy(mask.k, sizeof mask.k)) { set_error("cannot read OS entropy (getrandom and /dev/urandom both failed)"); return BFHE_ERR_IO; }
    return BFHE_OK;
  }
  SeedKey seed;
  if (int rc = make_seed_key(seed64, seed)) return rc;
  Rng r(seed, stream);
  for (auto &w : mask.k) w = r.next32();
  return BFHE_OK;
}

extern "C" int bfhe_btkeygen_compact(bfhe_ctx *c, uint64_t seed64) {
  if (!c) return BFHE_ERR_ARG;
  if (!c->has_sk) { set_error("BTKeyGen before KeyGen"); return BFHE_ERR_STATE; }
  MaskKey mask;
  if (int rc = make_mask_seed(seed64, 0x4D41534B, mask)) return rc;
  return btkeygen(c, seed64, &mask);
}

// upload: BK through the conversion kernel, KSK re-laid-out as [i][k][digit][row].  Keys held as mask seed + bodies (compact_only) have
// their masks generated on the device, into the same coefficient-form staging buffer and straight into the device KSK.  dbg_bk / dbg_ksk
// (bfhe_dbg_expand_keys, compact keys only): receive the staging buffer and the device KSK, in the BFHEKEY1 layouts.
static int upload_keys(bfhe_ctx *c, u32 *dbg_bk, u8 *dbg_ksk) {
  if (c->dev_keys) return BFHE_OK;
  if (c->device < 0) { set_error("no CUDA device attached (this engine has no CPU fallback)"); return BFHE_ERR_CUDA; }
  if (!c->has_bt) { set_error("bootstrapping keys missing: call bfhe_btkeygen or bfhe_import_keys first"); return BFHE_ERR_STATE; }
  BFHE_CUDA(cudaSetDevice(c->device));
  const bfhe_params &p = c->p;
  const u32 N = p.N;
  const bool compact = compact_only(c);
  const int ap = p.method == BFHE_AP;
  c->d_bk.reset(); c->d_bkf.reset(); c->d_bk4.reset(); c->d_bkx.reset(); c->d_ksk.reset();
  BFHE_CUDA(c->d_bk.alloc(c->bk_words));
  { // convert in slices so the temporary coefficient-form copy stays small
    const size_t npoly = c->bk_words / N, slice = 1 << 15; // even: a slice holds whole (mask, body) pairs
    DevBuf<u32> coef, body;
    BFHE_CUDA(coef.alloc(std::min(npoly, slice) * N));
    if (compact) BFHE_CUDA(body.alloc(std::min(npoly, slice) / 2 * N));
    for (size_t p0 = 0; p0 < npoly; p0 += slice) {
      const size_t np = std::min(slice, npoly - p0);
      if (compact) {
        BFHE_CUDA(cudaMemcpyAsync(body.get(), c->bk_body.data() + p0 / 2 * N, np / 2 * N * 4, cudaMemcpyHostToDevice, c->stream));
        int rc = launch_bk_mask_expand(c->mask_seed, body.get(), coef.get(), p0 / 2, np / 2, N, (u32)p.Q, c->stream);
        if (rc) return cuda_fail((cudaError_t)rc, "bk_mask_expand");
        if (dbg_bk) BFHE_CUDA(cudaMemcpyAsync(dbg_bk + p0 * N, coef.get(), np * N * 4, cudaMemcpyDeviceToHost, c->stream));
      } else {
        BFHE_CUDA(cudaMemcpyAsync(coef.get(), c->bk_coef.data() + p0 * N, np * N * 4, cudaMemcpyHostToDevice, c->stream));
      }
      int rc = launch_bk_convert(c->P, coef.get(), c->d_bk.get() + p0 * N, np, c->d_twl.get(), c->stream);
      if (rc) return cuda_fail((cudaError_t)rc, "bk_convert");
      BFHE_CUDA(cudaStreamSynchronize(c->stream));
    }
  }
  if (form_supported(c->P, ap, Form::CL2)) { // key copy of the 2-CTA cluster kernel: kernels_v2.cu's physical slot order
    DevBuf<u32> tmp;                         // (a temporary), split [step][quarter][polynomial][N/4]
    BFHE_CUDA(tmp.alloc(c->bk_words));
    int rc = launch_bk_permute_v2(c->d_bk.get(), tmp.get(), c->bk_words / N, c->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "bk_permute_v2");
    BFHE_CUDA(c->d_bk4.alloc(c->bk_words));
    rc = launch_bk_split_cl4(tmp.get(), c->d_bk4.get(), c->bk_words / N, c->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "bk_split_cl4");
    cudaStreamSynchronize(c->stream);
  }
  if (form_supported(c->P, ap, Form::CL4)) { // key copy of the slot-sliced cluster kernel: [step][rank][polynomial][N/4]
    BFHE_CUDA(c->d_bkx.alloc(c->bk_words));
    int rc = launch_bk_slice_clx(c->d_bk.get(), c->d_bkx.get(), c->bk_words / N, ap, c->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "bk_slice_clx");
    BFHE_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (bk_fold_supported(c->P, ap)) { // key copy of the GINX throughput kernel at this shape: the top digit folded into the other rows
    BFHE_CUDA(c->d_bkf.alloc(c->bk_words));
    int rc = launch_bk_fold(c->P, c->d_bk.get(), c->d_bkf.get(), p.n, c->stream);
    if (rc) return cuda_fail((cudaError_t)rc, "bk_fold");
    BFHE_CUDA(cudaStreamSynchronize(c->stream));
  }
  { // KSK: [i][j(digit value)][k(digit index)][n+1]  ->  [i][k][j][rowlen]
    const u32 rowlen = c->ksk_elem_bytes == 2 ? 512 : p.ct_stride; // elements per padded row
    if (c->ksk_elem_bytes == 2 && p.n + 1 > 512) { set_error("LWE dimension too large for the packed key-switch kernel"); return BFHE_ERR_ARG; }
    const size_t rows = ksk_rows(c), bytes = rows * rowlen * c->ksk_elem_bytes;
    const size_t src_row = (size_t)(p.n + 1) * c->ksk_elem_bytes, dst_row = (size_t)rowlen * c->ksk_elem_bytes;
    auto relayout = [&](u8 *full, u8 *dev, bool to_dev) { // full [i][j][k][n+1] <-> device [i][k][j][rowlen]
#pragma omp parallel for schedule(static)
      for (i64 i = 0; i < (i64)N; i++)
        for (u32 j = 0; j < p.baseKS; j++)
          for (u32 k = 0; k < p.dKS; k++) {
            const size_t s = (((size_t)i * p.baseKS + j) * p.dKS + k), d = (((size_t)i * p.dKS + k) * p.baseKS + j);
            if (to_dev) std::memcpy(dev + d * dst_row, full + s * src_row, src_row);
            else std::memcpy(full + s * src_row, dev + d * dst_row, src_row);
          }
    };
    if (compact) {
      BFHE_CUDA(c->d_ksk.alloc(bytes));
      DevBuf<u8> kb;
      BFHE_CUDA(kb.alloc(c->ksk_body.size()));
      BFHE_CUDA(cudaMemcpyAsync(kb.get(), c->ksk_body.data(), c->ksk_body.size(), cudaMemcpyHostToDevice, c->stream));
      int rc = launch_ksk_expand(c->mask_seed, kb.get(), c->d_ksk.get(), c->ksk_elem_bytes, N, p.baseKS, p.dKS, p.n, rowlen, (u32)p.qKS, c->stream);
      if (rc) return cuda_fail((cudaError_t)rc, "ksk_expand");
      BFHE_CUDA(cudaStreamSynchronize(c->stream));
      if (dbg_ksk) {
        std::vector<u8> dev(bytes);
        BFHE_CUDA(cudaMemcpy(dev.data(), c->d_ksk.get(), bytes, cudaMemcpyDeviceToHost));
        relayout(dbg_ksk, dev.data(), false);
      }
    } else {
      std::vector<u8> dev(bytes, 0);
      relayout(c->ksk.data(), dev.data(), true);
      BFHE_CUDA(upload(c->d_ksk, dev));
    }
  }
  c->dev_keys = true;
  return BFHE_OK;
}
int bfhe::ensure_device_keys(bfhe_ctx *c) { return upload_keys(c, nullptr, nullptr); }

// -------------------------------------------------------------------------------------------------
// key blob
// -------------------------------------------------------------------------------------------------
extern "C" size_t bfhe_keyblob_size(const bfhe_ctx *c) {
  if (!c) return 0;
  return sizeof(KeyBlobHeader) + pad8((size_t)c->p.n * 4) + pad8(c->bk_words * 4) + pad8(c->ksk_elems * c->ksk_elem_bytes);
}
extern "C" size_t bfhe_keyblob_compact_size(const bfhe_ctx *c) {
  if (!c) return 0;
  return sizeof(KeyBlobHeader) + sizeof(MaskKey) + pad8((size_t)c->p.n * 4) + pad8(c->bk_words / 2 * 4) + pad8(ksk_rows(c) * c->ksk_elem_bytes);
}
// header (BFHEKEY1 / BFHEKEY2) and, for BFHEKEY2, the mask seed, then the sk section; returns the first byte after it
static u8 *put_header(const bfhe_ctx *c, u8 *o, bool compact, bool include_sk) {
  KeyBlobHeader h{};
  std::memcpy(h.magic, compact ? "BFHEKEY2" : "BFHEKEY1", 8);
  const bfhe_params &p = c->p;
  h.version = 1; h.paramset = p.paramset; h.method = p.method; h.n = p.n; h.N = p.N; h.q = p.q;
  h.baseKS = p.baseKS; h.dKS = p.dKS; h.baseG = p.baseG; h.dG = p.dG; h.baseR = p.baseR; h.dR = p.dR;
  h.has_sk = (include_sk && c->has_sk) ? 1 : 0; h.ksk_elem_bytes = c->ksk_elem_bytes;
  h.Q = p.Q; h.qKS = p.qKS; h.bk_words = c->bk_words; h.ksk_elems = c->ksk_elems;
  std::memcpy(o, &h, sizeof h); o += sizeof h;
  if (compact) { std::memcpy(o, &c->mask_seed, sizeof c->mask_seed); o += sizeof c->mask_seed; }
  std::memset(o, 0, pad8((size_t)p.n * 4));
  if (h.has_sk) std::memcpy(o, c->sk.data(), (size_t)p.n * 4);
  return o + pad8((size_t)p.n * 4);
}
extern "C" int bfhe_export_keys(const bfhe_ctx *c, void *buf, size_t cap, int include_sk) {
  if (!c || !buf) return BFHE_ERR_ARG;
  if (!c->has_bt) { set_error("no keys to export"); return BFHE_ERR_STATE; }
  if (cap < bfhe_keyblob_size(c)) { set_error("export buffer too small"); return BFHE_ERR_ARG; }
  u8 *o = put_header(c, (u8 *)buf, false, include_sk);
  host_full_bk(c, (u32 *)o); o += pad8(c->bk_words * 4);
  host_full_ksk(c, o);
  return BFHE_OK;
}
extern "C" int bfhe_export_keys_compact(const bfhe_ctx *c, void *buf, size_t cap, int include_sk) {
  if (!c || !buf) return BFHE_ERR_ARG;
  if (!c->has_bt) { set_error("no keys to export"); return BFHE_ERR_STATE; }
  if (!c->has_mask_seed) { set_error("these keys have no mask seed (made by bfhe_btkeygen or imported in full): only bfhe_export_keys can export them"); return BFHE_ERR_STATE; }
  if (cap < bfhe_keyblob_compact_size(c)) { set_error("export buffer too small"); return BFHE_ERR_ARG; }
  u8 *o = put_header(c, (u8 *)buf, true, include_sk);
  const size_t N = c->p.N, pairs = c->bk_words / (2 * N), rows = ksk_rows(c);
  const u32 n = c->p.n, eb = c->ksk_elem_bytes;
  u32 *bk = (u32 *)o;
  u8 *ksk = o + pad8(pairs * N * 4);
  if (compact_only(c)) {
    std::memcpy(bk, c->bk_body.data(), pairs * N * 4);
    std::memcpy(ksk, c->ksk_body.data(), rows * eb);
  } else {
    for (size_t s = 0; s < pairs; s++) std::memcpy(bk + s * N, c->bk_coef.data() + (2 * s + 1) * N, N * 4);
    for (size_t r = 0; r < rows; r++) elem_put(ksk, r, elem_get(c->ksk.data(), r * (n + 1) + n, eb), eb);
  }
  std::memset(bk + pairs * N, 0, pad8(pairs * N * 4) - pairs * N * 4);
  std::memset(ksk + rows * eb, 0, pad8(rows * eb) - rows * eb);
  return BFHE_OK;
}

// BFHEKEY2 import: every check before the context changes; dbg_bk / dbg_ksk as upload_keys
static int import_compact(bfhe_ctx *c, const KeyBlobHeader &h, const u8 *buf, size_t len, u32 *dbg_bk, u8 *dbg_ksk) {
  if (len < bfhe_keyblob_compact_size(c)) { set_error("BFHEKEY2 key blob truncated"); return BFHE_ERR_FORMAT; }
  const bfhe_params &p = c->p;
  const size_t N = p.N, pairs = c->bk_words / (2 * N), rows = ksk_rows(c);
  const u32 eb = c->ksk_elem_bytes;
  MaskKey mask;
  const u8 *in = buf + sizeof h;
  std::memcpy(&mask, in, sizeof mask); in += sizeof mask;
  const u8 *sk = in; in += pad8((size_t)p.n * 4);
  const u32 *bk = (const u32 *)in; in += pad8(pairs * N * 4);
  const u8 *ksk = in;
  for (size_t i = 0; i < pairs * N; i++)
    if (bk[i] >= p.Q) { set_error("BFHEKEY2: BK body word " + std::to_string(i) + " = " + std::to_string(bk[i]) + " is not below Q"); return BFHE_ERR_FORMAT; }
  for (size_t i = 0; i < rows; i++)
    if (elem_get(ksk, i, eb) >= p.qKS) {
      set_error("BFHEKEY2: KSK body word " + std::to_string(i) + " = " + std::to_string(elem_get(ksk, i, eb)) + " is not below qKS");
      return BFHE_ERR_FORMAT;
    }
  if (h.has_sk) { c->sk.resize(p.n); std::memcpy(c->sk.data(), sk, (size_t)p.n * 4); c->has_sk = true; }
  c->has_mask_seed = true;
  c->mask_seed = mask;
  c->bk_body.assign(bk, bk + pairs * N);
  c->ksk_body.assign(ksk, ksk + rows * eb);
  std::vector<u32>().swap(c->bk_coef); // compact_only from here on
  std::vector<u8>().swap(c->ksk);
  c->has_bt = true;
  c->dev_keys = false;
  if (c->device >= 0) return upload_keys(c, dbg_bk, dbg_ksk);
  std::vector<u32> full_bk(c->bk_words); // host-only context: the full forms, as after bfhe_btkeygen_compact
  std::vector<u8> full_ksk(c->ksk_elems * eb);
  host_full_bk(c, full_bk.data());
  host_full_ksk(c, full_ksk.data());
  c->bk_coef.swap(full_bk);
  c->ksk.swap(full_ksk);
  std::vector<u32>().swap(c->bk_body);
  std::vector<u8>().swap(c->ksk_body);
  return BFHE_OK;
}
static int read_header(const bfhe_ctx *c, const void *buf, size_t len, KeyBlobHeader &h, bool &compact) {
  if (len < sizeof h) { set_error("key blob truncated"); return BFHE_ERR_FORMAT; }
  std::memcpy(&h, buf, sizeof h);
  compact = !std::memcmp(h.magic, "BFHEKEY2", 8);
  if ((!compact && std::memcmp(h.magic, "BFHEKEY1", 8)) || h.version != 1) { set_error("not a BFHEKEY1 or BFHEKEY2 blob"); return BFHE_ERR_FORMAT; }
  const bfhe_params &p = c->p;
  if (h.paramset != p.paramset || h.method != p.method || h.n != p.n || h.N != p.N || h.q != p.q || h.Q != p.Q || h.qKS != p.qKS ||
      h.baseKS != p.baseKS || h.dKS != p.dKS || h.baseG != p.baseG || h.dG != p.dG || h.baseR != p.baseR || h.dR != p.dR ||
      h.bk_words != c->bk_words || h.ksk_elems != c->ksk_elems || h.ksk_elem_bytes != c->ksk_elem_bytes) {
    set_error("key blob parameters do not match this context");
    return BFHE_ERR_FORMAT;
  }
  return BFHE_OK;
}
extern "C" int bfhe_import_keys(bfhe_ctx *c, const void *buf, size_t len) {
  if (!c || !buf) return BFHE_ERR_ARG;
  KeyBlobHeader h;
  bool compact = false;
  if (int rc = read_header(c, buf, len, h, compact)) return rc;
  if (compact) return import_compact(c, h, (const u8 *)buf, len, nullptr, nullptr);
  if (len < bfhe_keyblob_size(c)) { set_error("key blob truncated"); return BFHE_ERR_FORMAT; }
  const bfhe_params &p = c->p;
  const u8 *in = (const u8 *)buf + sizeof h;
  if (h.has_sk) { c->sk.resize(p.n); std::memcpy(c->sk.data(), in, (size_t)p.n * 4); c->has_sk = true; }
  in += pad8((size_t)p.n * 4);
  c->bk_coef.resize(c->bk_words);
  std::memcpy(c->bk_coef.data(), in, c->bk_words * 4); in += pad8(c->bk_words * 4);
  c->ksk.resize(c->ksk_elems * c->ksk_elem_bytes);
  std::memcpy(c->ksk.data(), in, c->ksk.size());
  clear_compact(c);
  c->has_bt = true;
  c->dev_keys = false;
  if (c->device >= 0) return ensure_device_keys(c);
  return BFHE_OK;
}
extern "C" int bfhe_dbg_expand_keys(bfhe_ctx *c, const void *compact_blob, size_t len, void *full_blob, size_t cap) {
  if (!c || !compact_blob || !full_blob) return BFHE_ERR_ARG;
  if (c->device < 0) { set_error("no CUDA device attached (bfhe_dbg_expand_keys runs the device expansion)"); return BFHE_ERR_CUDA; }
  if (cap < bfhe_keyblob_size(c)) { set_error("expansion buffer too small"); return BFHE_ERR_ARG; }
  KeyBlobHeader h;
  bool compact = false;
  if (int rc = read_header(c, compact_blob, len, h, compact)) return rc;
  if (!compact) { set_error("not a BFHEKEY2 blob"); return BFHE_ERR_FORMAT; }
  u8 *bk = (u8 *)full_blob + sizeof h + pad8((size_t)c->p.n * 4), *ksk = bk + pad8(c->bk_words * 4);
  if (int rc = import_compact(c, h, (const u8 *)compact_blob, len, (u32 *)bk, ksk)) return rc;
  put_header(c, (u8 *)full_blob, false, h.has_sk != 0);
  std::memset(bk + c->bk_words * 4, 0, pad8(c->bk_words * 4) - c->bk_words * 4);
  return BFHE_OK;
}
extern "C" int bfhe_save_keys(const bfhe_ctx *c, const char *path, int include_sk) {
  if (!c || !path) return BFHE_ERR_ARG;
  std::vector<u8> buf(bfhe_keyblob_size(c));
  int rc = bfhe_export_keys(c, buf.data(), buf.size(), include_sk);
  if (rc) return rc;
  FILE *f = std::fopen(path, "wb");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  size_t w = std::fwrite(buf.data(), 1, buf.size(), f);
  std::fclose(f);
  if (w != buf.size()) { set_error("short write"); return BFHE_ERR_IO; }
  return BFHE_OK;
}
extern "C" int bfhe_load_keys(bfhe_ctx *c, const char *path) {
  if (!c || !path) return BFHE_ERR_ARG;
  FILE *f = std::fopen(path, "rb");
  if (!f) { set_error(std::string("cannot open ") + path); return BFHE_ERR_IO; }
  std::fseek(f, 0, SEEK_END);
  long sz = std::ftell(f);
  std::fseek(f, 0, SEEK_SET);
  std::vector<u8> buf((size_t)sz);
  size_t r = std::fread(buf.data(), 1, buf.size(), f);
  std::fclose(f);
  if (r != buf.size()) { set_error("short read"); return BFHE_ERR_IO; }
  return bfhe_import_keys(c, buf.data(), buf.size());
}

// -------------------------------------------------------------------------------------------------
// host LWE: Encrypt (FRESH) / Decrypt
// -------------------------------------------------------------------------------------------------
extern "C" int bfhe_encrypt(const bfhe_ctx *c, const uint8_t *bits, size_t count, uint64_t seed, uint32_t *ct) {
  if (!c || !bits || !ct) return BFHE_ERR_ARG;
  if (!c->has_sk) { set_error("Encrypt before KeyGen"); return BFHE_ERR_STATE; }
  const u32 n = c->p.n, q = c->p.q, stride = c->p.ct_stride;
  SeedKey key;
  if (int rc = make_seed_key(seed, key)) return rc;
#pragma omp parallel for schedule(static) if (count > 256)
  for (i64 g = 0; g < (i64)count; g++) {
    Rng r(key, 0x900000 + (u64)g);
    u32 *row = ct + (size_t)g * stride;
    i64 b = (i64)(bits[g] % 4) * (q / 4) + gauss_table().sample(r);
    for (u32 i = 0; i < n; i++) {
      row[i] = (u32)r.uniform(q);
      b += (i64)row[i] * c->sk[i];
    }
    b %= (i64)q;
    if (b < 0) b += q;
    row[n] = (u32)b;
    for (u32 i = n + 1; i < stride; i++) row[i] = 0;
  }
  return BFHE_OK;
}
extern "C" int bfhe_decrypt(const bfhe_ctx *c, const uint32_t *ct, size_t count, uint8_t *out) {
  if (!c || !ct || !out) return BFHE_ERR_ARG;
  if (!c->has_sk) { set_error("Decrypt without a secret key"); return BFHE_ERR_STATE; }
  const u32 n = c->p.n, stride = c->p.ct_stride;
  const i64 q = c->p.q;
#pragma omp parallel for schedule(static) if (count > 256)
  for (i64 g = 0; g < (i64)count; g++) {
    const u32 *row = ct + (size_t)g * stride;
    i64 r = row[n];
    for (u32 i = 0; i < n; i++) r -= (i64)row[i] * c->sk[i];
    r = ((r % q) + q) % q;
    r = (r + q / 8) % q;
    out[g] = (u8)(4 * r / q);
  }
  return BFHE_OK;
}

// -------------------------------------------------------------------------------------------------
// slabs
// -------------------------------------------------------------------------------------------------
static int need_device(const bfhe_ctx *c) {
  if (!c) return BFHE_ERR_ARG;
  if (c->device < 0) { set_error("no CUDA device attached (this engine has no CPU fallback)"); return BFHE_ERR_CUDA; }
  cudaError_t e = cudaSetDevice(c->device);
  if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
  return BFHE_OK;
}
extern "C" int bfhe_slab_alloc(bfhe_ctx *c, size_t rows, uint32_t **dev_ptr) {
  int rc = need_device(c);
  if (rc) return rc;
  BFHE_CUDA(cudaMalloc(dev_ptr, std::max<size_t>(rows, 1) * c->p.ct_stride * 4));
  BFHE_CUDA(cudaMemsetAsync(*dev_ptr, 0, std::max<size_t>(rows, 1) * c->p.ct_stride * 4, c->stream));
  return BFHE_OK;
}
extern "C" int bfhe_slab_free(bfhe_ctx *c, uint32_t *p) {
  int rc = need_device(c);
  if (rc) return rc;
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  BFHE_CUDA(cudaFree(p));
  return BFHE_OK;
}
extern "C" int bfhe_slab_upload(bfhe_ctx *c, uint32_t *slab, size_t first, const uint32_t *host, size_t rows) {
  int rc = need_device(c);
  if (rc) return rc;
  const size_t st = c->p.ct_stride;
  BFHE_CUDA(cudaMemcpyAsync(slab + first * st, host, rows * st * 4, cudaMemcpyHostToDevice, c->stream));
  return BFHE_OK;
}
extern "C" int bfhe_slab_download(bfhe_ctx *c, const uint32_t *slab, size_t first, uint32_t *host, size_t rows) {
  int rc = need_device(c);
  if (rc) return rc;
  const size_t st = c->p.ct_stride;
  BFHE_CUDA(cudaMemcpyAsync(host, slab + first * st, rows * st * 4, cudaMemcpyDeviceToHost, c->stream));
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  return BFHE_OK;
}
int bfhe::check_device_buffer(const bfhe_ctx *c, const void *p, const char *what) {
  cudaPointerAttributes pa{};
  if (cudaPointerGetAttributes(&pa, p) != cudaSuccess || (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) ||
      pa.device != c->device) {
    cudaGetLastError();
    set_error(std::string(what) + " is not memory of device " + std::to_string(c->device));
    return BFHE_ERR_ARG;
  }
  return BFHE_OK;
}

// -------------------------------------------------------------------------------------------------
// compact fresh ciphertexts (BFHECTS1, include/bfhe.h): a public mask seed and one body per bit
// -------------------------------------------------------------------------------------------------
struct CtBlobHeader {
  char magic[8];
  u32 version, paramset, n, q;
  u64 count;
  MaskKey seed;
};
static_assert(sizeof(CtBlobHeader) == 64, "the BFHECTS1 header is 64 bytes");
static constexpr u64 CT_MASK_SEED_STREAM = 0x43544D534Bull; // stream of the secret SeedKey giving a reproducible mask seed (keys: 0x4D41534B)
static constexpr u64 CT_NOISE_STREAM = 1ull << 48;          // + g: the noise of row g (bfhe_encrypt uses 0x900000 + g)

static u32 ct_body(const u8 *bodies, size_t g) {
  u16 v;
  std::memcpy(&v, bodies + 2 * g, 2);
  return v;
}

extern "C" size_t bfhe_ct_compact_size(const bfhe_ctx *c, size_t count) {
  if (!c || count > (SIZE_MAX - sizeof(CtBlobHeader) - 8) / 2) return 0;
  return sizeof(CtBlobHeader) + pad8(2 * count);
}

extern "C" int bfhe_encrypt_compact(const bfhe_ctx *c, const uint8_t *bits, size_t count, uint64_t seed, void *blob, size_t cap) {
  if (!c || (!bits && count) || !blob) return BFHE_ERR_ARG;
  if (!c->has_sk) { set_error("Encrypt before KeyGen"); return BFHE_ERR_STATE; }
  const size_t size = bfhe_ct_compact_size(c, count);
  if (!size || cap < size) { set_error("bfhe_encrypt_compact: blob buffer too small"); return BFHE_ERR_ARG; }
  SeedKey key;
  if (int rc = make_seed_key(seed, key)) return rc;
  CtBlobHeader h{};
  std::memcpy(h.magic, "BFHECTS1", 8);
  h.version = 1; h.paramset = c->p.paramset; h.n = c->p.n; h.q = c->p.q; h.count = count;
  if (int rc = make_mask_seed(seed, CT_MASK_SEED_STREAM, h.seed)) return rc;
  const u32 n = c->p.n, q = c->p.q;
  u8 *bodies = (u8 *)blob + sizeof h;
#pragma omp parallel for schedule(static) if (count > 256)
  for (i64 g = 0; g < (i64)count; g++) {
    Rng r(key, CT_NOISE_STREAM + (u64)g);
    i64 b = (i64)(bits[g] % 4) * (q / 4) + gauss_table().sample(r);
    expand_mask(h.seed, (u64)g, q, n, [&](size_t t, u32 a) { b += (i64)a * c->sk[t]; });
    b %= (i64)q;
    if (b < 0) b += q;
    const u16 v = (u16)b;
    std::memcpy(bodies + 2 * (size_t)g, &v, 2);
  }
  std::memcpy(blob, &h, sizeof h);
  std::memset(bodies + 2 * count, 0, pad8(2 * count) - 2 * count);
  return BFHE_OK;
}

int bfhe::read_ct_blob(const bfhe_ctx *c, const void *blob, size_t len, CtBlob &out) {
  CtBlobHeader h;
  if (len < sizeof h) { set_error("BFHECTS1: " + std::to_string(len) + " bytes, shorter than the 64-byte header"); return BFHE_ERR_FORMAT; }
  std::memcpy(&h, blob, sizeof h);
  if (std::memcmp(h.magic, "BFHECTS1", 8)) { set_error("BFHECTS1: bad magic, not a compact ciphertext blob"); return BFHE_ERR_FORMAT; }
  if (h.version != 1) { set_error("BFHECTS1: version " + std::to_string(h.version) + " is not 1"); return BFHE_ERR_FORMAT; }
  const bfhe_params &p = c->p;
  if (h.paramset != p.paramset || h.n != p.n || h.q != p.q) {
    set_error("BFHECTS1: paramset " + std::to_string(h.paramset) + ", n " + std::to_string(h.n) + ", q " + std::to_string(h.q) +
              " do not match this context (paramset " + std::to_string(p.paramset) + ", n " + std::to_string(p.n) + ", q " + std::to_string(p.q) + ")");
    return BFHE_ERR_FORMAT;
  }
  if (h.count > (len - sizeof h) / 2 || len != sizeof h + pad8(2 * h.count)) {
    set_error("BFHECTS1: length " + std::to_string(len) + " bytes does not match count " + std::to_string(h.count) + " (64 + pad8(2 count) bytes)");
    return BFHE_ERR_FORMAT;
  }
  const u8 *bodies = (const u8 *)blob + sizeof h;
  for (size_t g = 0; g < h.count; g++)
    if (ct_body(bodies, g) >= p.q) {
      set_error("BFHECTS1: body " + std::to_string(g) + " = " + std::to_string(ct_body(bodies, g)) + " is not below q = " + std::to_string(p.q));
      return BFHE_ERR_FORMAT;
    }
  for (size_t i = 2 * h.count; i < len - sizeof h; i++)
    if (bodies[i]) { set_error("BFHECTS1: nonzero padding byte at offset " + std::to_string(sizeof h + i)); return BFHE_ERR_FORMAT; }
  out.seed = h.seed;
  out.count = h.count;
  out.bodies = bodies;
  return BFHE_OK;
}

int bfhe::expand_ct_rows(bfhe_ctx *c, const CtBlob &b, u32 *d_rows, std::vector<u32> &wide) {
  if (b.count == 0) return BFHE_OK;
  wide.resize(b.count);
  for (size_t g = 0; g < b.count; g++) wide[g] = ct_body(b.bodies, g);
  // the bodies go through the per-call scratch rows (kept between calls; a stream-ordered allocation would map fresh memory every time)
  BFHE_CUDA(c->d_tmp.reserve(b.count, c->stream));
  BFHE_CUDA(cudaMemcpyAsync(c->d_tmp.get(), wide.data(), b.count * 4, cudaMemcpyHostToDevice, c->stream));
  int rc = launch_ct_expand(b.seed, c->d_tmp.get(), d_rows, b.count, c->p.n, c->p.ct_stride, c->p.q, c->stream);
  if (rc) return cuda_fail((cudaError_t)rc, "ct_expand");
  return BFHE_OK;
}

extern "C" int bfhe_expand_cts(bfhe_ctx *c, const void *blob, size_t len, uint32_t *cts, size_t cap_rows, int on_device) {
  if (!c || !blob) return BFHE_ERR_ARG;
  CtBlob b;
  if (int rc = read_ct_blob(c, blob, len, b)) return rc;
  if (cap_rows < b.count) {
    set_error("bfhe_expand_cts: the blob holds " + std::to_string(b.count) + " rows, the destination " + std::to_string(cap_rows));
    return BFHE_ERR_ARG;
  }
  if (!cts && b.count) { set_error("bfhe_expand_cts: null destination"); return BFHE_ERR_ARG; }
  if (!on_device) {
    const u32 n = c->p.n, q = c->p.q, st = c->p.ct_stride;
#pragma omp parallel for schedule(static) if (b.count > 256)
    for (i64 g = 0; g < (i64)b.count; g++) {
      u32 *row = cts + (size_t)g * st;
      expand_mask(b.seed, (u64)g, q, n, [&](size_t t, u32 a) { row[t] = a; });
      row[n] = ct_body(b.bodies, (size_t)g);
      for (u32 i = n + 1; i < st; i++) row[i] = 0;
    }
    return BFHE_OK;
  }
  if (int rc = need_device(c)) return rc;
  if (b.count == 0) return BFHE_OK;
  std::lock_guard<std::mutex> lk(c->mtx);
  if (int rc = check_device_buffer(c, cts, "bfhe_expand_cts: the destination")) return rc;
  if ((uintptr_t)cts % 16) { set_error("bfhe_expand_cts: the destination is not 16-byte aligned"); return BFHE_ERR_ARG; }
  std::vector<u32> wide;
  if (int rc = expand_ct_rows(c, b, cts, wide)) return rc;
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  return BFHE_OK;
}

// -------------------------------------------------------------------------------------------------
// hot path
// -------------------------------------------------------------------------------------------------
static void prof_begin(bfhe_ctx *c, int kernel, cudaStream_t st = nullptr) {
  if (!c->profiling) return;
  ProfSpan s;
  s.kernel = kernel;
  cudaEventCreate(&s.a);
  cudaEventCreate(&s.b);
  cudaEventRecord(s.a, st ? st : c->stream);
  c->spans.push_back(s);
}
static void prof_end(bfhe_ctx *c, cudaStream_t st = nullptr) {
  if (!c->profiling) return;
  cudaEventRecord(c->spans.back().b, st ? st : c->stream);
}

int bfhe::run_gate_list(bfhe_ctx *c, const DevGate *list, size_t count, u32 *acc_dbg_host) {
  const u32 N = c->p.N;
  DevBuf<u32> d_acc;
  if (acc_dbg_host) BFHE_CUDA(d_acc.alloc(std::min(count, c->chunk) * 2 * N));
  // Gates of one list are independent, so with several chunks the (HBM-bound) key switch of chunk k runs on a side
  // stream underneath the (integer-bound) blind rotation of chunk k+1; two sets of descriptor / ext buffers.
  const bool overlap = count > c->chunk && !acc_dbg_host;
  int k = 0;
  for (size_t off = 0; off < count; off += c->chunk, k++) {
    const size_t m = std::min(c->chunk, count - off);
    const int b = overlap ? (k & 1) : 0;
    DevGate *dg = (b ? c->d_gates_b : c->d_gates).get();
    u32 *de = (b ? c->d_ext_b : c->d_ext).get();
    if (overlap && k >= 2) BFHE_CUDA(cudaStreamWaitEvent(c->stream, c->ev_ks[b], 0)); // buffers of chunk k-2 are free again
    const int sb = c->stage_next;
    c->stage_next ^= 1;
    BFHE_CUDA(cudaEventSynchronize(c->stage_ev[sb])); // staging buffer free again?
    std::memcpy(c->h_gates[sb].get(), list + off, m * sizeof(DevGate));
    BFHE_CUDA(cudaMemcpyAsync(dg, c->h_gates[sb].get(), m * sizeof(DevGate), cudaMemcpyHostToDevice, c->stream));
    BFHE_CUDA(cudaEventRecord(c->stage_ev[sb], c->stream));
    prof_begin(c, 0);
    int rc = launch_blind_rotate(c->P, c->p.method == BFHE_AP, dg, (int)m, c->keys(), de, d_acc.get(), (Form)c->force_g, c->stream);
    prof_end(c);
    if (rc) return cuda_fail((cudaError_t)rc, "blind_rotate launch");
    if (acc_dbg_host) {
      BFHE_CUDA(cudaMemcpyAsync(acc_dbg_host + off * 2 * N, d_acc.get(), m * 2 * N * 4, cudaMemcpyDeviceToHost, c->stream));
      BFHE_CUDA(cudaStreamSynchronize(c->stream));
    }
    cudaStream_t kst = overlap ? c->ks_stream : c->stream;
    if (overlap) {
      BFHE_CUDA(cudaEventRecord(c->ev_br[b], c->stream));
      BFHE_CUDA(cudaStreamWaitEvent(c->ks_stream, c->ev_br[b], 0));
    }
    prof_begin(c, 1, kst);
    rc = launch_keyswitch(c->P, de, dg, (int)m, c->keys(), kst);
    prof_end(c, kst);
    if (rc) return cuda_fail((cudaError_t)rc, "keyswitch launch");
    if (overlap) BFHE_CUDA(cudaEventRecord(c->ev_ks[b], c->ks_stream));
  }
  if (overlap) { // the caller's stream sees every output before anything it enqueues next
    BFHE_CUDA(cudaStreamWaitEvent(c->stream, c->ev_ks[0], 0));
    if (k >= 2) BFHE_CUDA(cudaStreamWaitEvent(c->stream, c->ev_ks[1], 0));
  }
  if (acc_dbg_host) cudaStreamSynchronize(c->stream);
  return BFHE_OK;
}

int bfhe::not_ptr_batch(bfhe_ctx *c, const std::vector<const u32 *> &in, const std::vector<u32 *> &out) {
  if (in.empty()) return BFHE_OK;
  BFHE_CUDA(c->d_ptr_in.reserve(in.size(), c->stream));
  BFHE_CUDA(c->d_ptr_out.reserve(in.size(), c->stream));
  // pointer lists are small; a synchronous copy keeps the host vectors' lifetime trivial
  BFHE_CUDA(cudaMemcpyAsync(c->d_ptr_in.get(), in.data(), in.size() * sizeof(void *), cudaMemcpyHostToDevice, c->stream));
  BFHE_CUDA(cudaMemcpyAsync(c->d_ptr_out.get(), out.data(), out.size() * sizeof(void *), cudaMemcpyHostToDevice, c->stream));
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  prof_begin(c, 2);
  int r2 = launch_eval_not(c->P, c->d_ptr_in.get(), c->d_ptr_out.get(), (int)in.size(), c->stream);
  prof_end(c);
  if (r2) return cuda_fail((cudaError_t)r2, "eval_not launch");
  return BFHE_OK;
}

extern "C" int bfhe_eval_not_batch(bfhe_ctx *c, uint32_t *slab, const uint32_t *in_rows, const uint32_t *out_rows, size_t count) {
  int rc = need_device(c);
  if (rc) return rc;
  if (!slab || !in_rows || !out_rows) return BFHE_ERR_ARG;
  std::lock_guard<std::mutex> lk(c->mtx);
  const size_t st = c->p.ct_stride;
  std::vector<const u32 *> in(count);
  std::vector<u32 *> out(count);
  for (size_t i = 0; i < count; i++) { in[i] = slab + in_rows[i] * st; out[i] = slab + out_rows[i] * st; }
  return not_ptr_batch(c, in, out);
}

// every gate's op in range, and no gate reading the very same ciphertext twice
static int check_gates(const bfhe_gate *gates, size_t count) {
  for (size_t i = 0; i < count; i++) {
    const u32 g = gates[i].op & 0xff;
    if (g > BFHE_BOOTSTRAP) { set_error("unknown gate type"); return BFHE_ERR_ARG; }
    // a and NOT(a) are distinct ciphertext objects for OpenFHE; only the very same ciphertext twice is rejected
    if (g != BFHE_BOOTSTRAP && gates[i].in0 == gates[i].in1 &&
        (((gates[i].op & BFHE_NEG0) != 0) == ((gates[i].op & BFHE_NEG1) != 0))) {
      set_error("EvalBinGate: please only use independent ciphertexts as inputs (gate " + std::to_string(i) + ")");
      return BFHE_ERR_ALIAS;
    }
  }
  return BFHE_OK;
}

static int eval_batch_locked(bfhe_ctx *c, uint32_t *slab, const bfhe_gate *gates, size_t count, u32 *acc_dbg_host) {
  int rc = ensure_device_keys(c);
  if (rc) return rc;
  if ((rc = check_gates(gates, count))) return rc;
  const size_t st = c->p.ct_stride;
  size_t ncomp = 0;
  for (size_t i = 0; i < count; i++)
    if ((gates[i].op & 0xff) == BFHE_XOR || (gates[i].op & 0xff) == BFHE_XNOR) ncomp++;
  if (acc_dbg_host && ncomp) { set_error("debug blind rotation does not take composite gates"); return BFHE_ERR_ARG; }
  BFHE_CUDA(c->d_tmp.reserve(2 * ncomp * st, c->stream));
  std::vector<DevGate> l1, l2;
  std::vector<const u32 *> not_in;
  std::vector<u32 *> not_out;
  l1.reserve(count + ncomp);
  l2.reserve(ncomp);
  size_t t = 0;
  for (size_t i = 0; i < count; i++) {
    const bfhe_gate &g = gates[i];
    const u32 gate = g.op & 0xff;
    const u32 *a = slab + (size_t)g.in0 * st, *b = slab + (size_t)g.in1 * st;
    u32 *o = slab + (size_t)g.out * st;
    if (gate == BFHE_XOR || gate == BFHE_XNOR) { // OR(AND(a, !b), AND(!a, b)), operand order as src/gate.cpp:198-202
      const u32 f0 = g.op & BFHE_NEG0, f1 = g.op & BFHE_NEG1;
      u32 *t1 = c->d_tmp.get() + (2 * t) * st, *t2 = c->d_tmp.get() + (2 * t + 1) * st;
      t++;
      l1.push_back(DevGate{a, b, t1, BFHE_AND | f0 | (f1 ^ BFHE_NEG1), 0});
      l1.push_back(DevGate{a, b, t2, BFHE_AND | (f0 ^ BFHE_NEG0) | f1, 0});
      l2.push_back(DevGate{t1, t2, o, BFHE_OR, 0});
      if (gate == BFHE_XNOR) { not_in.push_back(o); not_out.push_back(o); }
    } else {
      l1.push_back(DevGate{a, gate == BFHE_BOOTSTRAP ? a : b, o, g.op, 0});
    }
  }
  rc = run_gate_list(c, l1.data(), l1.size(), acc_dbg_host);
  if (rc) return rc;
  rc = run_gate_list(c, l2.data(), l2.size(), nullptr);
  if (rc) return rc;
  return not_ptr_batch(c, not_in, not_out);
}

extern "C" int bfhe_eval_bingate_batch(bfhe_ctx *c, uint32_t *slab, const bfhe_gate *gates, size_t count) {
  int rc = need_device(c);
  if (rc) return rc;
  if (!slab || (!gates && count)) return BFHE_ERR_ARG;
  std::lock_guard<std::mutex> lk(c->mtx);
  return eval_batch_locked(c, slab, gates, count, nullptr);
}

extern "C" int bfhe_bootstrap_batch(bfhe_ctx *c, uint32_t *slab, const uint32_t *in_rows, const uint32_t *out_rows, size_t count) {
  int rc = need_device(c);
  if (rc) return rc;
  if (!slab || !in_rows || !out_rows) return BFHE_ERR_ARG;
  std::vector<bfhe_gate> g(count);
  for (size_t i = 0; i < count; i++) g[i] = bfhe_gate{BFHE_BOOTSTRAP, in_rows[i], in_rows[i], out_rows[i]};
  std::lock_guard<std::mutex> lk(c->mtx);
  return eval_batch_locked(c, slab, g.data(), count, nullptr);
}

// ---- combining of concurrent bfhe_eval_bingate_host calls (flat combining; DESIGN.md section 7) ----
// Each call is validated in its own thread, then queued.  With no batch in flight the call leads at once with whatever is queued; calls
// arriving while a batch runs queue up, and when it finishes the front of the queue leads the next batch with everything queued.  A
// gate's output words do not depend on the batch it runs in, so a combined call returns exactly what it would have returned alone.

// the checks of eval_batch_locked and the row ranges of one call, before it may join a batch
static int check_host_call(const bfhe_gate *gates, size_t count, size_t in_rows, size_t out_rows) {
  const size_t rows = in_rows + out_rows;
  for (size_t i = 0; i < count; i++)
    if (gates[i].out < in_rows || gates[i].out >= rows || gates[i].in0 >= rows || gates[i].in1 >= rows) {
      set_error("bfhe_eval_bingate_host: gate rows out of range");
      return BFHE_ERR_ARG;
    }
  return check_gates(gates, count);
}

// one batch.  Staging slab: every request's input rows, in queue order, then every request's output rows, in the same order (a lone call
// gets today's layout: its in_rows, then its out_rows).  One H2D copy per request, one memset of the output block (the kernels write
// ciphertext words only, so padding words come out zero whatever the slab held before), one eval_batch_locked over the concatenated gate
// list with every row translated to its request's block, one D2H copy per request, one synchronise.
static int run_host_batch(bfhe_ctx *c, const std::vector<HostGateReq *> &batch) {
  std::lock_guard<std::mutex> lk(c->mtx);
  const size_t st = c->p.ct_stride;
  size_t in_total = 0, out_total = 0, count = 0;
  for (const HostGateReq *r : batch) { in_total += r->in_rows; out_total += r->out_rows; count += r->count; }
  const size_t rows = in_total + out_total;
  if (rows > 0xffffffffu) { set_error("bfhe_eval_bingate_host: combined batch exceeds 2^32 rows"); return BFHE_ERR_ARG; }
  BFHE_CUDA(c->e2e_slab.reserve(rows * st, c->stream));
  u32 *slab = c->e2e_slab.get();
  std::vector<bfhe_gate> all;
  const bfhe_gate *list = batch[0]->gates; // a lone call: the translation is the identity
  if (batch.size() > 1) {
    all.reserve(count);
    size_t ib = 0, ob = in_total;
    for (const HostGateReq *r : batch) {
      auto at = [&](u32 row) { return (u32)(row < r->in_rows ? ib + row : ob + (row - r->in_rows)); };
      for (size_t i = 0; i < r->count; i++) {
        const bfhe_gate &g = r->gates[i];
        all.push_back(bfhe_gate{g.op, at(g.in0), at(g.in1), at(g.out)});
      }
      ib += r->in_rows;
      ob += r->out_rows;
    }
    list = all.data();
  }
  int rc = BFHE_OK;
  size_t ib = 0;
  for (const HostGateReq *r : batch) {
    if (r->in_rows) {
      cudaError_t e = cudaMemcpyAsync(slab + ib * st, r->in_host, r->in_rows * st * 4, cudaMemcpyHostToDevice, c->stream);
      if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync (bfhe_eval_bingate_host inputs)"); break; }
    }
    ib += r->in_rows;
  }
  if (!rc && out_total) {
    cudaError_t e = cudaMemsetAsync(slab + in_total * st, 0, out_total * st * 4, c->stream);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemsetAsync (bfhe_eval_bingate_host outputs)");
  }
  if (!rc) rc = eval_batch_locked(c, slab, list, count, nullptr);
  size_t ob = in_total;
  for (const HostGateReq *r : batch) {
    if (rc) break;
    if (r->out_rows) {
      cudaError_t e = cudaMemcpyAsync(r->out_host, slab + ob * st, r->out_rows * st * 4, cudaMemcpyDeviceToHost, c->stream);
      if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemcpyAsync (bfhe_eval_bingate_host outputs)");
    }
    ob += r->out_rows;
  }
  // also after a failure: nothing may still read or write a caller's buffer once its call returns
  cudaError_t e = cudaStreamSynchronize(c->stream);
  if (!rc && e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize (bfhe_eval_bingate_host)");
  return rc;
}

// with c->q_mtx held: the front of the queue leads the next batch, unless a batch is in flight or the hold is on
static void hand_off(bfhe_ctx *c) {
  if (c->q_busy || c->q_hold || c->q.empty()) return;
  c->q_busy = true;
  c->q.front()->state = HostGateReq::LEAD;
  c->q.front()->cv.notify_one();
}

extern "C" int bfhe_eval_bingate_host(bfhe_ctx *c, const bfhe_gate *gates, size_t count, const uint32_t *in_host, size_t in_rows,
                                      uint32_t *out_host, size_t out_rows) {
  int rc = need_device(c);
  if (rc) return rc;
  if (!gates || !in_host || !out_host) return BFHE_ERR_ARG;
  if ((rc = check_host_call(gates, count, in_rows, out_rows))) return rc;
  HostGateReq req;
  req.gates = gates; req.count = count;
  req.in_host = in_host; req.in_rows = in_rows;
  req.out_host = out_host; req.out_rows = out_rows;
  std::unique_lock<std::mutex> lk(c->q_mtx);
  c->q.push_back(&req);
  hand_off(c);
  while (req.state == HostGateReq::QUEUED) req.cv.wait(lk);
  if (req.state == HostGateReq::LEAD) {
    std::vector<HostGateReq *> batch(c->q.begin(), c->q.end());
    c->q.clear();
    lk.unlock();
    rc = run_host_batch(c, batch);
    const std::string err = rc ? bfhe_last_error() : std::string();
    lk.lock();
    for (HostGateReq *r : batch) { // a waiter returns once it sees DONE, after this lock is released; its request is not touched again
      r->rc = rc;
      r->err = err;
      r->state = HostGateReq::DONE;
      if (r != &req) r->cv.notify_one();
    }
    c->q_busy = false;
    hand_off(c);
  }
  lk.unlock();
  if (req.rc) set_error(req.err); // bfhe_last_error is per thread: every caller of a failed batch gets the message in its own
  return req.rc;
}

extern "C" int bfhe_eval_not_host(const bfhe_ctx *c, const uint32_t *ct_in, size_t count, uint32_t *ct_out) {
  if (!c || !ct_in || !ct_out) return BFHE_ERR_ARG;
  const u32 n = c->p.n, q = c->p.q, st = c->p.ct_stride;
  for (size_t r = 0; r < count; r++) // every row checked before any is written (ct_in == ct_out is allowed)
    for (u32 i = 0; i <= n; i++)
      if (ct_in[r * st + i] >= q) {
        set_error("EvalNOT: input ciphertext row " + std::to_string(r) + " has a word >= q");
        return BFHE_ERR_FORMAT;
      }
  for (size_t r = 0; r < count; r++) { // the words of eval_not_kernel
    const u32 *x = ct_in + r * st;
    u32 *y = ct_out + r * st;
    for (u32 i = 0; i < n; i++) y[i] = (q - x[i]) % q;
    y[n] = (q / 4 + q - x[n]) % q;
    for (u32 i = n + 1; i < st; i++) y[i] = 0;
  }
  return BFHE_OK;
}

// -------------------------------------------------------------------------------------------------
// measurement + debug hooks
// -------------------------------------------------------------------------------------------------
extern "C" int bfhe_profile_enable(bfhe_ctx *c, int on) {
  if (!c) return BFHE_ERR_ARG;
  c->profiling = on != 0;
  return BFHE_OK;
}
extern "C" int bfhe_profile_read(bfhe_ctx *c, int kernel, double *ms, uint64_t *launches) {
  int rc = need_device(c);
  if (rc) return rc;
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  double tot = 0;
  uint64_t cnt = 0;
  std::vector<ProfSpan> keep;
  for (auto &s : c->spans) {
    if (s.kernel != kernel) { keep.push_back(s); continue; }
    float t = 0;
    cudaEventElapsedTime(&t, s.a, s.b);
    tot += t;
    cnt++;
    cudaEventDestroy(s.a);
    cudaEventDestroy(s.b);
  }
  c->spans.swap(keep);
  if (ms) *ms = tot;
  if (launches) *launches = cnt;
  return BFHE_OK;
}
extern "C" int bfhe_microbench_int(bfhe_ctx *c, int which, double *ginstr_per_s) {
  int rc = need_device(c);
  if (rc) return rc;
  DevBuf<u32> sink;
  BFHE_CUDA(sink.alloc(16));
  BFHE_CUDA(cudaMemset(sink.get(), 0x5a, 64));
  DevEvent a, b;
  a.create();
  b.create();
  int threads = 0, ops = 0;
  const int iters = 4096;
  launch_microbench(which, sink.get(), 64, &threads, &ops, c->stream); // warm-up
  cudaEventRecord(a.e, c->stream);
  int r2 = launch_microbench(which, sink.get(), iters, &threads, &ops, c->stream);
  cudaEventRecord(b.e, c->stream);
  if (r2) return cuda_fail((cudaError_t)r2, "microbench");
  BFHE_CUDA(cudaEventSynchronize(b.e));
  float ms = 0;
  cudaEventElapsedTime(&ms, a.e, b.e);
  double per_iter = which == 4 ? 3.0 : 1.0; // the Shoup half-butterfly issues 3 multiply-class instructions
  if (ginstr_per_s) *ginstr_per_s = (double)threads * ops * iters * per_iter / (ms * 1e-3) / 1e9;
  return BFHE_OK;
}

extern "C" int bfhe_dbg_ntt_roundtrip(bfhe_ctx *c, const uint32_t *a, size_t npoly, uint32_t *rt, uint32_t *prod, const uint32_t *b) {
  int rc = need_device(c);
  if (rc) return rc;
  const size_t words = npoly * c->p.N, bytes = words * 4;
  DevBuf<u32> da, db, drt, dpr;
  BFHE_CUDA(da.alloc(words));
  BFHE_CUDA(drt.alloc(words));
  BFHE_CUDA(cudaMemcpy(da.get(), a, bytes, cudaMemcpyHostToDevice));
  if (b) {
    BFHE_CUDA(db.alloc(words));
    BFHE_CUDA(dpr.alloc(words));
    BFHE_CUDA(cudaMemcpy(db.get(), b, bytes, cudaMemcpyHostToDevice));
  }
  int r2 = launch_dbg_ntt(c->P, da.get(), db.get(), drt.get(), dpr.get(), (int)npoly, c->d_twl.get(), c->stream);
  if (r2) return cuda_fail((cudaError_t)r2, "dbg_ntt");
  BFHE_CUDA(cudaStreamSynchronize(c->stream));
  BFHE_CUDA(cudaMemcpy(rt, drt.get(), bytes, cudaMemcpyDeviceToHost));
  if (b) BFHE_CUDA(cudaMemcpy(prod, dpr.get(), bytes, cudaMemcpyDeviceToHost));
  return BFHE_OK;
}

extern "C" int bfhe_dbg_blind_rotate(bfhe_ctx *c, uint32_t *slab, const bfhe_gate *gates, size_t count, uint32_t *acc_host) {
  int rc = need_device(c);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(c->mtx);
  return eval_batch_locked(c, slab, gates, count, acc_host);
}

extern "C" int bfhe_dbg_cluster_limits(bfhe_ctx *c, int *cl2_gates, int *cl4_gates) {
  if (!c || c->device < 0) return BFHE_ERR_ARG;
  BFHE_CUDA(cudaSetDevice(c->device));
  if (cl2_gates) *cl2_gates = cl2_max_gates();
  if (cl4_gates) *cl4_gates = clx_max_gates();
  return BFHE_OK;
}
extern "C" int bfhe_dbg_set_gates_per_cta(bfhe_ctx *c, int g) {
  if (!c) return BFHE_ERR_ARG;
  c->force_g = g;
  return BFHE_OK;
}
extern "C" int bfhe_dbg_hold_batches(bfhe_ctx *c, int hold) {
  if (!c) return BFHE_ERR_ARG;
  std::lock_guard<std::mutex> lk(c->q_mtx);
  const int queued = (int)c->q.size();
  c->q_hold = hold != 0;
  hand_off(c); // release: the front of the queue leads one batch of everything queued
  return queued;
}
