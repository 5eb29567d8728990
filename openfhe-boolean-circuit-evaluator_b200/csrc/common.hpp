// common.hpp -- types shared between the host engine and the sm_100a kernels.
#pragma once
#include <cstddef>
#include <cstdint>

namespace bfhe {

using u8 = uint8_t;
using u16 = uint16_t;
using u32 = uint32_t;
using u64 = uint64_t;
using i32 = int32_t;
using i64 = int64_t;

// Passed to every kernel as a __grid_constant__ parameter: lands in the constant bank, so the
// compile-time-indexed "uniform" twiddles below become immediate-like operands of IMAD.
struct DevConst {
  u32 Q, Q2;       // ring modulus (2^26 < Q < 2^27) and 2Q
  u32 qinv_neg;    // -Q^-1 mod 2^32 (Montgomery)
  u32 unused_mu;   // unused, like reserved_ below
  u32 oneM;        // 2^32 mod Q  (Montgomery form of 1)
  u32 Q8;          // Q/8 + 1
  u32 n, N, q, factor; // LWE dim, ring dim, LWE modulus, 2N/q
  u32 qKS, baseKS, dKS;
  u32 baseR, dR, dG, logBG;
  u32 ct_stride;
  u32 ninv, ninvs; // N^-1 mod Q and its Shoup companion (debug kernels only)
  u32 nM, nMs;     // N^-1 * 2^32 mod Q (+Shoup): coefficient-form key -> device form
  u32 gate_const[9];
  u32 reserved_[3]; // unused: with unused_mu they keep tw[] / itw[] at their constant-bank offsets, which decide ptxas's vector constant loads
  // psi^bitrev(k), k in [1,32): the twiddles of every NTT stage whose butterflies span >= 32 indices.
  u32 tw[32], tws[32], itw[32], itws[32];
};

// one gate as the kernels see it (built on the host from bfhe_gate)
struct DevGate {
  const u32 *in0;
  const u32 *in1;
  u32 *out;
  u32 op;
  u32 pad;
};

enum : u32 { OP_OR = 0, OP_AND = 1, OP_NOR = 2, OP_NAND = 3, OP_XOR_FAST = 4, OP_XNOR_FAST = 5, OP_XOR = 6, OP_XNOR = 7,
             OP_BOOTSTRAP = 8, OP_NEG0 = 0x100, OP_NEG1 = 0x200 };

// blind-rotation kernel forms; the values are the ones the test hook bfhe_dbg_set_gates_per_cta takes (THRn: n gates per CTA)
enum class Form : int {
  AUTO = 0,  // the launch's own choice by gate count
  THR1 = 1,  // throughput form, 1, 2 or 4 gates per CTA
  THR2 = 2,
  THR4 = 4,
  LAT = 8,   // latency form: one gate per CTA, TMA-staged key
  CL2 = 32,  // one gate on a 2-CTA cluster (kernels_v2.cu)
  CL4 = 128, // one gate on a 4-CTA cluster, slot-sliced (kernels_cl.cu)
};
// whether this parameter set has the form (parameters only: a circuit plans before the keys are on the device).  AUTO: some form exists.
bool form_supported(const DevConst &P, int method_ap, Form f);

// the device key set: everything the blind rotation and the key switch read.  A view; bfhe_ctx owns the buffers.  Null where the parameter
// set has no use for a copy, and the key copies are null until the keys are uploaded.
struct DevKeys {
  const u32 *bk = nullptr;   // bootstrapping key in device form (bk_convert)
  const u32 *bkf = nullptr;  // GINX throughput kernel at the STD128_OPT shape: bk with the top digit folded in (launch_bk_fold)
  const u32 *bk4 = nullptr;  // 2-CTA cluster form: bk rows in kernels_v2.cu's physical slot order, split [step][quarter of the slots][polynomial][N/4]
  const u32 *bkx = nullptr;  // 4-CTA cluster form (kernels_cl.cu): bk as [step][rank][polynomial][N/4]
  const u32 *twl = nullptr;  // fwd w | fwd ws | inv w | inv ws, each N words: per-lane twiddles of the narrow pass
  const u32 *psiM = nullptr; // psi^k in Montgomery form, k < 2N
  const u32 *tw2 = nullptr;  // 2-CTA cluster form: fwd w | fwd ws | inv w | inv ws, each N words (order: kernels_v2.cu Tabs)
  const u32 *F = nullptr;    // (psi^k - 1) * 2^32 mod Q, k < 2N: read by the 2-CTA form and by the GINX 4-CTA form
  const u32 *twx = nullptr;  // 4-CTA cluster form: its per-rank twiddle blocks
  const void *ksk = nullptr; // key-switching key, [i][digit][digit value][row], ksk_elem_bytes per element
  int ksk_elem_bytes = 4;
};

// kernels.cu entry points (all asynchronous on `stream`; return cudaError_t as int).  A form this parameter set lacks: cudaErrorInvalidValue.
int launch_blind_rotate(const DevConst &P, int method_ap, const DevGate *d_gates, int count, const DevKeys &keys,
                        u32 *d_ext /*count * (N+4)*/, u32 *d_acc_dbg /*nullable: count*2*N*/, Form form, void *stream);
// kernels_v2.cu
bool cl2_supported(const DevConst &P, int method_ap); // parameters of the 2-CTA cluster form
int v2_set_attrs();
int launch_bk_permute_v2(const u32 *d_src, u32 *d_dst, size_t npoly, void *stream);
int cl2_max_gates(); // gates the cluster form can run concurrently on this device (0 = unavailable)
int launch_bk_split_cl4(const u32 *d_src, u32 *d_dst, size_t npoly, void *stream);
// one gate on a 2-CTA cluster (two SMs): the latency form for wavefronts narrower than half the SM count
int launch_blind_rotate_cl2(const DevConst &P, const DevGate *d_gates, int count, const DevKeys &keys, u32 *d_ext, u32 *d_acc_dbg,
                            void *stream);
// kernels_cl.cu: one gate on a 4-CTA cluster, everything sliced by evaluation slot, one exchange per step
bool clx_supported(const DevConst &P, int method_ap);
size_t clx_tw_words();
int clx_set_attrs();
int clx_max_gates();  // 4-CTA clusters the device keeps co-resident
int clx_fast_gates(); // up to this many gates the 4-CTA form runs all clusters in one round at full speed
int launch_bk_slice_clx(const u32 *d_src, u32 *d_dst, size_t npoly, int method_ap, void *stream);
int launch_blind_rotate_clx(const DevConst &P, int method_ap, const DevGate *d_gates, int count, const DevKeys &keys, u32 *d_ext,
                            u32 *d_acc_dbg, void *stream);
// Multi-GPU exchange fused into the key switch (SURVEY 8(e)): every output ciphertext is stored into every rank's wire slab (the peers'
// slabs are mapped through CUDA IPC, the stores travel over NVLink), and the last CTA of the launch raises this rank's flag in every
// peer's flag array.  Flag values only grow: value(epoch, index) = epoch * per_epoch + index + 1, `epoch` read from device memory so
// that the launches can sit in a CUDA graph.  slabs == nullptr: single-GPU behaviour.
struct PeerX {
  u32 *const *slabs = nullptr; // [world] slab base of every rank as mapped HERE (own entry = local slab)
  const u32 *local_base = nullptr;
  u32 *const *flags = nullptr; // [world] flag array (u32[world]) of every rank as mapped here
  u32 *counter = nullptr;      // local: CTAs of this launch that have finished their stores
  const u32 *epoch = nullptr;  // local: Clock() count
  u32 world = 1, rank = 0, index = 0, per_epoch = 1;
};
int launch_keyswitch(const DevConst &P, const u32 *d_ext, const DevGate *d_gates, int count, const DevKeys &keys, void *stream,
                     const PeerX *px = nullptr);
// exchange plumbing (one tiny launch each): epoch += 1; wait until every peer's flag has reached value(epoch, index) -- index -1 = the
// end-of-Clock signal of the previous epoch -- with a timeout (30 s, BFHE_EXCHANGE_TIMEOUT_S) that sets *err instead of hanging; raise my flag at every peer
int launch_peer_epoch_bump(u32 *epoch, void *stream);
int launch_peer_wait(const u32 *local_flags, const u32 *epoch, u32 world, u32 rank, int index, u32 per_epoch, u32 *err, void *stream);
int launch_peer_signal(const PeerX &px, void *stream);
int launch_eval_not(const DevConst &P, const u32 *const *d_in, u32 *const *d_out, int count, void *stream);
// count rows of ct_stride words from outside the program: zero the padding words, atomicMin the index of every row holding a word >= q
// into *d_bad_row
int launch_ct_ingest(const DevConst &P, u32 *d_rows, int count, u32 *d_bad_row, void *stream);
int launch_bk_convert(const DevConst &P, const u32 *d_coef, u32 *d_dev, size_t npoly, const u32 *d_twl, void *stream);
// key copy of the GINX throughput kernel at the STD128_OPT shape (N 1024, dG 4, base 2^7): the device-form key with its top digit row folded
// into the others (kernels.cu bk_fold_kernel); nsteps = n
bool bk_fold_supported(const DevConst &P, int method_ap);
int launch_bk_fold(const DevConst &P, const u32 *d_bk, u32 *d_bkf, size_t nsteps, void *stream);
// key_expand.cu: the public masks of a compact key blob (include/bfhe.h) from its 256-bit mask seed.  KSK mask row r has ChaCha20 stream id r,
// BK mask polynomial p (the p-th column-0 polynomial of the BFHEKEY1 order) has stream id BK_MASK_STREAM + p.
struct MaskKey {
  u32 k[8];
};
constexpr u64 BK_MASK_STREAM = 1ull << 40;
// the device KSK ([i][k][j][rowlen], as ensure_device_keys lays it out) from the bodies ([N][baseKS][dKS], elem_bytes each)
int launch_ksk_expand(const MaskKey &key, const void *d_bodies, void *d_ksk, int elem_bytes, u32 N, u32 baseKS, u32 dKS, u32 n, u32 rowlen,
                      u32 qKS, void *stream);
// `count` fresh ciphertext rows (stride words, 16-byte aligned) of a compact blob: row g is mask row g mod q, body d_bodies[g]; the
// same kernel as launch_ksk_expand with baseKS = dKS = 1
int launch_ct_expand(const MaskKey &key, const u32 *d_bodies, u32 *d_rows, size_t count, u32 n, u32 stride, u32 q, void *stream);
// `pairs` (mask, body) polynomial pairs of the coefficient-form BK, starting at mask polynomial p_first, into d_stage (2 * pairs * N words)
int launch_bk_mask_expand(const MaskKey &key, const u32 *d_bodies, u32 *d_stage, u64 p_first, size_t pairs, u32 N, u32 Q, void *stream);
int launch_dbg_ntt(const DevConst &P, const u32 *d_a, const u32 *d_b, u32 *d_rt, u32 *d_prod, int npoly, const u32 *d_twl,
                   void *stream);
int launch_microbench(int which, u32 *d_sink, int iters, int *threads_total, int *ops_per_thread_iter, void *stream);
int blind_rotate_set_attrs();

} // namespace bfhe
