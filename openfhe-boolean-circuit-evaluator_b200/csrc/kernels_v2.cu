// kernels_v2.cu -- the GINX blind rotation of ONE gate on a 2-CTA thread-block cluster, on 16-value / 8-value register tiles
// (STD128_OPT shape: N = 1024, dG = 4, Bg = 2^7; waves of 34..74 gates; data exchanged over DSMEM with st.async + mbarrier).
// Same arithmetic as blind_rotate_kernel in kernels.cu (SURVEY.md 8(a) rows a8-a15; the reference reaches it through
// BinFHEContext::EvalBinGate, src/gate.cpp:133,172,200-202 in /root/reference), a different mapping to the SM.
//
// History (git): this file also held a 16-warp four-gates-per-CTA throughput kernel (two independent pairs of gates per CTA, 16-value
// tiles) and a row-split 4-CTA cluster kernel.  The throughput form never beat kernels.cu's (79.5 k vs 79.0 k gates/s on all-NAND
// batches, 76.7 k vs 77.5 k in bench.py's mix: bound by its per-pair barrier chain, DESIGN.md 5.4) and cost a second 65.8 MB key copy
// on every context; the row-split 4-CTA form (1.17 ms per wave) is superseded by the slot-sliced one in kernels_cl.cu (1.02 ms).  Both
// were removed in round 2.  What remains of the shared machinery: one shared-memory row layout (phys()) that serves 32-bit column,
// 64-bit pair and 128-bit row access conflict-free (tools/smem_layout_check.py), and the 16- / 8-value tile transforms.
#include "device.cuh"
#include <type_traits>

namespace bfhe {
namespace v2 {

constexpr int LOGN = 10, N = 1 << LOGN, DG = 4, LOGBG = 7, ROWS = 2 * DG, NPAD = 512;
constexpr u32 DIGIT_OFF = 64u + (64u << 7) + (64u << 14) + (64u << 21);

// ptxas turns many 2-input adds into IMAD.IADD "to balance the pipes" -- onto the FMA-heavy pipe, the unit that bounds
// this kernel (it counts IMAD.HI as one slot; the hardware takes two).  A 3-input add with a run-time zero stays an IADD3.
__device__ __forceinline__ u32 add3(u32 a, u32 b, u32 z) { return a + b + z; }

// position p of a polynomial (coefficient index going in, bit-reversed evaluation slot coming out) -> word offset in its
// shared-memory row.  Rows of 16 words; 16-byte chunks XOR-swizzled by the row number; row pairs swapped by bit 3 of the row.
__host__ __device__ __forceinline__ int phys(int p) {
  const int T3 = p >> 4, c = (p >> 2) & 3;
  return 16 * (T3 ^ ((T3 >> 3) & 1)) + 4 * (c ^ ((T3 >> 1) & 3)) + (p & 3);
}
__host__ __device__ __forceinline__ int unphys(int o) {
  const int rho = o >> 4, T3 = rho ^ ((rho >> 3) & 1);
  return 16 * T3 + 4 * (((o >> 2) & 3) ^ ((T3 >> 1) & 3)) + (o & 3);
}

// ---- butterfly stages on a 16-register tile -------------------------------------------------------------------------
// Cooley-Tukey, half-sizes TBEG, TBEG/2, ..., TEND; group gi of the stage with half-size t uses twiddle w[16/(2t) + gi].
// No range correction: values grow by 2Q per stage (21Q < 2^32 after all ten).
// Written batch-wise (all high products of a stage, then all low products, then the corrections, then the sums): ptxas keeps
// close to source order inside these very long basic blocks, and butterfly-by-butterfly source order left every instruction
// waiting on its predecessor (profiles/r1_v2_*: 27 % of warp cycles in fixed-latency "wait").
template <int TBEG, int TEND>
__device__ __forceinline__ void ct_stages(u32 (&x)[16], const u32 *__restrict__ w, const u32 *__restrict__ ws, u32 Q, u32 Q2, u32 Z) {
#pragma unroll
  for (int t = TBEG; t >= TEND; t >>= 1) {
    u32 hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { // butterfly i: group gi = i / t, member j = i % t
      const int gi = i / t, b = gi * 2 * t + (i % t) + t, p = 16 / (2 * t) + gi;
      hi[i] = __umulhi(x[b], ws[p]);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int gi = i / t, b = gi * 2 * t + (i % t) + t, p = 16 / (2 * t) + gi;
      lo[i] = x[b] * w[p];
    }
#pragma unroll
    for (int i = 0; i < 8; i++) lo[i] = lo[i] - hi[i] * Q;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int gi = i / t, a = gi * 2 * t + (i % t), b = a + t;
      x[b] = x[a] - lo[i] + Q2;
      x[a] = add3(x[a], lo[i], Z);
    }
  }
}
// Gentleman-Sande, half-sizes T, 2T, ..., TEND.  B = bound of the inputs in units of Q (<= 16).  Sums double per stage and are
// pulled back below 2Q with one lazy Barrett step when they would pass 32Q; differences go through the Shoup multiply.
__host__ __device__ constexpr int gs_bound(int T, int TEND, int B, int MAXOUT) {
  for (; T <= TEND; T *= 2) {
    const int NB = 2 * B;
    B = ((T == TEND) ? NB > MAXOUT : NB > 16) ? 2 : NB;
  }
  return B;
}
template <int T, int TEND, int B, int MAXOUT> struct Gs {
  static constexpr int NB = 2 * B;
  static constexpr bool LAST = (T == TEND);
  static constexpr bool RED = LAST ? (NB > MAXOUT) : (NB > 16);
  static constexpr int OUTB = RED ? 2 : NB;
  __device__ __forceinline__ static void run(u32 (&x)[16], const u32 *__restrict__ w, const u32 *__restrict__ ws, u32 Q, u32 Z) {
    static_assert(B <= 16, "GS input bound too large");
    const u32 off = B * Q;
    u32 D[8], hi[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { // butterfly i: group gi = i / T, member j = i % T
      const int gi = i / T, a = gi * 2 * T + (i % T), b = a + T;
      D[i] = x[a] - x[b] + off;
      const u32 S = add3(x[a], x[b], Z);
      x[a] = RED ? lazy_reduce(S, Q) : S;
    }
#pragma unroll
    for (int i = 0; i < 8; i++) hi[i] = __umulhi(D[i], ws[16 / (2 * T) + i / T]);
#pragma unroll
    for (int i = 0; i < 8; i++) D[i] = D[i] * w[16 / (2 * T) + i / T];
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const int gi = i / T, b = gi * 2 * T + (i % T) + T;
      x[b] = D[i] - hi[i] * Q;
    }
    if constexpr (!LAST) Gs<2 * T, TEND, OUTB, MAXOUT>::run(x, w, ws, Q, Z);
  }
};

// host-side index of twiddle (m groups, group i) in the tables: natural order m + i, except the last stage (m = 512), whose
// groups 8t + j sit at 512 + 256*(j >> 2) + 4t + (j & 3)
struct Tabs { // shared memory
  const u32 *fw, *fws, *iw, *iws;
};

// per-thread twiddles of the middle pass (positions 64u + 8r + 2w + b: stages with 16, 32, 64 groups) and of the narrow
// pass (positions 16*T3 + j: stages with 128, 256, 512 groups), fetched as 32/64/128-bit loads from the natural-order tables
__device__ __forceinline__ void load_tw_mid(const u32 *tab, u32 (&w)[16], int u) {
  w[1] = tab[16 + u];
  const uint2 a = *reinterpret_cast<const uint2 *>(tab + 32 + 2 * u);
  w[2] = a.x; w[3] = a.y;
  const uint4 b = *reinterpret_cast<const uint4 *>(tab + 64 + 4 * u);
  w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}
__device__ __forceinline__ void load_tw_narrow(const u32 *tab, u32 (&w)[16], int T3) {
  const uint2 a = *reinterpret_cast<const uint2 *>(tab + 128 + 2 * T3);
  w[2] = a.x; w[3] = a.y;
  const uint4 b = *reinterpret_cast<const uint4 *>(tab + 256 + 4 * T3);
  w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
  // the 512-group stage is stored de-interleaved (groups 8*T3+0..3 | groups 8*T3+4..7) so both loads are contiguous across lanes
  const uint4 c = *reinterpret_cast<const uint4 *>(tab + 512 + 4 * T3);
  const uint4 d = *reinterpret_cast<const uint4 *>(tab + 768 + 4 * T3);
  w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w; w[12] = d.x; w[13] = d.y; w[14] = d.z; w[15] = d.w;
}
// tile I/O in the three shapes (T = logical thread 0..63 of the polynomial).  Every address is one per-thread base XOR a
// compile-time constant (tools/smem_layout_check.py proves these forms equal phys()).
__device__ __forceinline__ int col_base(int T) { return 16 * (T >> 4) + 4 * (((T >> 2) & 3) ^ (T >> 5)) + (T & 3); }
__device__ __forceinline__ int mid_base(int T) {
  const int u = T >> 2, w = T & 3;
  return 64 * u + 16 * ((u >> 1) & 1) + 8 * (u & 1) + 4 * (w >> 1) + 2 * (w & 1);
}
__device__ __forceinline__ int row_base(int T3) { return 16 * (T3 ^ ((T3 >> 3) & 1)) + 4 * ((T3 >> 1) & 3); }
__device__ __forceinline__ void col_load(const u32 *buf, u32 (&x)[16], int T) { // positions T + 64k
  const int b = col_base(T);
  const u32 *a0 = buf + b, *a1 = buf + (b ^ 8), *a2 = buf + (b ^ 16), *a3 = buf + (b ^ 24);
#pragma unroll
  for (int k = 0; k < 16; k++) x[k] = ((k & 3) == 0 ? a0 : (k & 3) == 1 ? a1 : (k & 3) == 2 ? a2 : a3)[64 * k];
}
__device__ __forceinline__ void col_store(u32 *buf, const u32 (&x)[16], int T) {
  const int b = col_base(T);
  u32 *a0 = buf + b, *a1 = buf + (b ^ 8), *a2 = buf + (b ^ 16), *a3 = buf + (b ^ 24);
#pragma unroll
  for (int k = 0; k < 16; k++) ((k & 3) == 0 ? a0 : (k & 3) == 1 ? a1 : (k & 3) == 2 ? a2 : a3)[64 * k] = x[k];
}
__device__ __forceinline__ constexpr int mid_k(int r) { return 32 * (r >> 2) + 16 * ((r >> 1) & 1) + 8 * (r & 1) + 4 * (r >> 2); }
__device__ __forceinline__ void mid_load(const u32 *buf, u32 (&x)[16], int T) { // positions 64u + 8r + 2w + {0,1}, T = 4u + w
  const int b = mid_base(T);
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const uint2 v = *reinterpret_cast<const uint2 *>(buf + (b ^ mid_k(r)));
    x[2 * r] = v.x; x[2 * r + 1] = v.y;
  }
}
__device__ __forceinline__ void mid_store(u32 *buf, const u32 (&x)[16], int T) {
  const int b = mid_base(T);
#pragma unroll
  for (int r = 0; r < 8; r++) *reinterpret_cast<uint2 *>(buf + (b ^ mid_k(r))) = make_uint2(x[2 * r], x[2 * r + 1]);
}
__device__ __forceinline__ void row_load(const u32 *buf, u32 (&x)[16], int T3) { // positions 16*T3 + j
  const int b = row_base(T3);
#pragma unroll
  for (int c = 0; c < 4; c++) {
    const uint4 v = *reinterpret_cast<const uint4 *>(buf + (b ^ (4 * c)));
    x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
  }
}
__device__ __forceinline__ void row_store(u32 *buf, const u32 (&x)[16], int T3) {
  const int b = row_base(T3);
#pragma unroll
  for (int c = 0; c < 4; c++) *reinterpret_cast<uint4 *>(buf + (b ^ (4 * c))) = make_uint4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
}



// ------------------------------------------------------------------------------------------------------------------
// Latency form on a 2-CTA thread-block cluster: ONE gate on TWO SMs (narrow circuit wavefronts: fewer gates than half the
// SMs, where the time of a level is the latency of one bootstrap -- SHA-256 / MD5, and every circuit once its levels are
// sharded over several GPUs).  CTA r of the cluster owns accumulator component r:
//   inverse transform of product row r -> accumulate -> its four digit transforms (two warps per digit row, one 16-value
//   tile per thread and pass) -> cluster barrier -> external product on ITS half of the evaluation slots (rows of the
//   other component are read from the peer CTA's shared memory over DSMEM; the peer component's product is written into
//   the peer's row) -> cluster barrier.
// Each CTA does exactly half of the arithmetic of a step; per step 2 cluster barriers and 8 KB read + 2 KB written over
// DSMEM.  The CTA's half of the step's key tile (64 KB) is staged by TMA bulk copies behind an mbarrier, issued right after
// the previous product.
// ------------------------------------------------------------------------------------------------------------------
// ---- inverse transform on 8-value tiles by FOUR warps (T = 0..127): three register stages per pass, the widest stage (span 512)
// across lanes 16 apart.  Same row layout; used by the cluster kernel, where the inverse transform of the one product row is the
// serial part of a step.  On return x[k] = coefficient T6 + 64*(k + 8*hi), fully reduced (T6 = 16*warp + lane % 16, hi = lane / 16).
template <int T, int TEND, int B, int MAXOUT> struct Gs8 {
  static constexpr int NB = 2 * B;
  static constexpr bool LAST = (T == TEND);
  static constexpr bool RED = LAST ? (NB > MAXOUT) : (NB > 16);
  static constexpr int OUTB = RED ? 2 : NB;
  __device__ __forceinline__ static void run(u32 (&x)[8], const u32 *__restrict__ w, const u32 *__restrict__ ws, u32 Q, u32 Z) {
    static_assert(B <= 16, "GS input bound too large");
    const u32 off = B * Q;
    u32 D[4], hi[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int gi = i / T, a = gi * 2 * T + (i % T), b = a + T;
      D[i] = x[a] - x[b] + off;
      const u32 S = add3(x[a], x[b], Z);
      x[a] = RED ? lazy_reduce(S, Q) : S;
    }
#pragma unroll
    for (int i = 0; i < 4; i++) hi[i] = __umulhi(D[i], ws[8 / (2 * T) + i / T]);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int gi = i / T, b = gi * 2 * T + (i % T) + T;
      x[b] = D[i] * w[8 / (2 * T) + gi] - hi[i] * Q;
    }
    if constexpr (!LAST) Gs8<2 * T, TEND, OUTB, MAXOUT>::run(x, w, ws, Q, Z);
  }
};
__host__ __device__ constexpr int gs8_bound(int B) { // three stages, sums pulled back when they would pass 16Q going in
  for (int s = 0; s < 3; s++) B = (2 * B > 16) ? 2 : 2 * B;
  return B;
}
template <int B0> __device__ __forceinline__ void ntt_inverse_quad8(u32 (&x)[8], u32 *buf, const DevConst &P, const Tabs &tt, int T, int bar_id, u32 Z) {
  const u32 Q = P.Q;
  u32 w[8], ws[8];
  { // narrow pass: positions 8*T + j, stages with 512, 256, 128 groups
    const int T3 = T >> 1, hb = T & 1, b = row_base(T3);
    const uint4 a0 = *reinterpret_cast<const uint4 *>(buf + (b ^ (8 * hb))), a1 = *reinterpret_cast<const uint4 *>(buf + (b ^ (8 * hb + 4)));
    x[0] = a0.x; x[1] = a0.y; x[2] = a0.z; x[3] = a0.w; x[4] = a1.x; x[5] = a1.y; x[6] = a1.z; x[7] = a1.w;
    const uint4 t4 = *reinterpret_cast<const uint4 *>(tt.iw + 512 + 256 * hb + 4 * T3), t4s = *reinterpret_cast<const uint4 *>(tt.iws + 512 + 256 * hb + 4 * T3);
    const uint2 t2 = *reinterpret_cast<const uint2 *>(tt.iw + 256 + 2 * T), t2s = *reinterpret_cast<const uint2 *>(tt.iws + 256 + 2 * T);
    w[4] = t4.x; w[5] = t4.y; w[6] = t4.z; w[7] = t4.w; ws[4] = t4s.x; ws[5] = t4s.y; ws[6] = t4s.z; ws[7] = t4s.w;
    w[2] = t2.x; w[3] = t2.y; ws[2] = t2s.x; ws[3] = t2s.y;
    w[1] = tt.iw[128 + T]; ws[1] = tt.iws[128 + T];
    Gs8<1, 4, B0, 16>::run(x, w, ws, Q, Z);
    *reinterpret_cast<uint4 *>(buf + (b ^ (8 * hb))) = make_uint4(x[0], x[1], x[2], x[3]);
    *reinterpret_cast<uint4 *>(buf + (b ^ (8 * hb + 4))) = make_uint4(x[4], x[5], x[6], x[7]);
  }
  constexpr int B1 = gs8_bound(B0);
  bar_sync(bar_id, 128);
  { // middle pass: positions 64u + 8r + v, stages with 64, 32, 16 groups
    const int u = T >> 3, v = T & 7;
    const int b = 64 * u + 16 * ((u >> 1) & 1) + 8 * (u & 1) + v; // mid_base with w = v >> 1, plus the low bit of v
    const uint4 t4 = *reinterpret_cast<const uint4 *>(tt.iw + 64 + 4 * u), t4s = *reinterpret_cast<const uint4 *>(tt.iws + 64 + 4 * u);
    const uint2 t2 = *reinterpret_cast<const uint2 *>(tt.iw + 32 + 2 * u), t2s = *reinterpret_cast<const uint2 *>(tt.iws + 32 + 2 * u);
    w[4] = t4.x; w[5] = t4.y; w[6] = t4.z; w[7] = t4.w; ws[4] = t4s.x; ws[5] = t4s.y; ws[6] = t4s.z; ws[7] = t4s.w;
    w[2] = t2.x; w[3] = t2.y; ws[2] = t2s.x; ws[3] = t2s.y;
    w[1] = tt.iw[16 + u]; ws[1] = tt.iws[16 + u];
#pragma unroll
    for (int r = 0; r < 8; r++) x[r] = buf[b ^ mid_k(r)];
    Gs8<1, 4, B1, 16>::run(x, w, ws, Q, Z);
#pragma unroll
    for (int r = 0; r < 8; r++) buf[b ^ mid_k(r)] = x[r];
  }
  constexpr int B2 = gs8_bound(B1);
  bar_sync(bar_id, 128);
  { // wide pass: positions T6 + 64*(k + 8*hi); stages with 8, 4, 2 groups in registers, the last one across lanes
    const int lane = T & 31, hi = lane >> 4, T6 = 16 * (T >> 5) + (lane & 15);
    const int cb = col_base(T6);
    const u32 *a0 = buf + cb, *a1 = buf + (cb ^ 8), *a2 = buf + (cb ^ 16), *a3 = buf + (cb ^ 24);
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = ((k & 3) == 0 ? a0 : (k & 3) == 1 ? a1 : (k & 3) == 2 ? a2 : a3)[64 * (k + 8 * hi)];
#pragma unroll
    for (int g = 0; g < 4; g++) { w[4 + g] = tt.iw[8 + 4 * hi + g]; ws[4 + g] = tt.iws[8 + 4 * hi + g]; }
#pragma unroll
    for (int g = 0; g < 2; g++) { w[2 + g] = tt.iw[4 + 2 * hi + g]; ws[2 + g] = tt.iws[4 + 2 * hi + g]; }
    w[1] = tt.iw[2 + hi]; ws[1] = tt.iws[2 + hi];
    Gs8<1, 4, B2, 16>::run(x, w, ws, Q, Z);
    constexpr int B3 = gs8_bound(B2);
    static_assert(B3 <= 16, "bound");
    const u32 w1 = tt.iw[1], w1s = tt.iws[1], off = B3 * Q;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const u32 o = __shfl_xor_sync(0xffffffffu, x[k], 16);
      const u32 D = o - x[k] + off; // upper lane: (lower - upper) * w
      const u32 m = D * w1 - __umulhi(D, w1s) * Q;
      x[k] = hi ? m : x[k] + o;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = csub(lazy_reduce(x[k], Q), Q);
  }
}

// forward transform of one digit by TWO warps (T = 32*h + lane), one tile per thread and pass
// push_dst != 0: the finished tile (16 consecutive words of the row) is not stored here but sent to the peer CTA at shared::cluster
// address push_dst + 4 * (word offset in the row), counted on the peer's mbarrier push_bar
__device__ __forceinline__ void ntt_forward_split(const u32 *dp, int l, u32 *buf, const DevConst &P, const Tabs &tt, int T, int bar_id, u32 Z,
                                                  u32 push_dst = 0, u32 push_bar = 0) {
  const u32 Q = P.Q, Q2 = P.Q2, qoff = P.Q - (1u << (LOGBG - 1));
  u32 x[16];
#pragma unroll
  for (int k = 0; k < 16; k++) x[k] = ((dp[T + 64 * k] >> (LOGBG * l)) & ((1u << LOGBG) - 1)) + qoff;
  ct_stages<8, 1>(x, P.tw, P.tws, Q, Q2, Z);
  col_store(buf, x, T);
  bar_sync(bar_id, 64);
  {
    u32 w[16], ws[16];
    load_tw_mid(tt.fw, w, T >> 2);
    load_tw_mid(tt.fws, ws, T >> 2);
    mid_load(buf, x, T);
    ct_stages<8, 2>(x, w, ws, Q, Q2, Z);
    mid_store(buf, x, T);
  }
  bar_sync(bar_id, 64);
  {
    u32 w[16], ws[16];
    load_tw_narrow(tt.fw, w, T);
    load_tw_narrow(tt.fws, ws, T);
    row_load(buf, x, T);
    ct_stages<4, 1>(x, w, ws, Q, Q2, Z);
    if (push_dst == 0) row_store(buf, x, T);
    else {
      const int b = row_base(T);
#pragma unroll
      for (int c = 0; c < 4; c++) st_async4(push_dst + 4u * (u32)(b ^ (4 * c)), make_uint4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]), push_bar);
    }
  }
}

struct Cl2Cfg {
  static constexpr int THREADS = 256, HALF = N / 2, KEYPOLYS = 2 * ROWS * 2;
  static constexpr u32 KEYBYTES = (u32)KEYPOLYS * HALF * 4;
  // words: digit rows [DG][N] | peer's digit rows, my slots [DG][HALF] | dp [N] | twiddles [4N] | F [2N] | key tile [KEYPOLYS][HALF];
  // then u16 idx[NPAD]; then three mbarriers (key tile, peer rows, peer product)
  static constexpr size_t words = (size_t)DG * N + (size_t)DG * HALF + N + 4 * N + 2 * N + (size_t)KEYPOLYS * HALF;
  static constexpr size_t smem_bytes = words * 4 + NPAD * 2 + 32;
  static constexpr u32 ROWS_TX = (u32)DG * HALF * 4, PROD_TX = (u32)HALF * 4; // bytes pushed to a CTA per step
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cl2Cfg::THREADS, 1)
blind_rotate_cl2_kernel(const __grid_constant__ DevConst P, const DevGate *__restrict__ gates, int count, const u32 *__restrict__ bk,
                        const u32 *__restrict__ g_tw, const u32 *__restrict__ g_F, u32 *__restrict__ ext, u32 *__restrict__ acc_dbg) {
  constexpr int HALF = Cl2Cfg::HALF, KEYPOLYS = Cl2Cfg::KEYPOLYS;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  u32 *rows = reinterpret_cast<u32 *>(smem_raw);   // [DG][N]: digit l of MY component (only my half of the slots is kept); row 0 doubles as the product row
  u32 *stage = rows + (size_t)DG * N;              // [DG][HALF]: digit l of the PEER's component at my slots, pushed by the peer
  u32 *dp = stage + (size_t)DG * HALF;             // centred accumulator + DIGIT_OFF, natural order
  u32 *s_tw = dp + N;
  u32 *s_F = s_tw + 4 * N;
  u32 *s_key = s_F + 2 * N;                        // [sign][row][cc][HALF]: this CTA's slots of the step's two RGSW ciphertexts
  u16 *s_idx = reinterpret_cast<u16 *>(s_key + (size_t)KEYPOLYS * HALF);
  u64 *s_bar = reinterpret_cast<u64 *>(s_idx + NPAD); // [0] key tile (TMA), [1] peer rows, [2] peer product
  __shared__ u32 s_b, s_zero;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 r = cluster_rank(), peer = r ^ 1u; // r = accumulator component this CTA owns
  const size_t gi = blockIdx.x >> 1;
  const u32 Q = P.Q, q = P.q, n = P.n;
  const DevGate dg = gates[gi];

  if (tid == 0) {
    s_zero = 0;
    mbar_init(s_bar + 0, 1);
    mbar_init(s_bar + 1, 1);
    mbar_init(s_bar + 2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < 4 * N; i += Cl2Cfg::THREADS) s_tw[i] = g_tw[i];
  for (int i = tid; i < 2 * N; i += Cl2Cfg::THREADS) s_F[i] = g_F[i];
  const Tabs tt{s_tw, s_tw + N, s_tw + 2 * N, s_tw + 3 * N};
  { // LWE prep, as in the other kernels (both CTAs of the cluster compute it)
    const u32 gate = dg.op & 0xff;
    for (u32 i = tid; i <= n; i += Cl2Cfg::THREADS) {
      u32 x = dg.in0[i];
      if (dg.op & OP_NEG0) x = (i == n) ? (q / 4 + q - x) % q : (q - x) % q;
      u32 v;
      if (gate == OP_BOOTSTRAP) v = (i == n) ? (x + q / 4) % q : x;
      else {
        u32 y = dg.in1[i];
        if (dg.op & OP_NEG1) y = (i == n) ? (q / 4 + q - y) % q : (q - y) % q;
        v = (gate == OP_XOR_FAST || gate == OP_XNOR_FAST) ? (2 * (x + q - y)) % q : (x + y) % q;
      }
      if (i == n) s_b = v;
      else s_idx[i] = (u16)(((q - v) % q) * P.factor);
    }
  }
  __syncthreads();
  const u32 Z = *(volatile u32 *)&s_zero;
  // key copy of the cluster kernels: [step][quarter of the slots][polynomial][N/4] -- each CTA's 64 KB of a step (two quarters) are
  // contiguous (four 16 KB bulk copies; 32 copies of 2 KB out of the [step][polynomial][N] layout took 2.5 us to land and stalled
  // every step).  The 4-CTA kernel reads one quarter of the same copy, so alternating between the two forms keeps the L2 warm.
  auto issue_keys = [&](u32 step) { // the LAST warp (idle while warps 0-1 run the inverse transform)
    if (lane == 0) mbar_expect_tx(s_bar, Cl2Cfg::KEYBYTES);
    __syncwarp();
    const u32 *src = bk + ((size_t)step * 2 + r) * KEYPOLYS * HALF; // = quarters 2r and 2r + 1 of the [step][quarter][polynomial][N/4] copy
    if (lane < 4) bulk_g2s(s_key + (size_t)lane * 4096, src + (size_t)lane * 4096, 16384, s_bar);
  };
  static_assert(Cl2Cfg::KEYBYTES == 4 * 16384, "four bulk copies");
  if (warp == 7 && n > 0) issue_keys(0);
  { // accumulator init: component 0 = 0, component 1 = test vector
    u32 q1 = 0, q2 = 0, b = 0;
    if (r == 1) {
      const u32 gate = dg.op & 0xff;
      q1 = P.gate_const[gate == OP_BOOTSTRAP ? OP_AND : gate];
      q2 = (q1 + q / 2) % q;
      b = s_b;
    }
    for (u32 idx = tid; idx < (u32)N; idx += Cl2Cfg::THREADS) {
      u32 v = DIGIT_OFF;
      if (r == 1 && idx % P.factor == 0) {
        const u32 t = (b + q - idx / P.factor) % q;
        const bool in = (q1 < q2) ? (t >= q1 && t < q2) : !(t >= q2 && t < q1);
        v = in ? DIGIT_OFF - P.Q8 : DIGIT_OFF + P.Q8;
      }
      dp[idx] = v;
    }
  }
  cluster_sync_all(); // both CTAs' mbarriers are initialised before anything is pushed

  // external product: thread t owns slots (physical words) HALF*r + 2t, +1
  const int o = HALF * (int)r + 2 * tid;
  u32 ex[2];
#pragma unroll
  for (int sl = 0; sl < 2; sl++) ex[sl] = 2 * (__brev((u32)unphys(o + sl)) >> (32 - LOGN)) + 1;
  const u32 peer_row0 = dsmem_addr(rows, peer), peer_stage = dsmem_addr(stage, peer);
  const u32 peer_bar_rows = dsmem_addr(s_bar + 1, peer), peer_bar_prod = dsmem_addr(s_bar + 2, peer);
  const u32 qinv = P.qinv_neg;
  const int h = warp & 1, T = 32 * h + lane; // logical thread of a two-warp transform

  auto close_step = [&]() { // warps 0-3: inverse transform of product row 0 (8-value tiles), accumulate, publish
    u32 x[8];
    ntt_inverse_quad8<2>(x, rows, P, tt, tid, 5, Z);
    const int hi = lane >> 4, T6 = 16 * warp + (lane & 15);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const int j = T6 + 64 * (k + 8 * hi);
      const u32 s = dp[j] + x[k];
      dp[j] = (s >= DIGIT_OFF + (Q >> 1)) ? s - Q : s;
    }
  };

#ifdef BFHE_PHASE_TIMING
  long long tph[5] = {0, 0, 0, 0, 0}, tc0, tc1;
#define PH_T(i) do { tc1 = clock64(); tph[i] += tc1 - tc0; tc0 = tc1; } while (0)
  tc0 = clock64();
#else
#define PH_T(i)
#endif
  // Data moves between the two CTAs as st.async pushes counted on the RECEIVER's mbarrier, so the step loop contains no
  // cluster-scope fence (barrier.cluster.arrive.release alone cost ~1000 cycles per use here).  Order of events, CTA r:
  //   forward transforms: tiles at my slots are stored locally, tiles at the peer's slots are pushed into the peer's stage[]
  //   product: local rows first, then (peer-rows barrier) the staged rows; my component's result -> my row 0, the other
  //   component's -> pushed into the peer's row 0 (those words of the peer's row are dead: the peer pushed them to me before)
  //   inverse transform after the peer-product barrier.
  // WAR safety: the peer overwrites stage[] for step s+1 only after it received my whole product of step s, which every one of my
  // threads pushes after its last read of stage[]; it overwrites my row 0 only after I pushed the words it replaces.
  for (u32 step = 0; step < n; step++) {
    if (step > 0) {
      if (warp < 4) {
        mbar_wait(s_bar + 2, (step - 1) & 1); // the peer's half of my product row has landed
        PH_T(4);
        close_step();
      }
      __syncthreads();
    }
    if (tid == 0) { // this step's expectations (posted after the previous phases completed; early pushes just run the count negative)
      mbar_expect_tx(s_bar + 1, Cl2Cfg::ROWS_TX);
      mbar_expect_tx(s_bar + 2, Cl2Cfg::PROD_TX);
    }
    PH_T(0);
    {
      const int l = warp >> 1;
      const bool mine = (u32)h == r; // warp h finishes the tiles of slot half h
      ntt_forward_split(dp, l, rows + (size_t)l * N, P, tt, T, 1 + l, Z, mine ? 0u : peer_stage + 4u * (u32)(l * HALF) - 4u * (u32)(HALF * (int)peer),
                        peer_bar_rows);
    }
    PH_T(1);
    __syncthreads(); // my halves of my digit rows are visible to all warps of this CTA
    PH_T(2);
    mbar_wait(s_bar, step & 1);
    auto mac = [&](auto RC) {
      constexpr int r = decltype(RC)::value, peer = 1 - r; // compile-time copy of the rank: keeps everything in registers
      const int kq_off = ((2 * tid) >> 8) * KEYPOLYS * (HALF / 2), kq_in = (2 * tid) & (HALF / 2 - 1); // tile = [quarter][polynomial][N/4]
      const u32 m = s_idx[step];
      u32 fp[2], fn[2];
#pragma unroll
      for (int sl = 0; sl < 2; sl++) {
        const u32 y = m * ex[sl], ny = 0u - y;
        fp[sl] = s_F[f_index(y)];
        fn[sl] = s_F[f_index(ny)];
      }
      u64 sp[2][2] = {{0, 0}, {0, 0}}, sn[2][2] = {{0, 0}, {0, 0}}; // [cc][slot]
      // rows of component c sit at row index c + 2l of the RGSW ciphertexts; mine first (local), ...
#pragma unroll
      for (int l = 0; l < DG; l++) {
        const uint2 d = *reinterpret_cast<const uint2 *>(rows + (size_t)l * N + o);
#pragma unroll
        for (int cc = 0; cc < 2; cc++) {
          const uint2 kp = *reinterpret_cast<const uint2 *>(s_key + kq_off + (size_t)((0 * ROWS + 2 * l + r) * 2 + cc) * (HALF / 2) + kq_in);
          const uint2 kn = *reinterpret_cast<const uint2 *>(s_key + kq_off + (size_t)((1 * ROWS + 2 * l + r) * 2 + cc) * (HALF / 2) + kq_in);
          sp[cc][0] += (u64)d.x * kp.x; sp[cc][1] += (u64)d.y * kp.y;
          sn[cc][0] += (u64)d.x * kn.x; sn[cc][1] += (u64)d.y * kn.y;
        }
      }
      mbar_wait(s_bar + 1, step & 1); // ... then the peer's, whose push latency hides behind the local half
#pragma unroll
      for (int l = 0; l < DG; l++) {
        const uint2 d = *reinterpret_cast<const uint2 *>(stage + (size_t)l * HALF + 2 * tid);
#pragma unroll
        for (int cc = 0; cc < 2; cc++) {
          const uint2 kp = *reinterpret_cast<const uint2 *>(s_key + kq_off + (size_t)((0 * ROWS + 2 * l + peer) * 2 + cc) * (HALF / 2) + kq_in);
          const uint2 kn = *reinterpret_cast<const uint2 *>(s_key + kq_off + (size_t)((1 * ROWS + 2 * l + peer) * 2 + cc) * (HALF / 2) + kq_in);
          sp[cc][0] += (u64)d.x * kp.x; sp[cc][1] += (u64)d.y * kp.y;
          sn[cc][0] += (u64)d.x * kn.x; sn[cc][1] += (u64)d.y * kn.y;
        }
      }
      uint2 out[2];
#pragma unroll
      for (int cc = 0; cc < 2; cc++) {
        out[cc].x = redc((u64)redc(sp[cc][0], Q, qinv) * fp[0] + (u64)redc(sn[cc][0], Q, qinv) * fn[0], Q, qinv);
        out[cc].y = redc((u64)redc(sp[cc][1], Q, qinv) * fp[1] + (u64)redc(sn[cc][1], Q, qinv) * fn[1], Q, qinv);
      }
      // my component's product stays here (row 0, my slots); the other component's goes into the peer's row 0 (my slots)
      *reinterpret_cast<uint2 *>(rows + o) = out[r];
      st_async2(peer_row0 + (u32)(o * 4), out[peer], peer_bar_prod);
    };
    if (r == 0) mac(std::integral_constant<int, 0>{});
    else mac(std::integral_constant<int, 1>{});
    PH_T(3);
    __syncthreads(); // row 0 (my half) visible to warps 0-1; nobody reads the key tile any more
    PH_T(4);
    if (warp == 7 && step + 1 < n) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // generic-proxy reads of the tile above, async-proxy writes below
      issue_keys(step + 1);
    }
  }

  // ---- epilogue: last inverse transform, sample extraction (a14) and ModSwitch Q -> qKS (a15) ----
  if (n > 0 && warp < 4) {
    mbar_wait(s_bar + 2, (n - 1) & 1);
    close_step();
  }
  __syncthreads();
  u32 *e = ext + gi * (N + 4);
  const u64 qKS = P.qKS;
  for (u32 j = tid; j < (u32)N; j += Cl2Cfg::THREADS) {
    u32 a = dp[j] - DIGIT_OFF;
    a += ((int)a < 0) ? Q : 0u;
    if (acc_dbg) acc_dbg[(gi * 2 + r) * N + j] = a;
    if (r == 0) {
      const u32 v = (j == 0) ? a : (a == 0 ? 0 : Q - a); // Transpose: a'_0 = a_0, a'_k = -a_{N-k}
      e[(j == 0) ? 0 : N - j] = (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS);
    } else if (j == 0) {
      const u32 v = csub(a + P.Q8, Q);
      e[N] = (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS);
    }
  }
#ifdef BFHE_PHASE_TIMING
  if (acc_dbg && lane == 0 && (warp == 0 || warp == 7))
    for (int i = 0; i < 5; i++) acc_dbg[(gi * 2 + r) * N + 32 + 8 * (warp == 7) + i] = (u32)(tph[i] / 1000); // kilo-cycles
#endif
  cluster_sync_all(); // a CTA must not exit while its peer may still push into its shared memory
}

// key copy of the cluster kernels: [step][polynomial][N] -> [step][quarter][polynomial][N/4]
__global__ void bk_split_cl4_kernel(const u32 *__restrict__ src, u32 *__restrict__ dst, size_t nsteps) {
  constexpr int KP = Cl2Cfg::KEYPOLYS, QUARTER = N / 4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nsteps * KP * N; i += (size_t)gridDim.x * blockDim.x) {
    const size_t step = i / ((size_t)KP * N), rem = i % ((size_t)KP * N);
    const int pl = (int)(rem / N), o = (int)(rem % N), rk = o / QUARTER;
    dst[((step * 4 + rk) * KP + pl) * QUARTER + (o % QUARTER)] = src[i];
  }
}

// bootstrapping key: [chunk][lane][4] order of kernels.cu -> physical row order of this kernel (word phys(p) = slot p)
__global__ void bk_permute_v2_kernel(const u32 *__restrict__ src, u32 *__restrict__ dst, size_t npoly) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npoly * N; i += (size_t)gridDim.x * blockDim.x) {
    const size_t poly = i / N;
    const int p = (int)(i % N), t = p >> 5, j = p & 31;
    dst[poly * N + phys(p)] = src[poly * N + ((j >> 2) * 32 + t) * 4 + (j & 3)];
  }
}

} // namespace v2

bool cl2_supported(const DevConst &P, int method_ap) {
  return !method_ap && P.N == 1024 && P.dG == 4 && P.logBG == 7 && P.Q == SOLINAS_Q && P.n <= (u32)v2::NPAD;
}
int v2_set_attrs() {
  return (int)cudaFuncSetAttribute(v2::blind_rotate_cl2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v2::Cl2Cfg::smem_bytes);
}
static int v2_attrs_once() {
  static bool done[64];
  return once_per_device(done, v2_set_attrs);
}
int launch_bk_split_cl4(const u32 *d_src, u32 *d_dst, size_t npoly, void *stream) {
  if (npoly == 0) return 0;
  v2::bk_split_cl4_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_src, d_dst, npoly / v2::Cl2Cfg::KEYPOLYS);
  return (int)cudaGetLastError();
}
// how many gates the cluster form runs at once (2-CTA clusters must sit inside one GPC, so this can be less than SMs / 2); queried once
// per device, a 0 included
int cl2_max_gates() {
  static bool have[64];
  static int gates[64];
  const int d = device_slot();
  once_per_device(have, [&] {
    gates[d] = v2_attrs_once() ? 0 : max_active_clusters(v2::blind_rotate_cl2_kernel, 2, v2::Cl2Cfg::THREADS, v2::Cl2Cfg::smem_bytes);
    return cudaSuccess;
  });
  return gates[d];
}
int launch_blind_rotate_cl2(const DevConst &P, const DevGate *d_gates, int count, const DevKeys &k, u32 *d_ext, u32 *d_acc_dbg, void *stream) {
  if (count <= 0) return 0;
  if (int rc = v2_attrs_once()) return rc;
  v2::blind_rotate_cl2_kernel<<<2 * count, v2::Cl2Cfg::THREADS, v2::Cl2Cfg::smem_bytes, (cudaStream_t)stream>>>(P, d_gates, count, k.bk4, k.tw2, k.F,
                                                                                                         d_ext, d_acc_dbg);
  return (int)cudaGetLastError();
}
int launch_bk_permute_v2(const u32 *d_src, u32 *d_dst, size_t npoly, void *stream) {
  if (npoly == 0) return 0;
  v2::bk_permute_v2_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_src, d_dst, npoly);
  return (int)cudaGetLastError();
}
} // namespace bfhe
