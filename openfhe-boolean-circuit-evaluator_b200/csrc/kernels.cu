// kernels.cu -- hand-written sm_100a kernels for the gate-bootstrapping hot path.
//
// Replaces the arithmetic the reference reaches through lbcrypto::BinFHEContext::EvalBinGate /
// Bootstrap / EvalNOT (src/gate.cpp:112,133,172,198-202 in /root/reference); stage list in
// SURVEY.md 8(a) rows a8-a17.  Design notes (DESIGN.md has the full story):
//
//  * One warp owns one ring polynomial.  A size-N negacyclic NTT is two register passes of
//    E = N/32 points per thread with ONE shared-memory transpose between them (plus one
//    warp-shuffle butterfly stage when log2 N is odd).  No __syncthreads inside a transform.
//  * Pass "wide" (butterfly span >= 32) uses twiddles that are uniform across the warp: they sit in
//    the kernel-parameter constant bank and are consumed as constant operands by IMAD.
//    Pass "narrow" (span < 32) uses 31 per-lane twiddles read as conflict-free LDS.128.
//  * Arithmetic: 32-bit Shoup butterflies with lazy ranges (Q < 2^27, so the forward transform needs no
//    correction at all: values grow by 2Q per stage and stay below 2^32); the RGSW x RLWE
//    external product accumulates 2*dG 32x32->64 products per slot in one IMAD.WIDE chain and
//    Montgomery-reduces once (keys are stored pre-multiplied by 2^32 * N^-1).
//  * The throughput kernel keeps the accumulator in EVALUATION form only, as N^-1 * NTT(acc) in shared
//    memory, updated by the external product: each step is INTT (= the accumulator) -> signed digit
//    decomposition -> dG forward NTTs, all in registers of the warp that owns the polynomial (dG - 1 for
//    STD128_OPT GINX, whose top digit is folded into a key copy).
//  * A CTA carries G gates through the n blind-rotation steps in lock step so that every
//    bootstrapping-key word loaded from L2 is reused G times from registers (GINX).
#include "device.cuh"
#include <type_traits>
#include <cuda_runtime.h>
#include <cstdlib>

namespace bfhe {

// Masks of the latency kernel's forward transform: bit i = stage i of the pass (wide: span >= 32, narrow: span < 32) computes the t*Q term
// of its Shoup multiplies on the ALU pipe (mul_shoup<true>), the other stages on the FMA-heavy pipe; tuned with tools/perf_lat.py /
// phase_timing.py.  Every other transform uses the IMAD form: the throughput kernel is bound by instruction issue under dependency latency
// at two warps per scheduler, where one IMAD beats three ALU instructions (DESIGN.md 5.4, profiles/r2_sol_variants.md).
constexpr int SOL_LAT_WIDE = 0x05, SOL_LAT_NARROW = 0x0a;

// ------------------------------------------------------------------------------------------
// shared-memory polynomial layout: row t' (the E consecutive indices owned by lane t' in the narrow
// pass) is E words; its 16-byte chunks are XOR-swizzled so that both the row access (LDS.128 by the
// owning lane) and the column access (LDS.32 of index lane+32k by all lanes) are conflict free.
// ------------------------------------------------------------------------------------------
// position of entry u of the monomial-factor table: the low five bits are folded with the next five
__device__ __forceinline__ u32 f_phys(u32 u) { return (u & ~31u) | ((u ^ (u >> 5)) & 31u); }
template <int E> struct Lay {
  static constexpr int C = E / 4;
  __device__ __forceinline__ static int swz(int tp) { return E == 32 ? (tp & 7) : ((tp >> 1) & 3); }
  __device__ __forceinline__ static int chunk_off(int tp, int c) { return E * tp + 4 * (c ^ swz(tp)); }
  __device__ __forceinline__ static int elem_off(int k, int lane) { // index lane + 32k
    if (E == 32) return 32 * k + 4 * ((lane >> 2) ^ (k & 7)) + (lane & 3);
    int j = lane & 15;
    return 16 * (2 * k + (lane >> 4)) + 4 * ((j >> 2) ^ (k & 3)) + (j & 3);
  }
};
template <int E> __device__ __forceinline__ void row_load(const u32 *buf, u32 (&x)[E], int lane) {
#pragma unroll
  for (int c = 0; c < E / 4; c++) {
    uint4 v = *reinterpret_cast<const uint4 *>(buf + Lay<E>::chunk_off(lane, c));
    x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
  }
}
template <int E> __device__ __forceinline__ void row_store(u32 *buf, const u32 (&x)[E], int lane) {
#pragma unroll
  for (int c = 0; c < E / 4; c++)
    *reinterpret_cast<uint4 *>(buf + Lay<E>::chunk_off(lane, c)) = make_uint4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
}
template <int E> __device__ __forceinline__ void col_load(const u32 *buf, u32 (&x)[E], int lane) {
#pragma unroll
  for (int k = 0; k < E; k++) x[k] = buf[Lay<E>::elem_off(k, lane)];
}
template <int E> __device__ __forceinline__ void col_store(u32 *buf, const u32 (&x)[E], int lane) {
#pragma unroll
  for (int k = 0; k < E; k++) buf[Lay<E>::elem_off(k, lane)] = x[k];
}

// ------------------------------------------------------------------------------------------
// in-register passes.  The E-point sub-transform has the same shape in both passes: stage with
// half-size t has E/(2t) groups, group gi uses twiddle number p = E/(2t) + gi of the pass's table.
// ------------------------------------------------------------------------------------------
// Cooley-Tukey (forward).  No range correction: x + T and x - T + 2Q grow by 2Q per stage.
// UNI: twiddles uniform over the warp (kernel parameters).  Otherwise the per-lane twiddles (smem table [C][32] of uint4, entry p of
// lane t' = psi^br(m+i)) are read chunk by chunk as the stages need them (at most 8 registers live) instead of being preloaded into
// 2*E registers -- what lets 12 warps per SM fit the register file.
// SOLMASK: bit i = stage i uses mul_shoup<true>.
__device__ __forceinline__ u32 comp4(const uint4 &v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
// PRE: the products of the FIRST stage arrive precomputed in pre[0 .. E/2) (digit transforms: twiddle * small digit comes
// from a 128-entry table, see blind_rotate_kernel), x[E/2 ..) is not read.
template <int E, bool UNI, int SOLMASK = 0, bool PRE = false>
__device__ __forceinline__ void ct_pass(u32 (&x)[E], const u32 *__restrict__ utw, const u32 *__restrict__ utws, u32 Q, u32 Q2,
                                        const u32 *tab = nullptr, const u32 *tabs = nullptr, int lane = 0, const u32 *pre = nullptr) {
  int si = 0;
  uint4 cw = make_uint4(0, 0, 0, 0), cws = cw;
#pragma unroll
  for (int t = E / 2; t >= 1; t >>= 1, si++) {
    const bool sol = (SOLMASK >> si) & 1;
#pragma unroll
    for (int gi = 0; gi < E / (2 * t); gi++) {
      const int p = E / (2 * t) + gi;
      u32 ww, wws;
      if (UNI) { ww = utw[p]; wws = utws[p]; }
      else {
        if ((p & 3) == 0 || gi == 0) {
          cw = reinterpret_cast<const uint4 *>(tab)[(p >> 2) * 32 + lane];
          cws = reinterpret_cast<const uint4 *>(tabs)[(p >> 2) * 32 + lane];
        }
        ww = comp4(cw, p & 3); wws = comp4(cws, p & 3);
      }
#pragma unroll
      for (int j = 0; j < t; j++) {
        const int a = gi * 2 * t + j, b = a + t;
        u32 T;
        if (PRE && si == 0) T = pre[j];
        else T = sol ? mul_shoup<true>(x[b], ww, wws, Q) : mul_shoup<false>(x[b], ww, wws, Q);
        x[b] = x[a] - T + Q2;
        x[a] = x[a] + T;
      }
    }
  }
}

// Gentleman-Sande (inverse, unscaled).  B = bound of the inputs in units of Q (<= 16).  Sums double
// per stage; when they would pass 32Q (= just under 2^32) they are pulled back below 2Q with one
// lazy Barrett step.  Differences go through the Shoup multiply, which accepts any 32-bit input.
// Twiddles as in ct_pass.
template <int E, int T, int B, bool UNI, int MAXLAST> struct GsRun {
  static constexpr int NB = 2 * B;
  static constexpr bool LAST = (2 * T >= E);
  static constexpr bool RED = LAST ? (NB > MAXLAST) : (NB > 16); // pull the sums back below 2Q after this stage?
  static constexpr int OUTB = RED ? 2 : NB;
  __device__ __forceinline__ static void run(u32 (&x)[E], const u32 *__restrict__ utw, const u32 *__restrict__ utws, u32 Q,
                                             const u32 *tab = nullptr, const u32 *tabs = nullptr, int lane = 0) {
    static_assert(B <= 16, "GS input bound too large");
    const u32 off = B * Q;
    uint4 cw = make_uint4(0, 0, 0, 0), cws = cw;
#pragma unroll
    for (int gi = 0; gi < E / (2 * T); gi++) {
      const int p = E / (2 * T) + gi;
      u32 ww, wws;
      if (UNI) { ww = utw[p]; wws = utws[p]; }
      else {
        if ((p & 3) == 0 || gi == 0) {
          cw = reinterpret_cast<const uint4 *>(tab)[(p >> 2) * 32 + lane];
          cws = reinterpret_cast<const uint4 *>(tabs)[(p >> 2) * 32 + lane];
        }
        ww = comp4(cw, p & 3); wws = comp4(cws, p & 3);
      }
#pragma unroll
      for (int j = 0; j < T; j++) {
        const int a = gi * 2 * T + j, b = a + T;
        u32 S = x[a] + x[b];
        u32 D = x[a] - x[b] + off;
        x[b] = mul_shoup(D, ww, wws, Q);
        x[a] = RED ? lazy_reduce(S, Q) : S;
      }
    }
    if constexpr (!LAST) GsRun<E, 2 * T, OUTB, UNI, MAXLAST>::run(x, utw, utws, Q, tab, tabs, lane);
  }
};
// bound (in units of Q) of the values GsRun<E,1,B0,*,MAXLAST> leaves behind
__host__ __device__ constexpr int gs_out_bound(int E, int B0, int MAXLAST) {
  int B = B0;
  for (int T = 1; T < E; T *= 2) {
    const int NB = 2 * B;
    const bool last = 2 * T >= E;
    B = (last ? NB > MAXLAST : NB > 16) ? 2 : NB;
  }
  return B;
}

// ------------------------------------------------------------------------------------------
// whole transforms (one warp, E values per lane)
// ------------------------------------------------------------------------------------------
struct TwTabs { // shared-memory per-lane twiddle tables, each N words
  const u32 *fw, *fws, *iw, *iws;
};

// forward: x in column layout (index lane+32k, coefficient form, values < Q) -> row layout (index E*lane+j,
// evaluation form, lazy < (2*logN+1)Q).  buf: N-word smem scratch, left holding garbage.  SOLW / SOLN: SOLMASK of the wide / narrow pass.
template <int LOGN, bool PRE = false, int SOLW = 0, int SOLN = 0>
__device__ __forceinline__ void ntt_forward(u32 (&x)[(1 << LOGN) / 32], u32 *buf, const DevConst &P, const TwTabs &tt, int lane,
                                            const u32 *pre = nullptr) {
  constexpr int E = (1 << LOGN) / 32;
  const u32 Q = P.Q, Q2 = P.Q2;
  ct_pass<E, true, SOLW, PRE>(x, P.tw, P.tws, Q, Q2, nullptr, nullptr, 0, pre);
  if constexpr (LOGN & 1) { // span-16 stage across lanes (lane bit 4): group index = k, twiddle psi_br[16+k]
    const bool up = lane & 16;
#pragma unroll
    for (int k = 0; k < E; k++) {
      u32 v = up ? mul_shoup(x[k], P.tw[16 + k], P.tws[16 + k], Q) : x[k];
      u32 o = __shfl_xor_sync(0xffffffffu, v, 16);
      x[k] = up ? (o - v + Q2) : (v + o);
    }
  }
  __syncwarp();
  col_store<E>(buf, x, lane);
  __syncwarp();
  row_load<E>(buf, x, lane);
  ct_pass<E, false, SOLN>(x, P.tw, P.tws, Q, Q2, tt.fw, tt.fws, lane);
}

// inverse (unscaled: N * true value; the keys carry N^-1): x in row layout (evaluation form, values < B0*Q)
// -> column layout, coefficient form, fully reduced to [0,Q).
template <int LOGN, int B0>
__device__ __forceinline__ void ntt_inverse(u32 (&x)[(1 << LOGN) / 32], u32 *buf, const DevConst &P, const TwTabs &tt, int lane) {
  constexpr int E = (1 << LOGN) / 32;
  const u32 Q = P.Q;
  constexpr int ML = (LOGN & 1) ? 8 : 16; // what the next stage can take
  GsRun<E, 1, B0, false, ML>::run(x, P.itw, P.itws, Q, tt.iw, tt.iws, lane);
  constexpr int B1 = gs_out_bound(E, B0, ML);
  __syncwarp();
  row_store<E>(buf, x, lane);
  __syncwarp();
  col_load<E>(buf, x, lane);
  if constexpr (LOGN & 1) {
    static_assert(B1 <= 8, "bound");
    const bool up = lane & 16;
    const u32 off = B1 * Q;
#pragma unroll
    for (int k = 0; k < E; k++) {
      u32 o = __shfl_xor_sync(0xffffffffu, x[k], 16);
      // lower lane: U + V ; upper lane: (U - V) * w
      u32 D = o - x[k] + off;
      x[k] = up ? mul_shoup(D, P.itw[16 + k], P.itws[16 + k], Q) : (x[k] + o);
    }
    constexpr int B2 = 2 * B1;
    GsRun<E, 1, B2, true, 32>::run(x, P.itw, P.itws, Q);
  } else {
    GsRun<E, 1, B1, true, 32>::run(x, P.itw, P.itws, Q);
  }
#pragma unroll
  for (int k = 0; k < E; k++) x[k] = csub(lazy_reduce(x[k], Q), Q);
}

// ------------------------------------------------------------------------------------------
// blind rotation
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 brev(u32 x, int bits) { return __brev(x) >> (32 - bits); }
template <int DG, int LOGBG> constexpr u32 digit_offset() { // (B/2) * (1 + B + ... + B^(DG-1))
  u32 off = 0;
  for (int l = 0; l < DG; l++) off += (1u << (LOGBG - 1)) << (LOGBG * l);
  return off;
}

template <int LOGN, int DG, int LOGBG, int G, bool AP> struct BrCfg {
  static constexpr int N = 1 << LOGN, E = N / 32, C = E / 4, ROWS = 2 * DG; // ROWS: key rows per sign = dct rows the product multiplies
  static constexpr int W = 2 * G, THREADS = 32 * W;
  static constexpr int NPAD = AP ? 1024 : 512; // per-gate index table (>= n*dR for AP, >= n for GINX)
  // first-stage product table: twiddle * (digit - B/2) mod Q for the 2^LOGBG digit values, one copy per bank (STD128_OPT shape only)
  static constexpr bool LUT = (LOGBG == 7 && LOGN == 10);
  static constexpr size_t lut_words = LUT ? (size_t)32 << LOGBG : 0;
  // GINX at the same shape: the top digit is folded into the key (bk_fold_kernel), so each component transforms DG - 1 digits per step
  // and the product multiplies A_hat_c = N^-1 * NTT(acc_c) in place of the top digit (see blind_rotate_kernel)
  static constexpr bool FOLD = LUT && !AP;
  // dct rows of a gate: the digit rows (digit l of component c in row c + 2l) and A_hat_c, the accumulator in evaluation form, in row
  // AROW + c.  GINX adds to A_hat, so it must survive the step's digit transforms: FOLD keeps it in the top digit's rows, which the product
  // multiplies, TOY in two extra rows.  AP replaces A_hat by the product's output, so it lives in digit row c: phase A inverse-transforms
  // it before digit 0 is written there, and a skipped step writes no digits.
  static constexpr int DROWS = (FOLD || AP) ? ROWS : ROWS + 2;
  static constexpr int AROW = AP ? 0 : DROWS - 2;
  static constexpr size_t dct_words = (size_t)G * DROWS * N;
  static constexpr size_t smem_bytes = (dct_words + 4 * N + (AP ? 0 : 2 * N) + lut_words) * 4 + (size_t)G * NPAD * 2;
  static_assert(smem_bytes <= 227 * 1024, "more dynamic shared memory than a block may have");
};

template <int LOGN, int DG, int LOGBG, int G, bool AP>
__global__ void __launch_bounds__(64 * G, 1)
blind_rotate_kernel(const __grid_constant__ DevConst P, const DevGate *__restrict__ gates, int count,
                    const u32 *__restrict__ bk, const u32 *__restrict__ g_twl, const u32 *__restrict__ g_psiM,
                    u32 *__restrict__ ext, u32 *__restrict__ acc_dbg) {
  using Cfg = BrCfg<LOGN, DG, LOGBG, G, AP>;
  constexpr int N = Cfg::N, E = Cfg::E, C = Cfg::C, ROWS = Cfg::ROWS, W = Cfg::W, NPAD = Cfg::NPAD;
  constexpr u32 DIGIT_OFF = digit_offset<DG, LOGBG>();
  // FOLD: the DG digits of the centred accumulator a in [-(Q+1)/2, (Q-3)/2] are the base-B digits of a + DIGIT_OFF, each minus B/2.  When
  // that sum always lies in [0, B^DG), they represent a exactly: acc_c = sum_l B^l d_{c,l} as integers, so in evaluation form the top digit
  // is D_{c,DG-1} = B^-(DG-1) (A_c - sum_{l<DG-1} B^l D_{c,l}) mod Q, A_c = NTT(acc_c).  Substituted into the external product, the top key
  // row moves into the other rows and into a row that multiplies A_hat_c = N^-1 A_c (bk_fold_kernel), and the step needs no transform of
  // the top digit.
  // Every form keeps the accumulator ONLY as A_hat_c, in dct row AROW + c: the product's output row is N^-1 NTT of the accumulator's
  // increment (GINX: A_hat_c += output) or of the whole new accumulator (AP: A_hat_c = output), and phase A gets acc_c back, fully reduced,
  // as the unscaled inverse transform of A_hat_c.
  constexpr bool FOLD = Cfg::FOLD;
  static_assert(!FOLD || (DIGIT_OFF >= (SOLINAS_Q + 1) / 2 && (u64)DIGIT_OFF + (SOLINAS_Q - 3) / 2 < (1ull << (LOGBG * DG))),
                "the digits do not cover the centred accumulator: the top digit cannot be folded into the key");
  constexpr int ND = FOLD ? DG - 1 : DG; // digit transforms per component and step
  constexpr int DROWS = Cfg::DROWS, AROW = Cfg::AROW;
  static_assert(AP || AROW == 2 * ND, "GINX: the A_hat rows follow the digit rows");
  // input bound (units of Q) of the inverse transform of A_hat: GINX keeps it below 2Q (lazy_reduce); AP stores one redc of ROWS products
  constexpr int AB = AP ? 8 : 2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  u32 *dct = reinterpret_cast<u32 *>(smem_raw);                 // [G][DROWS][N]
  u32 *s_tw = dct + Cfg::dct_words;                             // fw | fws | iw | iws
  u32 *s_psiM = s_tw + 4 * N;                                   // [2N] monomial-factor table (GINX; N entries used)
  u32 *s_lut = s_psiM + (AP ? 0 : 2 * N);                       // [2^LOGBG][32] (Cfg::LUT)
  u16 *s_idx = reinterpret_cast<u16 *>(s_lut + Cfg::lut_words); // [G][NPAD]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = warp >> 1, c = warp & 1; // this warp owns accumulator component c of gate g
  if constexpr (Cfg::LUT) { // the first stage of every digit transform multiplies a digit in [-B/2, B/2) by the one twiddle psi^(N/2)
    for (int i = tid; i < (int)Cfg::lut_words; i += Cfg::THREADS) {
      const u32 d = (u32)i >> 5;
      s_lut[i] = (u32)(((u64)P.tw[1] * ((d + P.Q - (1u << (LOGBG - 1))) % P.Q)) % P.Q);
    }
  }
  const int gate0 = blockIdx.x * G;
  const int gcount = min(G, count - gate0);
  const u32 Q = P.Q, q = P.q, n = P.n;

  for (int i = tid; i < 4 * N; i += Cfg::THREADS) s_tw[i] = g_twl[i];
  if (!AP) // monomial-factor table (psi^(2u) - 1), see the external product
    for (int u = tid; u < N; u += Cfg::THREADS) s_psiM[f_phys((u32)u)] = (g_psiM[2 * u] + (P.Q - P.oneM)) % P.Q;
  const TwTabs tt{s_tw, s_tw + N, s_tw + 2 * N, s_tw + 3 * N};

  // ---- prologue: LWE prep (EvalBinGate's ct1+ct2 / 2(ct1-ct2) / Bootstrap's b+q/4, with fused EvalNOT) ----
  __shared__ u32 s_b[G];
  for (int gg = 0; gg < gcount; gg++) {
    const DevGate dg = gates[gate0 + gg];
    const u32 gate = dg.op & 0xff;
    for (u32 i = tid; i <= n; i += Cfg::THREADS) {
      u32 x = dg.in0[i];
      if (dg.op & OP_NEG0) x = (i == n) ? (q / 4 + q - x) % q : (q - x) % q;
      u32 v;
      if (gate == OP_BOOTSTRAP) {
        v = (i == n) ? (x + q / 4) % q : x;
      } else {
        u32 y = dg.in1[i];
        if (dg.op & OP_NEG1) y = (i == n) ? (q / 4 + q - y) % q : (q - y) % q;
        v = (gate == OP_XOR_FAST || gate == OP_XNOR_FAST) ? (2 * (x + q - y)) % q : (x + y) % q;
      }
      if (i == n) s_b[gg] = v;
      else {
        u32 aneg = (q - v) % q;
        if (!AP) s_idx[gg * NPAD + i] = (u16)(aneg * P.factor); // monomial exponent in [0,2N)
        else {
          u32 a = aneg;
          for (u32 k = 0; k < P.dR; k++, a /= P.baseR) s_idx[gg * NPAD + i * P.dR + k] = (u16)(a % P.baseR);
        }
      }
    }
  }
  __syncthreads();

  // ---- accumulator init: A_hat = N^-1 * NTT(0, testvector) ----
  const bool gvalid = g < gcount;
  u32 *ahat = dct + ((size_t)g * DROWS + AROW + c) * N; // A_hat_c of gate g
  u32 *dbuf = dct + ((size_t)g * DROWS + c) * N;        // digit 0 of component c: scratch of the inverse transforms (AP: = ahat)
  if (gvalid) {
    u32 acc[E]; // coefficient form, column layout
#pragma unroll
    for (int k = 0; k < E; k++) acc[k] = 0;
    if (c == 1) {
      const u32 gate = gates[gate0 + g].op & 0xff;
      const u32 q1 = P.gate_const[gate == OP_BOOTSTRAP ? OP_AND : gate], q2 = (q1 + q / 2) % q;
      const u32 b = s_b[g], Q8 = P.Q8, Q8n = Q - P.Q8;
#pragma unroll
      for (int k = 0; k < E; k++) {
        const u32 idx = lane + 32 * k;
        if (idx % P.factor == 0) {
          const u32 t = (b + q - idx / P.factor) % q;
          const bool in = (q1 < q2) ? (t >= q1 && t < q2) : !(t >= q2 && t < q1);
          acc[k] = in ? Q8n : Q8;
        }
      }
    }
    ntt_forward<LOGN>(acc, ahat, P, tt, lane);
#pragma unroll
    for (int k = 0; k < E; k++) acc[k] = mul_shoup(acc[k], P.ninv, P.ninvs, Q); // below 2Q
    row_store<E>(ahat, acc, lane);
  }

  const int nsteps = AP ? n * P.dR : n;

  // MAC work split: item -> (chunk qc, gate split)
  constexpr int GS = (W >= C) ? (W / C) : 1;
  const u32 eA = 2 * brev(lane, 5) + 1; // lane part of the evaluation-point exponent 2*br(idx)+1
  // GINX: the step's key words are requested BEFORE the warp's last digit transform, so the L2 round trip runs under the transform and the
  // wait at the CTA barrier instead of in front of the product (535 cycles of a 27 k-cycle step sat there, tools/phase_timing.py; DESIGN.md 5.1)
  constexpr bool KEY_HOIST = !AP;

#ifdef BFHE_PHASE_TIMING
  long long tpt[5] = {0, 0, 0, 0, 0}, tq0 = clock64(), tq1;
#define PT_T(i) do { tq1 = clock64(); tpt[i] += tq1 - tq0; tq0 = tq1; } while (0)
#else
#define PT_T(i)
#endif
  for (int step = 0; step < nsteps; step++) {
    // key words of the external product (GINX: [sign][row][column]; AP: a double buffer over the gates, see below)
    uint4 kr[2][ROWS][2];
#define BFHE_GX_LOAD(qc) /* GINX: this step's key words of chunk qc, both signs */                                    \
  do {                                                                                                                 \
    const u32 *kb_ = bk + (size_t)step * (2 * ROWS * 2) * N + ((qc) * 32 + lane) * 4;                                  \
    _Pragma("unroll") for (int s = 0; s < 2; s++)                                                                      \
      _Pragma("unroll") for (int r = 0; r < ROWS; r++)                                                                 \
        _Pragma("unroll") for (int cc = 0; cc < 2; cc++)                                                               \
          kr[s][r][cc] = __ldg(reinterpret_cast<const uint4 *>(kb_ + (size_t)((s * ROWS + r) * 2 + cc) * N));           \
  } while (0)
    // AP: every gate has its own key (BK[i][digit][k]), so nothing is shared between the gates of the CTA; the two halves of kr[] are a
    // double buffer instead -- gate j's words are requested while gate j - 1 is multiplied (the first two before the barrier), which takes
    // the L2 round trip of 16 LDG.128 per gate and step off the critical path
    constexpr int JN = (G + GS - 1) / GS; // gates per item
    auto ap_key = [&](int gg, int qc) -> const u32 * { // this step's key of gate gg at chunk qc (no such gate, or digit 0 = step skipped: any
      const u32 a0 = gg < gcount ? s_idx[gg * NPAD + step] : 0u; // valid key, the words are loaded and not used -- unconditional loads keep kr[] in registers)
      const u32 i = step / P.dR, k = step % P.dR;
      return bk + (((size_t)i * (P.baseR - 1) + (a0 ? a0 - 1 : 0u)) * P.dR + k) * (ROWS * 2) * N + (qc * 32 + lane) * 4;
    };
#define BFHE_AP_LOAD(buf, kb)                                                                                          \
  do {                                                                                                                 \
    const u32 *kb_ = (kb);                                                                                             \
    _Pragma("unroll") for (int r = 0; r < ROWS; r++)                                                                   \
      _Pragma("unroll") for (int cc = 0; cc < 2; cc++)                                                                 \
        kr[buf][r][cc] = __ldg(reinterpret_cast<const uint4 *>(kb_ + (size_t)(r * 2 + cc) * N));                        \
  } while (0)

    // ================= phase A: one warp per (gate, component) =================
    bool active = gvalid;
    if (AP && gvalid) active = s_idx[g * NPAD + step] != 0;
    if (active) {
      // acc_c = INTT(A_hat_c) in [0, Q).  The transform's scratch is digit row c, rewritten below: GINX's A_hat_c, in other rows, stays as
      // it is; AP's is that row and is replaced by the product anyway.
      u32 dp[E];
      row_load<E>(ahat, dp, lane);
      ntt_inverse<LOGN, AB>(dp, dbuf, P, tt, lane);
      // SignedDigitDecompose (a12): centre, peel DG signed base-2^LOGBG digits, digit l of component c -> row c+2l
      // Closed form of the sequential peel (r = signed low digit; d = (d - r) >> LOGBG): adding B/2 at every digit
      // position turns the balanced digits into the plain base-B digits of d + OFF, so digit l is one shift, one mask and
      // one subtraction with no dependency on the digits below it (the top digit wraps exactly like the reference's
      // sign-truncation when dG digits do not cover the centred range, e.g. TOY).  FOLD: the top digit is not needed.
#pragma unroll
      for (int k = 0; k < E; k++) dp[k] = ((dp[k] < (Q >> 1)) ? dp[k] : dp[k] - Q) + DIGIT_OFF;
#pragma unroll
      for (int l = 0; l < ND; l++) {
        u32 x[E], pre[Cfg::LUT ? E / 2 : 1];
#pragma unroll
        for (int k = 0; k < E; k++) {
          const u32 dgt = (dp[k] >> (LOGBG * l)) & ((1u << LOGBG) - 1);
          // digit - B/2 + Q: congruent to the signed digit, lazy in (Q - B/2, Q + B/2); the forward transform needs no canonical
          // input (values then stay below (2 logN + 2) Q < 2^32)
          if (Cfg::LUT && k >= E / 2) { pre[Cfg::LUT ? k - E / 2 : 0] = s_lut[(dgt << 5) + lane]; x[k] = 0; }
          else x[k] = dgt + (Q - (1u << (LOGBG - 1)));
        }
        u32 *buf = dct + ((size_t)g * DROWS + c + 2 * l) * N;
        if (KEY_HOIST && l == ND - 1 && warp < C * GS) BFHE_GX_LOAD(warp % C);
        ntt_forward<LOGN, Cfg::LUT>(x, buf, P, tt, lane, pre);
        row_store<E>(buf, x, lane);
      }
    } else if (KEY_HOIST && warp < C * GS) { // empty gate slot (ragged last CTA): no transform to hide behind, but the product still needs the words
      BFHE_GX_LOAD(warp % C);
    }
    PT_T(0);
    // the first key words of this warp's chunk are requested BEFORE the barrier, so the L2 round trip overlaps the wait for the slower
    // warps of the CTA instead of stalling the external product (ncu r1: 6 % of samples sat on these loads)
    if (AP && warp < C * GS) {
      BFHE_AP_LOAD(0, ap_key(warp / C, warp % C));
      if (JN > 1) BFHE_AP_LOAD(1, ap_key(warp / C + GS, warp % C));
    }
    __syncthreads();
    PT_T(1);

    // ================= phase B: external product, slot-parallel over the CTA =================
    for (int item = warp; item < C * GS; item += W) {
      const int qc = item % C, gs0 = item / C;
      if (!AP && item != warp) BFHE_GX_LOAD(qc); // further chunks of this warp (fewer warps than chunks)
      // exponent parts that depend on (chunk, slot-in-chunk)
      u32 eB[4];
#pragma unroll
      for (int r = 0; r < 4; r++) eB[r] = 2 * ((brev(r, 2) << (LOGN - 2)) | (brev(qc, LOGN - 7) << 5));

      if (AP && item != warp) { // further chunks of this warp: no prefetch across items
        BFHE_AP_LOAD(0, ap_key(gs0, qc));
        if (JN > 1) BFHE_AP_LOAD(1, ap_key(gs0 + GS, qc));
      }
#pragma unroll
      for (int j = 0; j < JN; j++) {
        const int gg = gs0 + j * GS;
        const bool ap_active = AP && gg < gcount && s_idx[(gg < gcount ? gg : 0) * NPAD + step] != 0;
        if (gg >= gcount || (AP && !ap_active)) { // nothing to multiply for this gate in this step; keep the double buffer moving
          if (AP && j + 2 < JN) { if ((j & 1) == 0) BFHE_AP_LOAD(0, ap_key(gs0 + (j + 2) * GS, qc)); else BFHE_AP_LOAD(1, ap_key(gs0 + (j + 2) * GS, qc)); }
          continue;
        }
        u32 fp[4], fn[4];
        if (!AP) {
          // monomial factors (X^m - 1), (X^-m - 1) at this thread's 4 evaluation points, Montgomery form
          // (exponents are even -- m is a multiple of 2N/q = 2 -- so the table has N entries, (psi^(2u) - 1) * 2^32 mod Q at f_phys(u): one
          // gather per factor instead of two gathers and a Montgomery product; the index fold keeps the 32 lanes of a warp, whose u differ
          // in five consecutive bits t .. t+4 (t = number of trailing zeros of m), on 32 different banks for every t)
          const u32 m = s_idx[gg * NPAD + step];
#pragma unroll
          for (int r = 0; r < 4; r++) {
            const u32 u = ((m * (eA + eB[r])) >> 1) & (N - 1);
            fp[r] = s_psiM[f_phys(u)];
            fn[r] = s_psiM[f_phys((0u - u) & (N - 1))];
          }
        }
        u32 *gd = dct + (size_t)gg * DROWS * N + Lay<E>::chunk_off(lane, qc);
        // the ROWS multiplied rows, and for GINX the A_hat rows the output is added to (FOLD: the same rows)
        constexpr int NLD = AP ? ROWS : DROWS;
        uint4 dv[NLD];
#pragma unroll
        for (int r = 0; r < NLD; r++) dv[r] = *reinterpret_cast<const uint4 *>(gd + (size_t)r * N);
#pragma unroll
        for (int cc = 0; cc < 2; cc++) {
          u32 out[4];
#pragma unroll
          for (int sl = 0; sl < 4; sl++) {
            u64 sp = 0, sn = 0;
#pragma unroll
            for (int r = 0; r < ROWS; r++) {
              const u32 dval = sl == 0 ? dv[r].x : sl == 1 ? dv[r].y : sl == 2 ? dv[r].z : dv[r].w;
              const uint4 kp = kr[AP ? (j & 1) : 0][r][cc];
              sp += (u64)dval * (sl == 0 ? kp.x : sl == 1 ? kp.y : sl == 2 ? kp.z : kp.w);
              if (!AP) {
                const uint4 kn = kr[AP ? 0 : 1][r][cc];
                sn += (u64)dval * (sl == 0 ? kn.x : sl == 1 ? kn.y : sl == 2 ? kn.z : kn.w);
              }
            }
            const u32 pp = redc(sp, Q, P.qinv_neg);
            if (AP) out[sl] = pp;
            else {
              const u32 pn = redc(sn, Q, P.qinv_neg);
              out[sl] = redc((u64)pp * fp[sl] + (u64)pn * fn[sl], Q, P.qinv_neg);
            }
          }
          // the output goes to A_hat_cc only (this thread has already consumed that chunk of every row).  GINX: A_hat_cc += output, kept
          // below 2Q (FOLD: the products' bounds assume < 22Q).  AP: the output is the whole new accumulator.
          u32 *ga = gd + (size_t)(AROW + cc) * N;
          if constexpr (AP) *reinterpret_cast<uint4 *>(ga) = make_uint4(out[0], out[1], out[2], out[3]);
          else {
            const uint4 a = dv[AROW + cc];
            *reinterpret_cast<uint4 *>(ga) =
                make_uint4(lazy_reduce(a.x + out[0], Q), lazy_reduce(a.y + out[1], Q), lazy_reduce(a.z + out[2], Q), lazy_reduce(a.w + out[3], Q));
          }
        }
        if (AP && j + 2 < JN) { // this buffer is free again: request the key of the gate after next
          if ((j & 1) == 0) BFHE_AP_LOAD(0, ap_key(gs0 + (j + 2) * GS, qc)); else BFHE_AP_LOAD(1, ap_key(gs0 + (j + 2) * GS, qc));
        }
      }
    }
    PT_T(2);
    __syncthreads();
    PT_T(3);
  }

  // ---- epilogue: last inverse transform, sample extraction (a14) and ModSwitch Q -> qKS (a15) ----
  if (gvalid) {
    u32 acc[E];
    row_load<E>(ahat, acc, lane);
    ntt_inverse<LOGN, AB>(acc, dbuf, P, tt, lane);
    const size_t gi = (size_t)gate0 + g;
    if (acc_dbg) {
#pragma unroll
      for (int k = 0; k < E; k++) acc_dbg[(gi * 2 + c) * N + lane + 32 * k] = acc[k];
    }
    u32 *e = ext + gi * (N + 4);
    const u64 qKS = P.qKS;
    if (c == 0) {
#pragma unroll
      for (int k = 0; k < E; k++) {
        const u32 j = lane + 32 * k;
        const u32 v = (j == 0) ? acc[k] : (acc[k] == 0 ? 0 : Q - acc[k]); // Transpose: a'_0 = a_0, a'_k = -a_{N-k}
        const u32 pos = (j == 0) ? 0 : N - j;
        e[pos] = (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS);
      }
    } else if (lane == 0) {
      const u32 v = csub(acc[0] + P.Q8, Q);
      e[N] = (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS);
    }
#ifdef BFHE_PHASE_TIMING
    if (acc_dbg && lane == 0)
      for (int i = 0; i < 5; i++) acc_dbg[(gi * 2 + c) * N + 32 + i] = (u32)(tpt[i] / 1000); // kilo-cycles
#endif
  }
}



// ------------------------------------------------------------------------------------------
// inverse transform spread over 4 warps (N = 1024) for the latency kernel, where only two polynomials need an inverse transform per
// step: THREE passes of three register stages on 8-value tiles, only the widest stage (span 512) across lanes (36 + 8 multiplies per
// thread; a first version with two passes and four cross-lane stages did 24 + 32).  nat / nats: inverse twiddles
// in natural order m + i (group i of the stage with m groups), the 512-group stage de-interleaved (groups 8t + j at
// 512 + 256 (j >> 2) + 4t + (j & 3)) -- built in shared memory by the latency kernel.  T = 0..127 within the polynomial's 4 warps;
// on return x[k] = coefficient T6 + 64 (k + 8 hi), T6 = 16 (T >> 5) + (T & 15), hi = (T >> 4) & 1.
// ------------------------------------------------------------------------------------------
template <int T, int B> struct Gs8Stage { // one Gentleman-Sande stage on 8 registers, half-size T; B = input bound in units of Q
  static constexpr bool RED = (2 * B > 16);
  static constexpr int OUTB = RED ? 2 : 2 * B;
  __device__ __forceinline__ static void run(u32 (&x)[8], const u32 (&w)[8], const u32 (&ws)[8], u32 Q) {
    static_assert(B <= 16, "bound");
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int gi = i / T, a = gi * 2 * T + (i % T), b = a + T, p = 4 / T + gi;
      const u32 S = x[a] + x[b], D = x[a] - x[b] + B * Q;
      x[b] = mul_shoup(D, w[p], ws[p], Q);
      x[a] = RED ? lazy_reduce(S, Q) : S;
    }
  }
};
template <int B0> __device__ __forceinline__ void ntt_inverse_quad8(u32 (&x)[8], u32 *buf, const DevConst &P, const u32 *nat, const u32 *nats, int T,
                                                                   int bar_id) {
  const u32 Q = P.Q;
  u32 w[8], ws[8];
  auto run3 = [&](auto BC) { // three stages, returns nothing; bounds advance at compile time
    constexpr int B = decltype(BC)::value;
    using S1 = Gs8Stage<1, B>; using S2 = Gs8Stage<2, S1::OUTB>; using S3 = Gs8Stage<4, S2::OUTB>;
    S1::run(x, w, ws, Q); S2::run(x, w, ws, Q); S3::run(x, w, ws, Q);
  };
  constexpr int B1 = Gs8Stage<4, Gs8Stage<2, Gs8Stage<1, B0>::OUTB>::OUTB>::OUTB;
  constexpr int B2 = Gs8Stage<4, Gs8Stage<2, Gs8Stage<1, B1>::OUTB>::OUTB>::OUTB;
  constexpr int B3 = Gs8Stage<4, Gs8Stage<2, Gs8Stage<1, B2>::OUTB>::OUTB>::OUTB;
  { // narrow pass: positions 8T + j (row T >> 2 of the row layout, chunks 2 (T & 3) and + 1)
    const int tp = T >> 2, c0 = 2 * (T & 3), T3 = T >> 1, hb = T & 1;
    u32 *p0 = buf + Lay<32>::chunk_off(tp, c0), *p1 = buf + Lay<32>::chunk_off(tp, c0 + 1);
    const uint4 a0 = *reinterpret_cast<const uint4 *>(p0), a1 = *reinterpret_cast<const uint4 *>(p1);
    x[0] = a0.x; x[1] = a0.y; x[2] = a0.z; x[3] = a0.w; x[4] = a1.x; x[5] = a1.y; x[6] = a1.z; x[7] = a1.w;
    const uint4 t4 = *reinterpret_cast<const uint4 *>(nat + 512 + 256 * hb + 4 * T3), t4s = *reinterpret_cast<const uint4 *>(nats + 512 + 256 * hb + 4 * T3);
    const uint2 t2 = *reinterpret_cast<const uint2 *>(nat + 256 + 2 * T), t2s = *reinterpret_cast<const uint2 *>(nats + 256 + 2 * T);
    w[4] = t4.x; w[5] = t4.y; w[6] = t4.z; w[7] = t4.w; ws[4] = t4s.x; ws[5] = t4s.y; ws[6] = t4s.z; ws[7] = t4s.w;
    w[2] = t2.x; w[3] = t2.y; ws[2] = t2s.x; ws[3] = t2s.y;
    w[1] = nat[128 + T]; ws[1] = nats[128 + T];
    run3(std::integral_constant<int, B0>{});
    *reinterpret_cast<uint4 *>(p0) = make_uint4(x[0], x[1], x[2], x[3]);
    *reinterpret_cast<uint4 *>(p1) = make_uint4(x[4], x[5], x[6], x[7]);
  }
  bar_sync(bar_id, 128);
  { // middle pass: positions 64u + 8r + v
    const int u = T >> 3, v = T & 7;
    const int b = 64 * u + 8 * (u & 3) + 4 * (v >> 2) + (v & 3); // address of r = 0; r flips bits: 32 (r >> 2) + 8 (r & 3) + 4 (r >> 2)
    const uint4 t4 = *reinterpret_cast<const uint4 *>(nat + 64 + 4 * u), t4s = *reinterpret_cast<const uint4 *>(nats + 64 + 4 * u);
    const uint2 t2 = *reinterpret_cast<const uint2 *>(nat + 32 + 2 * u), t2s = *reinterpret_cast<const uint2 *>(nats + 32 + 2 * u);
    w[4] = t4.x; w[5] = t4.y; w[6] = t4.z; w[7] = t4.w; ws[4] = t4s.x; ws[5] = t4s.y; ws[6] = t4s.z; ws[7] = t4s.w;
    w[2] = t2.x; w[3] = t2.y; ws[2] = t2s.x; ws[3] = t2s.y;
    w[1] = nat[16 + u]; ws[1] = nats[16 + u];
#pragma unroll
    for (int r = 0; r < 8; r++) x[r] = buf[b ^ (32 * (r >> 2) + 8 * (r & 3) + 4 * (r >> 2))];
    run3(std::integral_constant<int, B1>{});
#pragma unroll
    for (int r = 0; r < 8; r++) buf[b ^ (32 * (r >> 2) + 8 * (r & 3) + 4 * (r >> 2))] = x[r];
  }
  bar_sync(bar_id, 128);
  { // wide pass: positions T6 + 64 (k + 8 hi); the last stage across lanes 16 apart
    const int lane = T & 31, hi = lane >> 4, T6 = 16 * (T >> 5) + (lane & 15), l5 = T6 & 31, t5 = T6 >> 5;
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = buf[32 * t5 + 64 * (k + 8 * hi) + 4 * ((l5 >> 2) ^ (t5 + 2 * (k & 3))) + (l5 & 3)];
#pragma unroll
    for (int g = 0; g < 4; g++) { w[4 + g] = nat[8 + 4 * hi + g]; ws[4 + g] = nats[8 + 4 * hi + g]; }
#pragma unroll
    for (int g = 0; g < 2; g++) { w[2 + g] = nat[4 + 2 * hi + g]; ws[2 + g] = nats[4 + 2 * hi + g]; }
    w[1] = nat[2 + hi]; ws[1] = nats[2 + hi];
    run3(std::integral_constant<int, B2>{});
    static_assert(B3 <= 16, "bound");
    const u32 w1 = nat[1], w1s = nats[1];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const u32 o = __shfl_xor_sync(0xffffffffu, x[k], 16);
      const u32 m = mul_shoup(o - x[k] + B3 * Q, w1, w1s, Q); // upper lane: (lower - upper) * w
      x[k] = hi ? m : x[k] + o;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = csub(lazy_reduce(x[k], Q), Q);
  }
}

// ------------------------------------------------------------------------------------------
// blind rotation, latency variant: ONE gate per CTA, one warp per decomposition row (2*DG warps), so the 2*DG
// forward NTTs of a step run concurrently and the step's critical path is INTT -> NTT -> MAC instead of
// INTT -> DG x NTT -> MAC.  Used for narrow wavefronts (deep circuits: AES, SHA-256), where there are fewer gates
// than the GPU has room for and latency per level is what matters.
// The step's bootstrapping-key tile (GINX: 2 RGSW = 128 KB) is prefetched into shared memory by a TMA bulk copy
// (cp.async.bulk + mbarrier complete_tx) issued right after the previous step's external product, so the
// L2 latency of the key is hidden behind the next step's transforms at no register or issue cost.
// ------------------------------------------------------------------------------------------
template <int LOGN, int DG, int LOGBG, bool AP> struct LatCfg {
  static constexpr int N = 1 << LOGN, E = N / 32, C = E / 4, ROWS = 2 * DG;
  static constexpr int W = ROWS, THREADS = 32 * W;
  static constexpr int NPAD = 1024;
  static constexpr int KEYPOLYS = AP ? ROWS * 2 : 2 * ROWS * 2;
  // words: dct | digits | key tile | twiddles | psi powers ; then u16 idx + u16 active list ; then the mbarrier
  static constexpr bool QUAD = (LOGN == 10 && W == 8); // inverse transform spread over 4 warps per polynomial
  static constexpr size_t nat_words = QUAD ? 2 * N : 0; // inverse twiddles in natural order (w | w') for ntt_inverse_quad8
  static constexpr size_t words = (size_t)ROWS * N + 2 * N + (size_t)KEYPOLYS * N + 4 * N + (AP ? 0 : 2 * N) + nat_words;
  static constexpr size_t smem_bytes = words * 4 + 2 * NPAD * 2 + 16;
};

template <int LOGN, int DG, int LOGBG, bool AP>
__global__ void __launch_bounds__(64 * DG, 1)
blind_rotate_lat_kernel(const __grid_constant__ DevConst P, const DevGate *__restrict__ gates, int count,
                        const u32 *__restrict__ bk, const u32 *__restrict__ g_twl, const u32 *__restrict__ g_psiM,
                        u32 *__restrict__ ext, u32 *__restrict__ acc_dbg) {
  using Cfg = LatCfg<LOGN, DG, LOGBG, AP>;
  constexpr int N = Cfg::N, E = Cfg::E, C = Cfg::C, ROWS = Cfg::ROWS, W = Cfg::W, NPAD = Cfg::NPAD, KEYPOLYS = Cfg::KEYPOLYS;
  constexpr u32 DIGIT_OFF = digit_offset<DG, LOGBG>();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  u32 *dct = reinterpret_cast<u32 *>(smem_raw);         // [ROWS][N]
  u32 *dig = dct + (size_t)ROWS * N;                    // [2][N] packed signed digits of the accumulator
  u32 *s_key = dig + 2 * N;                             // [KEYPOLYS][N] this step's key tile
  u32 *s_tw = s_key + (size_t)KEYPOLYS * N;             // fw | fws | iw | iws
  u32 *s_psiM = s_tw + 4 * N;                           // [2N] (GINX)
  u32 *s_nat = s_psiM + (AP ? 0 : 2 * N);               // [2N] inverse twiddles, natural order (QUAD)
  u16 *s_idx = reinterpret_cast<u16 *>(s_nat + Cfg::nat_words); // [NPAD] monomial exponent / AP digit per step
  u16 *s_list = s_idx + NPAD;                           // [NPAD] steps that do work
  u64 *s_bar = reinterpret_cast<u64 *>(s_list + NPAD);
  __shared__ u32 s_b, s_nact;
  constexpr bool QUAD = Cfg::QUAD;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = warp & 1, l = warp >> 1; // this warp transforms digit l of accumulator component c (row c + 2l)
  const size_t gi = blockIdx.x;
  const u32 Q = P.Q, q = P.q, n = P.n;
  const DevGate dg = gates[gi];

  for (int i = tid; i < 4 * N; i += Cfg::THREADS) s_tw[i] = g_twl[i];
  if (!AP)
    for (int u = tid; u < N; u += Cfg::THREADS) s_psiM[f_phys((u32)u)] = (g_psiM[2 * u] + (P.Q - P.oneM)) % P.Q; // (psi^(2u) - 1) * 2^32
  const TwTabs tt{s_tw, s_tw + N, s_tw + 2 * N, s_tw + 3 * N};
  if constexpr (QUAD) { // natural-order copy of the inverse twiddles: entry k < 32 from the kernel parameters, the rest out of the
                        // per-lane tables ([chunk][lane][4]: entry pp of lane L is twiddle groups * (32 + L) + gi)
    auto nat_slot = [&](int k) { return k < N / 2 ? k : N / 2 + (N / 4) * (((k - N / 2) & 7) >> 2) + 4 * ((k - N / 2) >> 3) + ((k - N / 2) & 3); };
    for (int k = tid; k < 32; k += Cfg::THREADS) { s_nat[nat_slot(k)] = P.itw[k]; s_nat[N + nat_slot(k)] = P.itws[k]; }
    for (int i = tid; i < 32 * E; i += Cfg::THREADS) {
      const int L = i / E, pp = i % E;
      if (pp == 0) continue;
      int groups = 1;
      while (groups * 2 <= pp) groups *= 2;
      const int k = groups * (32 + L) + (pp - groups), off = ((pp / 4) * 32 + L) * 4 + (pp % 4);
      s_nat[nat_slot(k)] = g_twl[2 * N + off];
      s_nat[N + nat_slot(k)] = g_twl[3 * N + off];
    }
  }
  if (tid == 0) {
    mbar_init(s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  { // LWE prep (same as the throughput kernel)
    const u32 gate = dg.op & 0xff;
    for (u32 i = tid; i <= n; i += Cfg::THREADS) {
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
      else {
        const u32 aneg = (q - v) % q;
        if (!AP) s_idx[i] = (u16)(aneg * P.factor);
        else {
          u32 a = aneg;
          for (u32 k = 0; k < P.dR; k++, a /= P.baseR) s_idx[i * P.dR + k] = (u16)(a % P.baseR);
        }
      }
    }
  }
  __syncthreads();
  const int nsteps = AP ? n * P.dR : n;
  if (tid == 0) { // steps that do work (AP skips zero digits; X^0 - 1 = 0 makes a zero GINX exponent a no-op as well)
    u32 na = 0;
    for (int s = 0; s < nsteps; s++)
      if (s_idx[s] != 0) s_list[na++] = (u16)s;
    s_nact = na;
  }
  __syncthreads();
  const int nact = s_nact;
  constexpr u32 KEYBYTES = (u32)KEYPOLYS * N * 4;
  auto key_src = [&](int step) -> const u32 * {
    if (!AP) return bk + (size_t)step * KEYPOLYS * N;
    const u32 a0 = s_idx[step], i = step / P.dR, k = step % P.dR;
    return bk + (((size_t)i * (P.baseR - 1) + (a0 - 1)) * P.dR + k) * (size_t)KEYPOLYS * N;
  };
  if (tid == 0 && nact > 0) {
    mbar_expect_tx(s_bar, KEYBYTES);
    const u32 *src = key_src(s_list[0]);
#pragma unroll 1
    for (u32 off = 0; off < KEYBYTES; off += 16384) bulk_g2s(reinterpret_cast<char *>(s_key) + off, reinterpret_cast<const char *>(src) + off, min(16384u, KEYBYTES - off), s_bar);
  }

  // accumulator (coefficient form).  QUAD: 8 coefficients per thread, component qc = warp / 4, index qL + 32 * (8 * qs + kk);
  // otherwise 32 coefficients per lane in warps 0 and 1 (component = warp, index lane + 32k).
  const int qc = warp >> 2, q4 = warp & 3;
  auto qpos = [&](int k) { return 16 * q4 + (lane & 15) + 64 * (k + 8 * (lane >> 4)); }; // ntt_inverse_quad8's output positions
  u32 acc[QUAD ? 8 : E];
#pragma unroll
  for (int k = 0; k < (QUAD ? 8 : E); k++) acc[k] = 0;
  if (QUAD ? (qc == 1) : (warp == 1)) {
    const u32 gate = dg.op & 0xff;
    const u32 q1 = P.gate_const[gate == OP_BOOTSTRAP ? OP_AND : gate], q2 = (q1 + q / 2) % q;
    const u32 b = s_b, Q8 = P.Q8, Q8n = Q - P.Q8;
#pragma unroll
    for (int k = 0; k < (QUAD ? 8 : E); k++) {
      const u32 idx = QUAD ? (u32)qpos(k) : (u32)(lane + 32 * k);
      if (idx % P.factor == 0) {
        const u32 t = (b + q - idx / P.factor) % q;
        const bool in = (q1 < q2) ? (t >= q1 && t < q2) : !(t >= q2 && t < q1);
        acc[k] = in ? Q8n : Q8;
      }
    }
  }
  const u32 eA = 2 * brev(lane, 5) + 1;

#ifdef BFHE_PHASE_TIMING
  long long tph[5] = {0, 0, 0, 0, 0}, tc0, tc1;
#define PH_T(i) do { tc1 = clock64(); tph[i] += tc1 - tc0; tc0 = tc1; } while (0)
  tc0 = clock64();
#else
#define PH_T(i)
#endif
  for (int j = 0; j < nact; j++) {
    const int step = s_list[j];
    // ---- phase 1: close the previous step (INTT, accumulate) and publish the centred accumulator + digit offset ----
    if constexpr (QUAD) {
      if (j > 0) {
        u32 x[8];
        ntt_inverse_quad8<AP ? 8 : 4>(x, dct + (size_t)qc * N, P, s_nat, s_nat + N, 32 * q4 + lane, 1 + qc);
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] = AP ? x[k] : csub(acc[k] + x[k], Q);
      }
#pragma unroll
      for (int k = 0; k < 8; k++) dig[qc * N + qpos(k)] = ((acc[k] < (Q >> 1)) ? acc[k] : acc[k] - Q) + DIGIT_OFF;
    } else if (warp < 2) {
      if (j > 0) {
        u32 x[E];
        u32 *rb = dct + (size_t)warp * N;
        row_load<E>(rb, x, lane);
        ntt_inverse<LOGN, AP ? 8 : 4>(x, rb, P, tt, lane);
#pragma unroll
        for (int k = 0; k < E; k++) acc[k] = AP ? x[k] : csub(acc[k] + x[k], Q);
      }
      // centred accumulator + digit offset: every warp then cuts its own digit out with a shift and a mask
#pragma unroll
      for (int k = 0; k < E; k++) dig[warp * N + lane + 32 * k] = ((acc[k] < (Q >> 1)) ? acc[k] : acc[k] - Q) + DIGIT_OFF;
    }
    PH_T(0);
    __syncthreads();
    PH_T(1);
    // ---- phase 2: every warp transforms its own digit polynomial ----
    {
      u32 x[E];
#pragma unroll
      for (int k = 0; k < E; k++) {
        x[k] = ((dig[c * N + lane + 32 * k] >> (LOGBG * l)) & ((1u << LOGBG) - 1)) + (Q - (1u << (LOGBG - 1))); // lazy: digit - B/2 + Q
      }
      u32 *buf = dct + (size_t)warp * N;
      ntt_forward<LOGN, false, SOL_LAT_WIDE, SOL_LAT_NARROW>(x, buf, P, tt, lane);
      row_store<E>(buf, x, lane);
    }
    PH_T(2);
    __syncthreads();
    mbar_wait(s_bar, (u32)(j & 1));
    PH_T(3);
    // ---- phase 3: external product against the staged key tile ----
    for (int qc = warp; qc < C; qc += W) {
      u32 fp[4], fn[4];
      if (!AP) {
        const u32 m = s_idx[step]; // monomial-factor table, as in the throughput kernel
#pragma unroll
        for (int r = 0; r < 4; r++) {
          const u32 eB = 2 * ((brev(r, 2) << (LOGN - 2)) | (brev(qc, LOGN - 7) << 5));
          const u32 u = ((m * (eA + eB)) >> 1) & (N - 1);
          fp[r] = s_psiM[f_phys(u)];
          fn[r] = s_psiM[f_phys((0u - u) & (N - 1))];
        }
      }
      u32 *gd = dct + Lay<E>::chunk_off(lane, qc);
      const u32 *kb = s_key + (qc * 32 + lane) * 4;
      uint4 dv[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; r++) dv[r] = *reinterpret_cast<const uint4 *>(gd + (size_t)r * N);
#pragma unroll
      for (int cc = 0; cc < 2; cc++) {
        u64 sp[4] = {0, 0, 0, 0}, sn[4] = {0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
          const uint4 kp = *reinterpret_cast<const uint4 *>(kb + (size_t)(r * 2 + cc) * N);
          sp[0] += (u64)dv[r].x * kp.x; sp[1] += (u64)dv[r].y * kp.y; sp[2] += (u64)dv[r].z * kp.z; sp[3] += (u64)dv[r].w * kp.w;
          if (!AP) {
            const uint4 kn = *reinterpret_cast<const uint4 *>(kb + (size_t)((ROWS + r) * 2 + cc) * N);
            sn[0] += (u64)dv[r].x * kn.x; sn[1] += (u64)dv[r].y * kn.y; sn[2] += (u64)dv[r].z * kn.z; sn[3] += (u64)dv[r].w * kn.w;
          }
        }
        u32 out[4];
#pragma unroll
        for (int sl = 0; sl < 4; sl++) {
          const u32 pp = redc(sp[sl], Q, P.qinv_neg);
          if (AP) out[sl] = pp;
          else out[sl] = redc((u64)pp * fp[sl] + (u64)redc(sn[sl], Q, P.qinv_neg) * fn[sl], Q, P.qinv_neg);
        }
        *reinterpret_cast<uint4 *>(gd + (size_t)cc * N) = make_uint4(out[0], out[1], out[2], out[3]);
      }
    }
    PH_T(4);
    __syncthreads();
    // ---- prefetch the next step's key tile while the next transforms run ----
    if (tid == 0 && j + 1 < nact) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // generic-proxy reads above, async-proxy writes below
      mbar_expect_tx(s_bar, KEYBYTES);
      const u32 *src = key_src(s_list[j + 1]);
#pragma unroll 1
      for (u32 off = 0; off < KEYBYTES; off += 16384) bulk_g2s(reinterpret_cast<char *>(s_key) + off, reinterpret_cast<const char *>(src) + off, min(16384u, KEYBYTES - off), s_bar);
    }
  }

  // ---- epilogue ----
  const u64 qKS = P.qKS;
  u32 *e = ext + gi * (N + 4);
  auto modswitch = [&](u32 v) -> u32 { return (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS); };
  if constexpr (QUAD) {
    if (nact > 0) {
      u32 x[8];
      ntt_inverse_quad8<AP ? 8 : 4>(x, dct + (size_t)qc * N, P, s_nat, s_nat + N, 32 * q4 + lane, 1 + qc);
#pragma unroll
      for (int k = 0; k < 8; k++) acc[k] = AP ? x[k] : csub(acc[k] + x[k], Q);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const u32 jj = (u32)qpos(k);
      if (acc_dbg) acc_dbg[(gi * 2 + qc) * N + jj] = acc[k];
      if (qc == 0) {
        const u32 v = (jj == 0) ? acc[k] : (acc[k] == 0 ? 0 : Q - acc[k]); // a'_0 = a_0, a'_k = -a_{N-k}
        e[(jj == 0) ? 0 : N - jj] = modswitch(v);
      } else if (jj == 0) {
        e[N] = modswitch(csub(acc[k] + P.Q8, Q));
      }
    }
  } else if (warp < 2) {
    if (nact > 0) {
      u32 x[E];
      u32 *rb = dct + (size_t)warp * N;
      row_load<E>(rb, x, lane);
      ntt_inverse<LOGN, AP ? 8 : 4>(x, rb, P, tt, lane);
#pragma unroll
      for (int k = 0; k < E; k++) acc[k] = AP ? x[k] : csub(acc[k] + x[k], Q);
    }
    if (acc_dbg) {
#pragma unroll
      for (int k = 0; k < E; k++) acc_dbg[(gi * 2 + warp) * N + lane + 32 * k] = acc[k];
    }
    if (warp == 0) {
#pragma unroll
      for (int k = 0; k < E; k++) {
        const u32 jj = lane + 32 * k;
        const u32 v = (jj == 0) ? acc[k] : (acc[k] == 0 ? 0 : Q - acc[k]);
        e[(jj == 0) ? 0 : N - jj] = modswitch(v);
      }
    } else if (lane == 0) {
      e[N] = modswitch(csub(acc[0] + P.Q8, Q));
    }
  }
#ifdef BFHE_PHASE_TIMING
  if (acc_dbg && lane == 0 && (QUAD ? (q4 == 0) : (warp < 2)))
    for (int i = 0; i < 5; i++) acc_dbg[(gi * 2 + (QUAD ? qc : warp)) * N + 32 + i] = (u32)(tph[i] / 1000); // kilo-cycles
#endif
}

template <int LOGN, int DG, int LOGBG, bool AP>
static int launch_lat_inst(const DevConst &P, const DevGate *d_gates, int count, const u32 *d_bk, const u32 *d_twl,
                           const u32 *d_psiM, u32 *d_ext, u32 *d_acc, cudaStream_t st, LaunchInfo *info) {
  using Cfg = LatCfg<LOGN, DG, LOGBG, AP>;
  auto kern = blind_rotate_lat_kernel<LOGN, DG, LOGBG, AP>;
  static bool attr_done[64];
  if (int rc = once_per_device(attr_done, [&] { return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::smem_bytes); }))
    return rc;
  if (count <= 0) return 0; // attribute warm-up only
  if (info) { info->gates_per_cta = 1; info->ctas = count; info->smem_bytes = Cfg::smem_bytes; }
  kern<<<count, Cfg::THREADS, Cfg::smem_bytes, st>>>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc);
  return (int)cudaGetLastError();
}

template <int LOGN, int DG, int LOGBG, int G, bool AP>
static int launch_br_inst(const DevConst &P, const DevGate *d_gates, int count, const u32 *d_bk, const u32 *d_twl,
                          const u32 *d_psiM, u32 *d_ext, u32 *d_acc, cudaStream_t st, LaunchInfo *info) {
  using Cfg = BrCfg<LOGN, DG, LOGBG, G, AP>;
  auto kern = blind_rotate_kernel<LOGN, DG, LOGBG, G, AP>;
  static bool attr_done[64];
  if (int rc = once_per_device(attr_done, [&] { return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::smem_bytes); }))
    return rc;
  if (count <= 0) return 0; // attribute warm-up only
  const int ctas = (count + G - 1) / G;
  if (info) { info->gates_per_cta = G; info->ctas = ctas; info->smem_bytes = Cfg::smem_bytes; }
  kern<<<ctas, Cfg::THREADS, Cfg::smem_bytes, st>>>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc);
  return (int)cudaGetLastError();
}

template <int LOGN, int DG, int LOGBG, bool AP>
static int launch_br_g(int G, const DevConst &P, const DevGate *d_gates, int count, const u32 *d_bk, const u32 *d_twl,
                       const u32 *d_psiM, u32 *d_ext, u32 *d_acc, cudaStream_t st, LaunchInfo *info) {
  switch (G) {
  case 1: return launch_br_inst<LOGN, DG, LOGBG, 1, AP>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc, st, info);
  case 2: return launch_br_inst<LOGN, DG, LOGBG, 2, AP>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc, st, info);
  // (6 gates per CTA, 3 warps per scheduler with a register-lean product, measured 7 % slower than 4: DESIGN.md 5.4)
  default: return launch_br_inst<LOGN, DG, LOGBG, 4, AP>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc, st, info);
  }
}

template <int LOGN, int DG, int LOGBG> static int br_attrs() {
  DevConst P{};
  int rc = 0;
  for (int G : {1, 2, 4}) {
    rc |= launch_br_g<LOGN, DG, LOGBG, false>(G, P, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
    rc |= launch_br_g<LOGN, DG, LOGBG, true>(G, P, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
  }
  rc |= launch_lat_inst<LOGN, DG, LOGBG, false>(P, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
  rc |= launch_lat_inst<LOGN, DG, LOGBG, true>(P, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, nullptr);
  return rc;
}
int blind_rotate_set_attrs() {
  int rc = br_attrs<10, 4, 7>();
  rc |= br_attrs<9, 3, 9>();
  rc |= v2_set_attrs();
  rc |= clx_set_attrs();
  return rc;
}

int launch_blind_rotate(const DevConst &P, int method_ap, const DevGate *d_gates, int count, const u32 *d_bk, const u32 *d_twl,
                        const u32 *d_psiM, u32 *d_ext, u32 *d_acc_dbg, int force_g, void *stream, LaunchInfo *info, const V2Bufs *v2) {
  if (count <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const bool have_cl2 = v2 && v2->d_bk4 && v2->d_tw2 && v2->d_F && v2_supported(P, method_ap);
  const bool have_clx = v2 && v2->d_bkx && v2->d_twx && (method_ap || v2->d_F) && clx_supported(P, method_ap);
  if (force_g == 128) return have_clx ? launch_blind_rotate_clx(P, method_ap, d_gates, count, *v2, d_ext, d_acc_dbg, stream, info) : (int)cudaErrorInvalidValue;
  if (force_g == 32) return have_cl2 ? launch_blind_rotate_cl2(P, d_gates, count, *v2, d_ext, d_acc_dbg, stream, info) : (int)cudaErrorInvalidValue;
  if (force_g != 0 && force_g != 1 && force_g != 2 && force_g != 4 && force_g != 8) return (int)cudaErrorInvalidValue;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // Which variant?  Measured on B200, STD128_OPT GINX (profiles/): one gate on four SMs 0.98 ms per wave of up to 33 gates; one gate on two
  // SMs 1.48 ms up to 74; latency form (one gate per CTA) 2.22 ms per wave of `sms` gates; throughput form (4 gates per CTA share every
  // key word) 5.68 ms per wave of 4 * sms gates.  Narrow circuit levels go to the cluster forms, wide batches to the throughput form.
  if (force_g == 0 && have_clx && count <= clx_fast_gates()) return launch_blind_rotate_clx(P, method_ap, d_gates, count, *v2, d_ext, d_acc_dbg, stream, info);
  if (force_g == 0 && have_cl2 && count <= cl2_max_gates()) return launch_blind_rotate_cl2(P, d_gates, count, *v2, d_ext, d_acc_dbg, stream, info);
  const long lat_cost = (long)((count + sms - 1) / sms) * 222;           // 2.22 ms per wave of `sms` gates
  const long thr_cost = (long)((count + 4 * sms - 1) / (4 * sms)) * 568; // 5.68 ms per wave of 4 * sms gates
  const bool lat = force_g == 8 || (force_g == 0 && lat_cost <= thr_cost);
  if (lat) {
    if (P.N == 1024 && P.dG == 4 && P.logBG == 7)
      return method_ap ? launch_lat_inst<10, 4, 7, true>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info)
                       : launch_lat_inst<10, 4, 7, false>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info);
    if (P.N == 512 && P.dG == 3 && P.logBG == 9)
      return method_ap ? launch_lat_inst<9, 3, 9, true>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info)
                       : launch_lat_inst<9, 3, 9, false>(P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info);
    return (int)cudaErrorInvalidValue;
  }
  int G = force_g > 0 ? force_g : 4;
  if (P.N == 1024 && P.dG == 4 && P.logBG == 7) {
    if (method_ap) return launch_br_g<10, 4, 7, true>(G, P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info);
    static_assert(BrCfg<10, 4, 7, 4, false>::FOLD, "the GINX throughput kernel of this shape reads the folded key");
    if (!v2 || !v2->d_bkf) return (int)cudaErrorInvalidValue;
    return launch_br_g<10, 4, 7, false>(G, P, d_gates, count, v2->d_bkf, d_twl, d_psiM, d_ext, d_acc_dbg, st, info);
  }
  if (P.N == 512 && P.dG == 3 && P.logBG == 9) {
    return method_ap ? launch_br_g<9, 3, 9, true>(G, P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info)
                     : launch_br_g<9, 3, 9, false>(G, P, d_gates, count, d_bk, d_twl, d_psiM, d_ext, d_acc_dbg, st, info);
  }
  return (int)cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------------------
// key switch (a16) + ModSwitch qKS -> q (a17).  One CTA per gate; RG row groups x COLS column threads.
// Device KSK layout: [i][j][digit][ROWLEN] so that the 2048 (N*dKS) rows a gate gathers are each one
// contiguous, 128-byte-aligned run.  PACK16: two uint16 residues per 32-bit lane load (qKS <= 2^16,
// a power of two, so accumulating mod 2^32 per half and masking at the end is exact).
// ------------------------------------------------------------------------------------------
// ---- multi-GPU exchange fused into the key switch (PeerX, common.hpp) ----
__device__ __forceinline__ void peer_store(const PeerX &px, const u32 *out, int k, u32 v) {
  if (px.slabs == nullptr) return;
  const size_t off = (size_t)(out - px.local_base) + (size_t)k;
  for (u32 r = 0; r < px.world; r++)
    if (r != px.rank) px.slabs[r][off] = v; // NVLink store into rank r's slab, same row
}
__device__ __forceinline__ void st_release_sys(u32 *p, u32 v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ u32 ld_acquire_sys(const u32 *p) {
  u32 v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// called by every thread of the CTAs that count (all threads of the CTA, convergent): the last of `total` CTAs raises the flags
__device__ __forceinline__ void peer_publish(const PeerX &px, u32 total) {
  if (px.slabs == nullptr) return;
  __threadfence_system(); // my peer stores are performed system-wide before anything that follows
  __syncthreads();
  if (threadIdx.x == 0) {
    const u32 done = atomicAdd(px.counter, 1u) + 1u;
    if (done == total) {
      atomicExch(px.counter, 0u); // next launch on this stream
      __threadfence_system();
      const u32 v = *px.epoch * px.per_epoch + px.index + 1u;
      for (u32 r = 0; r < px.world; r++)
        if (r != px.rank) st_release_sys(px.flags[r] + px.rank, v);
    }
  }
}
__global__ void peer_epoch_bump_kernel(u32 *epoch) { *epoch += 1; }
__global__ void peer_wait_kernel(const u32 *flags, const u32 *epoch, u32 world, u32 rank, int index, u32 per_epoch, u32 *err, long long timeout_cycles) {
  const u32 r = threadIdx.x;
  if (r >= world || r == rank) return;
  const u32 target = *epoch * per_epoch + (u32)(index + 1);
  const long long t0 = clock64();
  while ((int)(ld_acquire_sys(flags + r) - target) < 0) {
    if (clock64() - t0 > timeout_cycles) { atomicExch(err, 1u + r); break; } // a peer died or the ranks disagree on the schedule
    __nanosleep(200);
  }
}
__global__ void peer_signal_kernel(const PeerX px) { // end-of-Clock signal: everything this rank did in the epoch is complete (stream order)
  const u32 r = threadIdx.x;
  if (r >= px.world || r == px.rank) return;
  __threadfence_system();
  st_release_sys(px.flags[r] + px.rank, *px.epoch * px.per_epoch + px.index + 1u);
}
int launch_peer_epoch_bump(u32 *epoch, void *stream) {
  peer_epoch_bump_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(epoch);
  return (int)cudaGetLastError();
}
int launch_peer_wait(const u32 *local_flags, const u32 *epoch, u32 world, u32 rank, int index, u32 per_epoch, u32 *err, void *stream) {
  if (world > 32) return (int)cudaErrorInvalidValue;
  // A rank may legitimately lag by seconds (host-side verify of a large circuit between two Clocks, graph instantiation): the limit only
  // has to turn a dead peer into an error instead of a hung GPU.  BFHE_EXCHANGE_TIMEOUT_S overrides the 30 s default.
  static const long long cycles = [] {
    const char *e = std::getenv("BFHE_EXCHANGE_TIMEOUT_S");
    const double sec = e && std::atof(e) > 0 ? std::atof(e) : 30.0;
    return (long long)(sec * 2.0e9);
  }();
  peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(local_flags, epoch, world, rank, index, per_epoch, err, cycles);
  return (int)cudaGetLastError();
}
int launch_peer_signal(const PeerX &px, void *stream) {
  if (px.world > 32) return (int)cudaErrorInvalidValue;
  peer_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(px);
  return (int)cudaGetLastError();
}

template <bool PACK16, int COLS, int RG>
__global__ void __launch_bounds__(COLS *RG) keyswitch_kernel(const __grid_constant__ DevConst P, const u32 *__restrict__ ext,
                                                             const DevGate *__restrict__ gates, const void *__restrict__ ksk,
                                                             int rowlen_words, const PeerX px) {
  extern __shared__ u32 s_row[]; // N*dKS row ids, then RG*COLS*2 partial sums (u64 for !PACK16)
  const int N = P.N, dKS = P.dKS, nrows = N * dKS;
  const int tid = threadIdx.x, col = tid % COLS, rg = tid / COLS;
  const u32 *e = ext + (size_t)blockIdx.x * (N + 4);
  for (int r = tid; r < nrows; r += COLS * RG) {
    const int i = r / dKS, j = r % dKS;
    u32 a = e[i];
    for (int t = 0; t < j; t++) a /= P.baseKS;
    s_row[r] = (u32)((i * dKS + j) * P.baseKS + a % P.baseKS);
  }
  __syncthreads();
  u64 *s_part = reinterpret_cast<u64 *>(s_row + ((nrows + 1) & ~1));
  const u32 *k32 = reinterpret_cast<const u32 *>(ksk);
  const bool colok = col < rowlen_words;
  if (PACK16) {
    u32 lo = 0, hi = 0;
    if (colok) {
#pragma unroll 8
      for (int r = rg; r < nrows; r += RG) {
        const u32 w = __ldg(k32 + (size_t)s_row[r] * rowlen_words + col);
        lo += w & 0xffffu;
        hi += w >> 16;
      }
    }
    s_part[(rg * COLS + col) * 2] = lo;
    s_part[(rg * COLS + col) * 2 + 1] = hi;
  } else {
    u64 s = 0;
    if (colok) {
#pragma unroll 8
      for (int r = rg; r < nrows; r += RG) s += __ldg(k32 + (size_t)s_row[r] * rowlen_words + col);
    }
    s_part[(rg * COLS + col) * 2] = s;
  }
  __syncthreads();
  if (rg == 0 && colok) {
    const u64 qKS = P.qKS, q = P.q;
    u32 *out = gates[blockIdx.x].out;
    const int n = P.n;
    for (int h = 0; h < (PACK16 ? 2 : 1); h++) {
      const int k = PACK16 ? 2 * col + h : col;
      if (k > n) break;
      u64 s = 0;
      for (int r = 0; r < RG; r++) s += s_part[(r * COLS + col) * 2 + h];
      s %= qKS;
      const u64 base = (k == n) ? e[N] : 0; // out = (0, b) - sum of selected KSK rows
      const u64 v = (base + qKS - s) % qKS;
      const u32 res = (u32)(((2 * v * q + qKS) / (2 * qKS)) % q); // RoundqQ, exact integer form (SURVEY C.5)
      out[k] = res;
      peer_store(px, out, k, res);
    }
  }
  peer_publish(px, gridDim.x);
}

constexpr int ks_cl4_unroll = 16; // row gathers in flight per thread; measured 8: 29.2 us, 16: 27.1 us, 32: 35.1 us per 33-gate wave
// The same key switch on a 4-CTA cluster per gate (packed uint16 KSK only): each CTA gathers a quarter of the N*dKS rows, rank 0 adds the
// four partial sums out of its peers' shared memory (DSMEM) and finishes.  The one-CTA form is latency-bound (512 dependent row
// gathers per thread, 55 us whatever the batch); narrow circuit waves (1.2 - 1.5 ms each) pay that every wave.
template <int COLS, int RG>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(COLS *RG) keyswitch_cl4_kernel(const __grid_constant__ DevConst P, const u32 *__restrict__ ext,
                                                                                             const DevGate *__restrict__ gates,
                                                                                             const void *__restrict__ ksk, int rowlen_words, const PeerX px) {
  __shared__ u32 s_row[512];               // row ids of this CTA's quarter
  __shared__ u32 s_part[RG * COLS * 2];    // per row group partial sums (lo, hi halves)
  __shared__ u32 s_tot[COLS * 2];          // this CTA's sums, read by rank 0
  const int N = P.N, dKS = P.dKS, nrows = N * dKS, quarter = nrows / 4;
  const int tid = threadIdx.x, col = tid % COLS, rg = tid / COLS;
  const u32 rank = cluster_rank();
  const size_t gate = blockIdx.x >> 2;
  const u32 *e = ext + gate * (N + 4);
  for (int r = tid; r < quarter; r += COLS * RG) {
    const int gr = (int)rank * quarter + r, i = gr / dKS, j = gr % dKS;
    u32 a = e[i];
    for (int t = 0; t < j; t++) a /= P.baseKS;
    s_row[r] = (u32)((i * dKS + j) * P.baseKS + a % P.baseKS);
  }
  __syncthreads();
  const u32 *k32 = reinterpret_cast<const u32 *>(ksk);
  u32 lo = 0, hi = 0;
  if (col < rowlen_words) {
#pragma unroll ks_cl4_unroll
    for (int r = rg; r < quarter; r += RG) {
      const u32 w = __ldg(k32 + (size_t)s_row[r] * rowlen_words + col);
      lo += w & 0xffffu;
      hi += w >> 16;
    }
  }
  s_part[(rg * COLS + col) * 2] = lo;
  s_part[(rg * COLS + col) * 2 + 1] = hi;
  __syncthreads();
  if (rg == 0) {
#pragma unroll
    for (int h = 0; h < 2; h++) {
      u32 t = 0;
      for (int r = 0; r < RG; r++) t += s_part[(r * COLS + col) * 2 + h];
      s_tot[col * 2 + h] = t;
    }
  }
  cluster_sync_all();
  if (rank == 0 && rg == 0 && col < rowlen_words) {
    const u64 qKS = P.qKS, q = P.q;
    u32 *out = gates[gate].out;
    const int n = P.n;
    for (int h = 0; h < 2; h++) {
      const int k = 2 * col + h;
      if (k > n) break;
      u64 sum = s_tot[col * 2 + h];
      for (u32 pr = 1; pr < 4; pr++) {
        u32 v;
        asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(dsmem_addr(&s_tot[col * 2 + h], pr)) : "memory");
        sum += v;
      }
      sum %= qKS;
      const u64 base = (k == n) ? e[N] : 0; // out = (0, b) - sum of selected KSK rows
      const u64 v = (base + qKS - sum) % qKS;
      const u32 res = (u32)(((2 * v * q + qKS) / (2 * qKS)) % q); // RoundqQ, exact integer form (SURVEY C.5)
      out[k] = res;
      peer_store(px, out, k, res);
    }
  }
  if (rank == 0) peer_publish(px, gridDim.x >> 2); // one count per gate
  cluster_sync_all(); // peers stay until rank 0 has read
}

int launch_keyswitch(const DevConst &P, const u32 *d_ext, const DevGate *d_gates, int count, const void *d_ksk, int elem_bytes,
                     void *stream, const PeerX *pxp) {
  if (count <= 0) return 0;
  const PeerX px = pxp ? *pxp : PeerX();
  cudaStream_t st = (cudaStream_t)stream;
  const int nrows = P.N * P.dKS;
  if (elem_bytes == 2) {
    constexpr int COLS = 256, RG = 4;
    const int rowlen_words = 256; // 512 uint16 per row
    size_t smem = (size_t)((nrows + 1) & ~1) * 4 + (size_t)RG * COLS * 2 * 8; // STD128_OPT: 24 KB, within the default 48 KB limit
    // while every CTA of the cluster form has an SM to itself it wins (measured: 1 gate 47 -> 23 us, 30 gates 56 -> 29 us; 74 gates
    // 57 -> 54 us; 148 gates 56 -> 82 us): used up to SMs / 4 gates, wider batches keep one CTA per gate
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (nrows % 4 == 0 && nrows / 4 <= 512 && 4 * count <= sms)
      keyswitch_cl4_kernel<COLS, RG><<<4 * count, COLS * RG, 0, st>>>(P, d_ext, d_gates, d_ksk, rowlen_words, px);
    else
      keyswitch_kernel<true, COLS, RG><<<count, COLS * RG, smem, st>>>(P, d_ext, d_gates, d_ksk, rowlen_words, px);
  } else {
    constexpr int COLS = 128, RG = 4;
    const int rowlen_words = P.ct_stride;
    if (rowlen_words > COLS) return (int)cudaErrorInvalidValue;
    size_t smem = (size_t)((nrows + 1) & ~1) * 4 + (size_t)RG * COLS * 2 * 8;
    keyswitch_kernel<false, COLS, RG><<<count, COLS * RG, smem, st>>>(P, d_ext, d_gates, d_ksk, rowlen_words, px);
  }
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// EvalNOT (a6): (-a, q/4 - b)
// ------------------------------------------------------------------------------------------
// low bit of the (16-byte aligned) input pointer set: plain copy of the ciphertext (DFF state moves of clocked circuits)
__global__ void eval_not_kernel(const __grid_constant__ DevConst P, const u32 *const *__restrict__ in, u32 *const *__restrict__ out) {
  const uintptr_t raw = reinterpret_cast<uintptr_t>(in[blockIdx.x]);
  const u32 *x = reinterpret_cast<const u32 *>(raw & ~(uintptr_t)15);
  const bool copy = raw & 1;
  u32 *y = out[blockIdx.x];
  const u32 q = P.q, n = P.n;
  for (u32 i = threadIdx.x; i <= n; i += blockDim.x) y[i] = copy ? x[i] : (i == n) ? (q / 4 + q - x[i]) % q : (q - x[i]) % q;
}
int launch_eval_not(const DevConst &P, const u32 *const *d_in, u32 *const *d_out, int count, void *stream) {
  if (count <= 0) return 0;
  eval_not_kernel<<<count, 128, 0, (cudaStream_t)stream>>>(P, d_in, d_out);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// ciphertext ingest: rows that came from outside the program (bfhe_circuit_set_input_ct)
// ------------------------------------------------------------------------------------------
// every word a_0..a_{n-1}, b must be below q (the kernels assume reduced operands); the lowest offending row goes to *bad_row,
// which the host set to 0xffffffff.  Padding words are zeroed.
__global__ void ct_ingest_kernel(const __grid_constant__ DevConst P, u32 *__restrict__ rows, u32 *bad_row) {
  u32 *row = rows + (size_t)blockIdx.x * P.ct_stride;
  bool bad = false;
  for (u32 i = threadIdx.x; i < P.ct_stride; i += blockDim.x) {
    if (i > P.n) row[i] = 0;
    else bad = bad || row[i] >= P.q;
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicMin(bad_row, blockIdx.x);
}
int launch_ct_ingest(const DevConst &P, u32 *d_rows, int count, u32 *d_bad_row, void *stream) {
  if (count <= 0) return 0;
  ct_ingest_kernel<<<count, 128, 0, (cudaStream_t)stream>>>(P, d_rows, d_bad_row);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// bootstrapping-key conversion: canonical coefficient form -> device form
// (forward NTT in this kernel's slot order, times N^-1 * 2^32, laid out [chunk][lane][4] per polynomial)
// ------------------------------------------------------------------------------------------
template <int LOGN> __global__ void __launch_bounds__(128) bk_convert_kernel(const __grid_constant__ DevConst P, const u32 *__restrict__ coef,
                                                                             u32 *__restrict__ dev, size_t npoly,
                                                                             const u32 *__restrict__ g_twl) {
  constexpr int N = 1 << LOGN, E = N / 32;
  __shared__ __align__(16) u32 s_tw[4 * N];
  __shared__ __align__(16) u32 s_buf[4][N];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < 4 * N; i += blockDim.x) s_tw[i] = g_twl[i];
  __syncthreads();
  const TwTabs tt{s_tw, s_tw + N, s_tw + 2 * N, s_tw + 3 * N};
  for (size_t p = (size_t)blockIdx.x * 4 + warp; p < npoly; p += (size_t)gridDim.x * 4) {
    u32 x[E];
#pragma unroll
    for (int k = 0; k < E; k++) x[k] = coef[p * N + lane + 32 * k];
    ntt_forward<LOGN>(x, s_buf[warp], P, tt, lane);
#pragma unroll
    for (int c = 0; c < E / 4; c++) {
      u32 o[4];
#pragma unroll
      for (int r = 0; r < 4; r++) o[r] = csub(mul_shoup(x[4 * c + r], P.nM, P.nMs, P.Q), P.Q);
      *reinterpret_cast<uint4 *>(dev + p * N + (c * 32 + lane) * 4) = make_uint4(o[0], o[1], o[2], o[3]);
    }
    __syncwarp();
  }
}
int launch_bk_convert(const DevConst &P, const u32 *d_coef, u32 *d_dev, size_t npoly, const u32 *d_twl, void *stream) {
  if (npoly == 0) return 0;
  int blocks = (int)((npoly + 3) / 4);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (P.N == 1024) bk_convert_kernel<10><<<blocks, 128, 0, (cudaStream_t)stream>>>(P, d_coef, d_dev, npoly, d_twl);
  else if (P.N == 512) bk_convert_kernel<9><<<blocks, 128, 0, (cudaStream_t)stream>>>(P, d_coef, d_dev, npoly, d_twl);
  else return (int)cudaErrorInvalidValue;
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// folded key copy of the GINX throughput kernel (BrCfg::FOLD): device-form key [step][sign][row][column][N] -> the same layout with the
// top digit's row folded into the others.  With K_r the row that multiplies digit l of accumulator component c (r = c + 2l), T = DG - 1:
//   K'_{c+2l} = K_{c+2l} - B^(l-T) * K_{c+2T}  (l < T),      K'_{c+2T} = N * B^-T * K_{c+2T}      (mod Q, fully reduced)
// Slot by slot, so the [chunk][lane][4] order within a polynomial does not matter.
// ------------------------------------------------------------------------------------------
struct FoldConst {
  u32 w[8]; // w[l] = B^(l-T) mod Q for l < T, w[T] = N * B^-T mod Q
};
template <int DG> __global__ void __launch_bounds__(256) bk_fold_kernel(const u32 *__restrict__ bk, u32 *__restrict__ bkf, size_t total, u32 N, u32 Q,
                                                                        const FoldConst F) {
  constexpr int ROWS = 2 * DG, T = DG - 1;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    // i -> (step and sign, component c, column and slot); row r of polynomial (sign, r, column) sits at r * 2N
    const size_t cs = i % (2 * (size_t)N), c = (i / (2 * (size_t)N)) & 1, ss = i / (4 * (size_t)N);
    const size_t base = ss * ROWS * 2 * N + cs;
    const u64 top = bk[base + (c + 2 * T) * 2 * N];
#pragma unroll
    for (int l = 0; l < T; l++) {
      const size_t o = base + (c + 2 * l) * 2 * N;
      bkf[o] = (u32)(((u64)bk[o] + Q - top * F.w[l] % Q) % Q);
    }
    bkf[base + (c + 2 * T) * 2 * N] = (u32)(top * F.w[T] % Q);
  }
}
static u64 powmod_q(u64 b, u64 e, u64 Q) {
  u64 r = 1;
  for (b %= Q; e; e >>= 1, b = b * b % Q)
    if (e & 1) r = r * b % Q;
  return r;
}
bool bk_fold_supported(const DevConst &P, int method_ap) { return !method_ap && P.N == 1024 && P.dG == 4 && P.logBG == 7; }
int launch_bk_fold(const DevConst &P, const u32 *d_bk, u32 *d_bkf, size_t nsteps, void *stream) {
  if (!bk_fold_supported(P, 0)) return (int)cudaErrorInvalidValue;
  constexpr int DG = 4, T = DG - 1;
  FoldConst F{};
  const u64 Q = P.Q, binv = powmod_q(1ull << P.logBG, Q - 2, Q);
  for (int l = 0; l < T; l++) F.w[l] = (u32)powmod_q(binv, T - l, Q);
  F.w[T] = (u32)((u64)P.N * powmod_q(binv, T, Q) % Q);
  const size_t total = nsteps * 2 * 2 * 2 * (size_t)P.N; // (step, sign) x component x (column, slot)
  bk_fold_kernel<DG><<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_bk, d_bkf, total, P.N, P.Q, F);
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// debug / parity kernel: rt = INTT(NTT(a)), prod = a (*) b negacyclic, through the same transforms
// ------------------------------------------------------------------------------------------
template <int LOGN> __global__ void __launch_bounds__(32) dbg_ntt_kernel(const __grid_constant__ DevConst P, const u32 *__restrict__ a,
                                                                         const u32 *__restrict__ b, u32 *__restrict__ rt,
                                                                         u32 *__restrict__ prod, const u32 *__restrict__ g_twl) {
  constexpr int N = 1 << LOGN, E = N / 32;
  __shared__ __align__(16) u32 s_tw[4 * N];
  __shared__ __align__(16) u32 s_buf[N];
  const int lane = threadIdx.x;
  for (int i = lane; i < 4 * N; i += 32) s_tw[i] = g_twl[i];
  __syncwarp();
  const TwTabs tt{s_tw, s_tw + N, s_tw + 2 * N, s_tw + 3 * N};
  const size_t p = blockIdx.x;
  const u32 Q = P.Q;
  u32 x[E], y[E];
#pragma unroll
  for (int k = 0; k < E; k++) x[k] = a[p * N + lane + 32 * k];
  ntt_forward<LOGN>(x, s_buf, P, tt, lane);
#pragma unroll
  for (int k = 0; k < E; k++) y[k] = csub(lazy_reduce(x[k], Q), Q);
  {
    u32 z[E];
#pragma unroll
    for (int k = 0; k < E; k++) z[k] = y[k];
    __syncwarp();
    ntt_inverse<LOGN, 2>(z, s_buf, P, tt, lane);
#pragma unroll
    for (int k = 0; k < E; k++) rt[p * N + lane + 32 * k] = csub(mul_shoup(z[k], P.ninv, P.ninvs, Q), Q);
  }
  if (b) {
    u32 z[E];
#pragma unroll
    for (int k = 0; k < E; k++) z[k] = b[p * N + lane + 32 * k];
    __syncwarp();
    ntt_forward<LOGN>(z, s_buf, P, tt, lane);
#pragma unroll
    for (int k = 0; k < E; k++) z[k] = (u32)(((u64)csub(lazy_reduce(z[k], Q), Q) * y[k]) % Q);
    __syncwarp();
    ntt_inverse<LOGN, 2>(z, s_buf, P, tt, lane);
#pragma unroll
    for (int k = 0; k < E; k++) prod[p * N + lane + 32 * k] = csub(mul_shoup(z[k], P.ninv, P.ninvs, Q), Q);
  }
}
int launch_dbg_ntt(const DevConst &P, const u32 *d_a, const u32 *d_b, u32 *d_rt, u32 *d_prod, int npoly, const u32 *d_twl,
                   void *stream) {
  if (npoly <= 0) return 0;
  if (P.N == 1024) dbg_ntt_kernel<10><<<npoly, 32, 0, (cudaStream_t)stream>>>(P, d_a, d_b, d_rt, d_prod, d_twl);
  else if (P.N == 512) dbg_ntt_kernel<9><<<npoly, 32, 0, (cudaStream_t)stream>>>(P, d_a, d_b, d_rt, d_prod, d_twl);
  else return (int)cudaErrorInvalidValue;
  return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// integer-pipe microbenchmark (roofline denominator: measured multiply-class instruction rate)
// ------------------------------------------------------------------------------------------
template <int WHICH> __global__ void __launch_bounds__(256) microbench_kernel(u32 *sink, int iters) {
  constexpr int U = 16;
  u32 a[U], b = sink[0] | 1u, c = sink[1];
  u64 wacc[U];
#pragma unroll
  for (int i = 0; i < U; i++) { a[i] = threadIdx.x * 2654435761u + i; wacc[i] = a[i]; }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < U; i++) {
      if (WHICH == 0) a[i] = a[i] * b + c;                        // IMAD
      else if (WHICH == 1) a[i] = __umulhi(a[i], b) + c;          // IMAD.HI
      else if (WHICH == 2) wacc[i] += (u64)(u32)wacc[i] * b;      // IMAD.WIDE with 64-bit accumulate
      else if (WHICH == 3) a[i] = min(a[i] + c, a[i] ^ b);        // ALU pipe pair (IADD3 + LOP3 + VIMNMX)
      else { u32 t = mul_shoup(a[i], b, c, 134215681u); a[i] = a[i] + t; } // Shoup butterfly half
    }
  }
  u32 r = 0;
#pragma unroll
  for (int i = 0; i < U; i++) r ^= a[i] ^ (u32)wacc[i] ^ (u32)(wacc[i] >> 32);
  if (r == 0x12345678u) sink[2] = r;
}
int launch_microbench(int which, u32 *d_sink, int iters, int *threads_total, int *ops_per_thread_iter, void *stream) {
  const int blocks = 148 * 8, threads = 256;
  *threads_total = blocks * threads;
  *ops_per_thread_iter = 16;
  cudaStream_t st = (cudaStream_t)stream;
  switch (which) {
  case 0: microbench_kernel<0><<<blocks, threads, 0, st>>>(d_sink, iters); break;
  case 1: microbench_kernel<1><<<blocks, threads, 0, st>>>(d_sink, iters); break;
  case 2: microbench_kernel<2><<<blocks, threads, 0, st>>>(d_sink, iters); break;
  case 3: microbench_kernel<3><<<blocks, threads, 0, st>>>(d_sink, iters); break;
  default: microbench_kernel<4><<<blocks, threads, 0, st>>>(d_sink, iters); break;
  }
  return (int)cudaGetLastError();
}

} // namespace bfhe
