// kernels_cl.cu -- GINX blind rotation of ONE gate on a 4-CTA thread-block cluster with ONE exchange per step ("slot-sliced" form).
// STD128_OPT shape (N = 1024, dG = 4, Bg = 2^7).  Same arithmetic as blind_rotate_kernel in kernels.cu (SURVEY.md 8(a) rows a8-a15; the
// reference reaches it through BinFHEContext::EvalBinGate, src/gate.cpp:133,172,200-202 in /root/reference).
//
// Round 1's cluster kernels split a step by ROWS for the transforms and by SLOTS for the external product, which costs two all-to-all
// exchanges over DSMEM per step (digit rows out, product rows back); ncu showed them waiting on those exchanges 35 % of the time
// (profiles/r1_blind_rotate_cluster4_ncu_summary.md).  This kernel slices everything by evaluation slot instead.  Write the transform of
// size N as (two stages across the four blocks of N/4 coefficients) o (four independent sub-transforms of size N/4):
//
//   * every CTA keeps the WHOLE accumulator (both components, coefficient form);
//   * CTA k computes, for all 8 digit polynomials, only block k of the two cross-block stages -- straight from the digits with three
//     table look-ups per value (digit x {w1, w2, w1 w2} precomputed for the 128 digit values), no multiplication -- and then its own
//     256-point sub-transform of each (one warp per digit polynomial, 8 values per lane: 3 + 3 + 2 register stages, two shared-memory
//     transposes);
//   * it multiplies ITS 256 slots of the 8 rows with ITS quarter of the step's key tile (32 KB, TMA bulk copy, double buffered, issued
//     two steps ahead), and runs the 256-point inverse sub-transform of the two product components;
//   * the only exchange: the 2 x 256 partial values go to the three peers (st.async, counted on the receiver's mbarrier, 6 KB in and
//     out per CTA and step); every CTA then finishes the inverse transform redundantly (two cross-block stages), adds to its copy of the
//     accumulator and cuts the next digits.
//
// Third revision (round 2).  In the second revision every phase was fenced from the next by a CTA barrier, one warp per component ran the
// last inverse stages before the exchange, and the key words came through LDG into registers (which stalled the look-up phase behind
// the loads once 30 clusters shared the L2).  Now:
//   * warps 4 c .. 4 c + 3 ("group c", 128 threads, one warp per scheduler) own accumulator component c: they hold its 1 024 coefficients
//     in registers, and everything that concerns only that component is ordered by 128-thread named barriers and by the component's own
//     mbarrier: the cross-block inverse stages, publishing centred + offset words in shared memory, cutting digit row c + 2 l out of them
//     (warp 4 c + l), the table look-ups and that row's sub-transform straight from registers.  The two groups meet once per step, at the
//     barrier in front of the external product;
//   * the product is split by component as well: group c computes component c at two adjacent slots per thread, which makes the first
//     inverse stage a register operation and the next five shuffles on two independent values; every thread then pushes its two values to
//     the three peers itself (8-byte st.async counted on the receiver's mbarrier) -- measured against TMA bulk copies of the finished 1 KB
//     row by a dedicated warp (shared::cta -> shared::cluster): 0.975 vs 1.000 ms, the hand-off to an issuing warp (barrier, proxy fence,
//     three copies) cost ~300 cycles of every step's critical path;
//   * the two remaining stages of the 256-point inverse sub-transforms run AFTER the exchange, on all four rows at once (warp l of group c
//     takes the row that came from CTA l);
//   * a ninth warp fetches the key tiles (32 KB per step and CTA, two TMA bulk copies, two steps ahead, double buffered); the product
//     reads them with one conflict-free LDS.128 per four rows.
// Per-step timeline and phase costs: tools/phase_timing.py (build with -DBFHE_PHASE_TIMING), profiles/r2_clx_*.
// No cluster-scope fence or barrier.cluster inside the step loop; receive buffers and their mbarriers alternate by step parity, so a
// CTA that runs one step ahead cannot overwrite or miscount data its peer is still reading.
#include "device.cuh"

namespace bfhe {
namespace clx {

constexpr int LOGN = 10, N = 1 << LOGN, DG = 4, LOGBG = 7, ROWS = 2 * DG, R = 4, NB = N / R, THREADS = 288; // 8 main warps + the warp that fetches the key tiles
constexpr int KEYPOLYS = 2 * ROWS * 2; // GINX: two RGSW ciphertexts (X^a, X^-a) per step; AP: one (KEYPOLYS / 2 polynomials)
constexpr int NSTEP_PAD = 1024;     // >= n (GINX) and >= n * dR (AP)
constexpr u32 DIGIT_OFF = 64u + (64u << 7) + (64u << 14) + (64u << 21);

// per-rank twiddle block (host-generated, engine.cu): fw[TWF] | fws[TWF] | iw[TWI] | iws[TWI]
//   fw:  [0, 8)            pass A (register stages across the 32-strided values), uniform over the warp: w[1], w[2..3], w[4..7]
//        [8, 264)          pass B (lane = 4 blk + q holds positions 32 blk + q + 4 m), [chunk 2][lane 32][4]: w[1], w[2..3], w[4..7] per lane
//        [264, 520)        pass C (lane holds positions 8 lane .. 8 lane + 7), same layout: w[2..3], w[4..7] per lane
//   iw:  [0, 8)            inverse pass A, uniform
//        [8 + 256 s, ..)   s = 0..4: the inverse stage with half-size 2^s for MAC slot t (the five stages done by shuffles), [t]
constexpr int TWF = 8 + 2 * 256, TWI = 8 + 5 * 256, TWR = 2 * TWF + 2 * TWI;

// ---- 8-value register stages.  Stage with half-size T pairs a = g * 2T + (i % T), b = a + T and uses twiddle w[8 / (2T) + g] ----
template <int T> __device__ __forceinline__ void ct8_stage(u32 (&x)[8], const u32 (&w)[8], const u32 (&ws)[8], u32 Q, u32 Q2) {
  u32 t[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int g = i / T, b = g * 2 * T + (i % T) + T, p = 4 / T + g;
    t[i] = mul_shoup(x[b], w[p], ws[p], Q);
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int g = i / T, a = g * 2 * T + (i % T), b = a + T;
    x[b] = x[a] - t[i] + Q2; // no range correction: values grow by 2Q per stage and stay below 2^32 (21Q after all ten stages)
    x[a] = x[a] + t[i];
  }
}
// Gentleman-Sande stage; B = bound of the inputs in units of Q.  Sums double per stage and are pulled back below 2Q when they would pass 32Q
// at the next stage (compile-time bound tracking through OUTB).
template <int B> struct GsShfl1 { // one inverse stage across lanes `mask` apart on ONE value per thread; the upper lane holds b
  static constexpr bool RED = (2 * B > 16);
  static constexpr int OUTB = RED ? 2 : 2 * B;
  __device__ __forceinline__ static u32 run(u32 x, u32 w, u32 ws, u32 Q, int mask, bool upper) {
    static_assert(B <= 16, "GS input bound too large");
    const u32 o = __shfl_xor_sync(0xffffffffu, x, mask);
    const u32 pr = mul_shoup(o - x + B * Q, w, ws, Q); // upper lane: (lower - upper) * w
    const u32 S = x + o;
    return upper ? pr : (RED ? lazy_reduce(S, Q) : S);
  }
};
__device__ __forceinline__ void load8(const u32 *tab, u32 (&w)[8], int lane) { // [chunk 2][lane 32][4]
  const uint4 a = reinterpret_cast<const uint4 *>(tab)[lane], b = reinterpret_cast<const uint4 *>(tab)[32 + lane];
  w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
}
// word offset of position i (0..255) of a sub-transform row: 32-word groups rotated by 4 * group, so that both the 32-strided access of
// pass A (i = lane + 32 m) and the 4-strided access of pass B (i = 32 blk + q + 4 m', lane = 4 blk + q) are bank-conflict free
__device__ __forceinline__ int rowpos(int i) { return (i & ~31) | ((i + 4 * (i >> 5)) & 31); }

// in-place position (0 .. N-1, Cooley-Tukey order: slot P holds the evaluation at psi^(2 bitrev(P) + 1)) of MAC slot t of CTA k
__host__ __device__ __forceinline__ int slot_position(int k, int t) { return NB * k + t; }

struct Smem { // word offsets
  static constexpr int rbuf = 0;                              // [parity 2][source CTA R][component 2][NB]
  static constexpr int dct = rbuf + 2 * R * 2 * NB;           // [parity 2][ROWS][NB]
  static constexpr int pbuf = dct + 2 * ROWS * NB;            // [component 2][source CTA R][NB] rows after the last sub-transform stages
  static constexpr int accs = pbuf + 2 * R * NB;              // [2][N] centred accumulator + digit offset
  static constexpr int lut = accs + 2 * N;                    // [3][128][32]
  static constexpr int F = lut + 3 * 128 * 32;                // [2N]
  static constexpr int key = F + 2 * N;                       // [parity 2][8 quads][NB][4]
  static constexpr int idx = key + 2 * KEYPOLYS * NB;         // u16 [NSTEP_PAD] monomial exponent (GINX) / digit (AP) per step
  static constexpr int list = idx + NSTEP_PAD / 2;            // u16 [NSTEP_PAD] AP: the steps that do work (digit != 0)
  static constexpr int bars = list + NSTEP_PAD / 2;           // rbar[parity 2][component 2], kbar[2]
  static constexpr int words = bars + 12;
  static constexpr size_t bytes = (size_t)words * 4;
};
static_assert(Smem::key % 32 == 0 && Smem::bars % 2 == 0, "TMA destination 128-byte aligned, mbarriers 8-byte aligned");
constexpr u32 KEYBYTES = KEYPOLYS * NB * 4;     // this CTA's quarter of one step's key tile (GINX; AP: half of it)
constexpr u32 RECV_TX_C = (u32)(R - 1) * NB * 4; // bytes the three peers push into a CTA per step and component

// named barriers (0 is left to __syncthreads in the prologue)
constexpr int BAR_DCT = 1, BAR_GROUP = 2 /* + c */, BAR_KEY = 4;

template <bool AP>
__global__ void __cluster_dims__(R, 1, 1) __launch_bounds__(THREADS, 1)
blind_rotate_clx_kernel(const __grid_constant__ DevConst P, const DevGate *__restrict__ gates, int count, const u32 *__restrict__ bkx,
                        const u32 *__restrict__ g_tw, const u32 *__restrict__ g_F, u32 *__restrict__ ext, u32 *__restrict__ acc_dbg) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  u32 *sm = reinterpret_cast<u32 *>(smem_raw);
  u32 *rbuf = sm + Smem::rbuf, *dct = sm + Smem::dct, *pbuf = sm + Smem::pbuf, *accs = sm + Smem::accs, *s_lut = sm + Smem::lut, *s_F = sm + Smem::F,
      *s_key = sm + Smem::key;
  u16 *s_idx = reinterpret_cast<u16 *>(sm + Smem::idx), *s_list = reinterpret_cast<u16 *>(sm + Smem::list);
  u64 *rbar = reinterpret_cast<u64 *>(sm + Smem::bars); // [parity][component]
  u64 *kbar = rbar + 4;
  __shared__ u32 s_b, s_nact;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 k = cluster_rank();
  const size_t gi = blockIdx.x / R;
  const u32 Q = P.Q, Q2 = P.Q2, q = P.q, n = P.n, qinv = P.qinv_neg;
  const DevGate dg = gates[gi];

  if (tid == 0) {
    for (int i = 0; i < 4; i++) mbar_init(rbar + i, 128); // one arrival per thread of the group that owns the component
    mbar_init(kbar + 0, 1); mbar_init(kbar + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (!AP)
    for (int i = tid; i < 2 * N; i += THREADS) s_F[i] = g_F[i];
  { // look-up tables of the two cross-block forward stages for block k: y_k = d0 + c1 d2 + c2 d1 + c3 d3 with
    //   k = 0: (+w1, +w2, +w2 w1)   k = 1: (+w1, -w2, -w2 w1)   k = 2: (-w1, +w3, -w3 w1)   k = 3: (-w1, -w3, +w3 w1)
    // (w1 = psi^bitrev(1), w2 = psi^bitrev(2), w3 = psi^bitrev(3): the twiddles of the stages with 1 and 2 groups), entries
    // c * (digit - B/2) mod Q for the 128 digit values, one copy per bank
    const u64 w1 = P.tw[1], wb = (k & 2) ? P.tw[3] : P.tw[2];
    const u64 c1 = (k & 2) ? Q - w1 : w1;
    const u64 c2 = (k & 1) ? Q - wb : wb;
    u64 c3 = wb * w1 % Q;
    if (k == 1 || k == 2) c3 = Q - c3;
    for (int e = tid; e < 3 * 128; e += THREADS) {
      const int tab = e >> 7, d = e & 127;
      const u64 c = tab == 0 ? c1 : tab == 1 ? c2 : c3;
      const u32 v = (u32)(c * (u64)((d + Q - 64) % Q) % Q);
#pragma unroll 4
      for (int l = 0; l < 32; l++) s_lut[e * 32 + l] = v;
    }
  }
  { // LWE prep, as in the other kernels (every CTA of the cluster computes it)
    const u32 gate = dg.op & 0xff;
    for (u32 i = tid; i <= n; i += THREADS) {
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
      else if (!AP) s_idx[i] = (u16)(((q - v) % q) * P.factor);
      else { // AP: digits of -a_i in base B_r, one step each; BK[i][digit][k] (digit 0: nothing to do)
        u32 a = (q - v) % q;
        for (u32 kk = 0; kk < P.dR; kk++, a /= P.baseR) s_idx[i * P.dR + kk] = (u16)(a % P.baseR);
      }
    }
  }
  __syncthreads();
  if (AP && tid == 0) { // the steps that do work, in order
    u32 na = 0;
    for (u32 st = 0; st < n * P.dR; st++)
      if (s_idx[st] != 0) s_list[na++] = (u16)st;
    s_nact = na;
  }
  if (AP) __syncthreads();
  const u32 nact = AP ? s_nact : n; // iterations of the main loop

  auto issue_keys = [&](u32 j) { // one thread: this CTA's key tile of iteration j (GINX 32 KB, AP 16 KB), contiguous in the sliced copy
    u64 *bar = kbar + (j & 1);
    u32 *dst = s_key + (size_t)(j & 1) * KEYPOLYS * NB;
    if (!AP) {
      mbar_expect_tx(bar, KEYBYTES);
      const u32 *src = bkx + ((size_t)j * R + k) * KEYPOLYS * NB;
      bulk_g2s(dst, src, 16384, bar);
      bulk_g2s(dst + 4096, src + 4096, 16384, bar);
    } else {
      const u32 st = s_list[j], a0 = s_idx[st], i = st / P.dR, kk = st % P.dR;
      const size_t keyi = ((size_t)i * (P.baseR - 1) + (a0 - 1)) * P.dR + kk;
      mbar_expect_tx(bar, KEYBYTES / 2);
      bulk_g2s(dst, bkx + (keyi * R + k) * (KEYPOLYS / 2) * NB, 16384, bar);
    }
  };
  static_assert(KEYBYTES == 2 * 16384, "two bulk copies");

  const u32 *twr = g_tw + (size_t)k * TWR, *g_fw = twr, *g_fws = twr + TWF, *g_iw = twr + 2 * TWF, *g_iws = twr + 2 * TWF + TWI;
#ifdef BFHE_PHASE_TIMING
  long long tph[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tc0 = clock64(), tc1;
  u32 tstamp[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tstep = 0; // absolute clock (low 32 bits) of every mark in step 200: one step's timeline
#define CLX_T(i) do { tc1 = clock64(); tph[i] += tc1 - tc0; tc0 = tc1; if (tstep == 200) tstamp[i] = (u32)tc1; } while (0)
#else
#define CLX_T(i)
#endif

  if (warp >= 8) {
    // ================= ninth warp: fetches the key tiles (TMA bulk copies, two steps ahead) =================
    if (lane == 0 && nact > 0) {
      issue_keys(0);
      if (nact > 1) issue_keys(1);
    }
    cluster_sync_all(); // every CTA's mbarriers are initialised before anything is pushed
    for (u32 step = 0; step + 2 < nact; step++) {
      bar_sync(BAR_KEY, 256 + 32); // all product threads are through with this step's key tile
      if (lane == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // their reads of the buffer, before the async proxy overwrites it
        issue_keys(step + 2);
      }
    }
    cluster_sync_all(); // a CTA must not exit while its peers may still push into its shared memory
    return;
  }

  // ================= main warps: warp 4 c + l transforms row c + 2 l; group c = warps 4 c .. 4 c + 3, one per scheduler =================
  const int c = warp >> 2, l = warp & 3, gt = l * 32 + lane; // gt: index inside the group, 0..127
  // accumulator: group c, thread gt holds coefficients gt + 128 jj + 256 i1 of component c, canonical [0, Q)
  u32 acc[2][4];
  {
    const u32 gate = dg.op & 0xff;
    const u32 q1 = P.gate_const[gate == OP_BOOTSTRAP ? OP_AND : gate], q2 = (q1 + q / 2) % q, b = s_b;
#pragma unroll
    for (int jj = 0; jj < 2; jj++)
#pragma unroll
      for (int i1 = 0; i1 < 4; i1++) {
        const u32 idx = gt + 128 * jj + NB * i1;
        u32 v = 0;
        if (c == 1 && idx % P.factor == 0) {
          const u32 t = (b + q - idx / P.factor) % q;
          const bool in = (q1 < q2) ? (t >= q1 && t < q2) : !(t >= q2 && t < q1);
          v = in ? Q - P.Q8 : P.Q8;
        }
        acc[jj][i1] = v;
        accs[c * N + idx] = ((v < (Q >> 1)) ? v : v - Q) + DIGIT_OFF; // centred + offset
      }
  }
  // ---- per-thread constants, kept in registers for the whole blind rotation ----
  // product: group c computes component c at slots 2 gt and 2 gt + 1 (slot t evaluates at psi^ex(t))
  const u32 ex0 = 2 * (__brev((u32)slot_position((int)k, 2 * gt)) >> (32 - LOGN)) + 1, ex1 = 2 * (__brev((u32)slot_position((int)k, 2 * gt + 1)) >> (32 - LOGN)) + 1;
  u32 fA[8], fAs[8], fB[8], fBs[8], fC[8], fCs[8], iS[5][2], iSs[5][2];
#pragma unroll
  for (int p = 0; p < 8; p++) { fA[p] = g_fw[p]; fAs[p] = g_fws[p]; }
  load8(g_fw + 8, fB, lane); load8(g_fws + 8, fBs, lane);
  load8(g_fw + 8 + 256, fC, lane); load8(g_fws + 8 + 256, fCs, lane);
#pragma unroll
  for (int s5 = 0; s5 < 5; s5++) // inverse stage with half-size 2^s5 at my two slots (s5 = 0 pairs them: one twiddle, the upper slot's entry)
#pragma unroll
    for (int e = 0; e < 2; e++) { iS[s5][e] = g_iw[8 + 256 * s5 + 2 * gt + e]; iSs[s5][e] = g_iws[8 + 256 * s5 + 2 * gt + e]; }
  const u32 iS5 = g_iw[4 + l], iS5s = g_iws[4 + l]; // half-size 32: one twiddle per 64 slots
  const u32 iw1 = P.itw[1], iw1s = P.itws[1], iwb = P.itw[2], iwbs = P.itws[2], iwc = P.itw[3], iwcs = P.itws[3];
  u32 iA[8], iAs[8]; // last three stages of the inverse sub-transform of block l (the row that CTA l sends)
#pragma unroll
  for (int p = 0; p < 8; p++) { iA[p] = g_tw[(size_t)l * TWR + 2 * TWF + p]; iAs[p] = g_tw[(size_t)l * TWR + 2 * TWF + TWI + p]; }
  const int blk = lane >> 2, qq = lane & 3;
  const u32 dsh = (u32)(LOGBG * l); // my row's digit
  u32 peer_mine[R - 1], peer_bar[R - 1]; // shared::cluster addresses in the three peers: my two words of this CTA's row of component c (parity 0), rbar[0][c]
#pragma unroll
  for (int p = 0; p < R - 1; p++) {
    const u32 dest = (k + 1 + p) % R;
    peer_mine[p] = dsmem_addr(rbuf + (size_t)(k * 2 + c) * NB + 2 * gt, dest);
    peer_bar[p] = dsmem_addr(rbar + c, dest);
  }
  cluster_sync_all(); // every CTA's mbarriers are initialised before anything is pushed

  for (u32 step = 0; step < nact; step++) { // (AP: `step` counts the steps that do work; s_list[step] is the blind-rotation step)
    const u32 par = step & 1;
#ifdef BFHE_PHASE_TIMING
    tstep = step;
#endif
    // the key tile of this step was requested two steps ago: test its barrier once now (the ~100 cycles of a try_wait then overlap the
    // transform); the monomial factors do not depend on the transform either
    const bool key_in = mbar_test(kbar + par, (step >> 1) & 1);
    const u32 mexp = AP ? 0u : (u32)s_idx[step];
    const u32 mono0 = mexp * ex0, mono1 = mexp * ex1; // GINX: (X^m - 1), (X^-m - 1) at my two slots, Montgomery form
    const u32 fp[2] = {AP ? 0u : s_F[f_index(mono0)], AP ? 0u : s_F[f_index(mono1)]},
              fn[2] = {AP ? 0u : s_F[f_index(0u - mono0)], AP ? 0u : s_F[f_index(0u - mono1)]};
    // ---- phase A: my group's accumulator words are published -> block k of the two cross-block forward stages of MY row, by look-up ----
    bar_sync(BAR_GROUP + c, 128);
    CLX_T(0);
    u32 *row = dct + (par * ROWS + c + 2 * l) * NB;
    {
      u32 x[8];
      const u32 *ap = accs + c * N + lane;
#pragma unroll
      for (int m = 0; m < 8; m++) {
        const u32 d0 = (ap[32 * m] >> dsh) & 127u, d1 = (ap[32 * m + NB] >> dsh) & 127u, d2 = (ap[32 * m + 2 * NB] >> dsh) & 127u,
                  d3 = (ap[32 * m + 3 * NB] >> dsh) & 127u;
        x[m] = (d0 + (Q - 64u)) + s_lut[((0 * 128 + d2) << 5) + lane] + s_lut[((1 * 128 + d1) << 5) + lane] + s_lut[((2 * 128 + d3) << 5) + lane]; // < 4Q + 64
      }
      CLX_T(1);
      // ---- phase B: the row's 256-point sub-transform, 8 values per lane: 3 + 3 + 2 register stages, two in-place transposes ----
      ct8_stage<4>(x, fA, fAs, Q, Q2); ct8_stage<2>(x, fA, fAs, Q, Q2); ct8_stage<1>(x, fA, fAs, Q, Q2);
#pragma unroll
      for (int m = 0; m < 8; m++) row[rowpos(lane + 32 * m)] = x[m];
      __syncwarp();
#pragma unroll
      for (int m = 0; m < 8; m++) x[m] = row[rowpos(32 * blk + qq + 4 * m)];
      ct8_stage<4>(x, fB, fBs, Q, Q2); ct8_stage<2>(x, fB, fBs, Q, Q2); ct8_stage<1>(x, fB, fBs, Q, Q2);
#pragma unroll
      for (int m = 0; m < 8; m++) row[rowpos(32 * blk + qq + 4 * m)] = x[m];
      __syncwarp();
      {
        const uint4 a = *reinterpret_cast<const uint4 *>(row + rowpos(8 * lane)), b = *reinterpret_cast<const uint4 *>(row + rowpos(8 * lane + 4));
        x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
      }
      ct8_stage<2>(x, fC, fCs, Q, Q2); ct8_stage<1>(x, fC, fCs, Q, Q2);
      __syncwarp(); // every lane has read its pass-C inputs before the row is overwritten in slot order
      *reinterpret_cast<uint4 *>(row + 8 * lane) = make_uint4(x[0], x[1], x[2], x[3]); // MAC slot t = position t
      *reinterpret_cast<uint4 *>(row + 8 * lane + 4) = make_uint4(x[4], x[5], x[6], x[7]);
    }
    CLX_T(2);
    bar_sync(BAR_DCT, 256); // all eight rows of this step are in dct[par]
    CLX_T(3);
    // ---- phase C: external product, group c computes component c: two adjacent slots per thread; then the six inverse stages that stay
    //      inside a warp (the first inside the thread, five by shuffle, two independent values per stage); the finished values go straight
    //      into this CTA's row of the receive buffer ----
    if (!key_in) mbar_wait(kbar + par, (step >> 1) & 1);
    CLX_T(4);
    {
      uint2 d[ROWS];
#pragma unroll
      for (int rw = 0; rw < ROWS; rw++) d[rw] = *reinterpret_cast<const uint2 *>(dct + (par * ROWS + rw) * NB + 2 * gt);
      // key tile: [quad g = (cc * 2 + sign) * 2 + half][slot parity e][gt][4 rows]
      // (AP: one RGSW ciphertext per step -- quad g = cc * 2 + half, no sign)
      const uint4 *k4 = reinterpret_cast<const uint4 *>(s_key + (size_t)par * KEYPOLYS * NB) + (size_t)c * (AP ? 2 : 4) * 2 * 128 + gt;
      u64 s2[2][2] = {{0, 0}, {0, 0}}; // [slot parity][sign]
#pragma unroll
      for (int sg = 0; sg < (AP ? 1 : 2); sg++)
#pragma unroll
        for (int hf = 0; hf < 2; hf++) {
          const uint4 k0 = k4[((sg * 2 + hf) * 2 + 0) * 128], k1 = k4[((sg * 2 + hf) * 2 + 1) * 128];
          s2[0][sg] += (u64)d[4 * hf + 0].x * k0.x; s2[1][sg] += (u64)d[4 * hf + 0].y * k1.x;
          s2[0][sg] += (u64)d[4 * hf + 1].x * k0.y; s2[1][sg] += (u64)d[4 * hf + 1].y * k1.y;
          s2[0][sg] += (u64)d[4 * hf + 2].x * k0.z; s2[1][sg] += (u64)d[4 * hf + 2].y * k1.z;
          s2[0][sg] += (u64)d[4 * hf + 3].x * k0.w; s2[1][sg] += (u64)d[4 * hf + 3].y * k1.w;
        }
      u32 v0, v1; // < 2Q
      if (AP) { // one Montgomery reduction of a sum of 8 products of (< 21 Q) x (< Q): < 7 Q, pulled back below 2 Q
        v0 = lazy_reduce(redc(s2[0][0], Q, qinv), Q); v1 = lazy_reduce(redc(s2[1][0], Q, qinv), Q);
      }
      else {
        v0 = redc((u64)redc(s2[0][0], Q, qinv) * fp[0] + (u64)redc(s2[0][1], Q, qinv) * fn[0], Q, qinv);
        v1 = redc((u64)redc(s2[1][0], Q, qinv) * fp[1] + (u64)redc(s2[1][1], Q, qinv) * fn[1], Q, qinv);
      }
      CLX_T(5);
      { // half-size 1: my two slots are the pair (bound 2 -> 4)
        const u32 df = v0 - v1 + 2 * Q;
        v0 = v0 + v1;
        v1 = mul_shoup(df, iS[0][1], iSs[0][1], Q);
      }
      using T1 = GsShfl1<4>; using T2 = GsShfl1<T1::OUTB>; using T3 = GsShfl1<T2::OUTB>; using T4 = GsShfl1<T3::OUTB>; using T5 = GsShfl1<T4::OUTB>;
      static_assert(T5::OUTB <= 8, "bound of the values handed to the last two inverse stages");
      v0 = T1::run(v0, iS[1][0], iSs[1][0], Q, 1, (lane & 1) != 0); v1 = T1::run(v1, iS[1][1], iSs[1][1], Q, 1, (lane & 1) != 0);
      v0 = T2::run(v0, iS[2][0], iSs[2][0], Q, 2, (lane & 2) != 0); v1 = T2::run(v1, iS[2][1], iSs[2][1], Q, 2, (lane & 2) != 0);
      v0 = T3::run(v0, iS[3][0], iSs[3][0], Q, 4, (lane & 4) != 0); v1 = T3::run(v1, iS[3][1], iSs[3][1], Q, 4, (lane & 4) != 0);
      v0 = T4::run(v0, iS[4][0], iSs[4][0], Q, 8, (lane & 8) != 0); v1 = T4::run(v1, iS[4][1], iSs[4][1], Q, 8, (lane & 8) != 0);
      v0 = T5::run(v0, iS5, iS5s, Q, 16, (lane & 16) != 0); v1 = T5::run(v1, iS5, iS5s, Q, 16, (lane & 16) != 0);
#pragma unroll
      for (int p = 0; p < R - 1; p++) st_async2(peer_mine[p] + par * (u32)(R * 2 * NB * 4), make_uint2(v0, v1), peer_bar[p] + 16u * par);
      *reinterpret_cast<uint2 *>(rbuf + (size_t)((par * R + k) * 2 + c) * NB + 2 * gt) = make_uint2(v0, v1);
      // 128 arrivals per step and component release the CTA's own row to group c; one of them also posts the bytes expected from the three
      // peers (stores that landed earlier merely ran the count negative)
      if (gt == 0) mbar_expect_tx(rbar + par * 2 + c, RECV_TX_C);
      else mbar_arrive(rbar + par * 2 + c);
      if (step + 2 < nact) bar_arrive(BAR_KEY, 256 + 32); // the ninth warp may overwrite this step's key tile
    }
    CLX_T(6);
    // ---- phase E: my component's four partial rows have landed (mine stored above, the peers' by bulk copy).  Warp l of the group runs the
    //      last three stages of the inverse sub-transform on the row that came from CTA l; then, across the rows, the two cross-block
    //      stages for coefficients gt + 128 jj + 256 i1; accumulate; publish centred + offset ----
    mbar_wait(rbar + par * 2 + c, (step >> 1) & 1);
    CLX_T(7);
    { // (not in place: this CTA's own row is still the source of bulk copies that may be in flight)
      const u32 *rrow = rbuf + (size_t)((par * R + l) * 2 + c) * NB + lane;
      u32 *prow = pbuf + (size_t)(c * R + l) * NB + lane;
#pragma unroll
      for (int jj = 0; jj < 2; jj++) { // values t + 64 j, t = lane + 32 jj: half-size 64 (twiddle 2 + (j >> 1)), then half-size 128 (twiddle 1)
        u32 x0 = rrow[32 * jj], x1 = rrow[32 * jj + 64], x2 = rrow[32 * jj + 128], x3 = rrow[32 * jj + 192]; // < 8Q
        const u32 d01 = mul_shoup(x0 - x1 + 8 * Q, iA[2], iAs[2], Q), d23 = mul_shoup(x2 - x3 + 8 * Q, iA[3], iAs[3], Q); // < 2Q
        const u32 s01 = x0 + x1, s23 = x2 + x3;                                                                          // < 16Q
        prow[32 * jj] = lazy_reduce(s01 + s23, Q);                                                                       // < 2Q
        prow[32 * jj + 128] = mul_shoup(s01 - s23 + 16 * Q, iA[1], iAs[1], Q);
        prow[32 * jj + 64] = d01 + d23;                                                                                  // < 4Q
        prow[32 * jj + 192] = mul_shoup(d01 - d23 + 2 * Q, iA[1], iAs[1], Q);
      }
    }
    bar_sync(BAR_GROUP + c, 128);
    CLX_T(9);
#pragma unroll
    for (int jj = 0; jj < 2; jj++) {
      const u32 *rb = pbuf + (size_t)c * R * NB + gt + 128 * jj;
      const u32 p0 = rb[0 * NB], p1 = rb[1 * NB], p2 = rb[2 * NB], p3 = rb[3 * NB]; // partial values of blocks 0..3, < 4Q
      const u32 u0 = p0 + p1, u1 = mul_shoup(p0 - p1 + 4 * Q, iwb, iwbs, Q);
      const u32 u2 = p2 + p3, u3 = mul_shoup(p2 - p3 + 4 * Q, iwc, iwcs, Q);
      const u32 x0 = u0 + u2, x2 = mul_shoup(u0 - u2 + 8 * Q, iw1, iw1s, Q); // u0, u2 < 8Q
      const u32 x1 = u1 + u3, x3 = mul_shoup(u1 - u3 + 2 * Q, iw1, iw1s, Q); // u1, u3 < 2Q
      // GINX: acc += (X^a - 1) acc (x) key+ + (X^-a - 1) acc (x) key-;  AP: acc = acc (x) key[digit]
      acc[jj][0] = csub((AP ? 0u : acc[jj][0]) + csub(lazy_reduce(x0, Q), Q), Q);
      acc[jj][1] = csub((AP ? 0u : acc[jj][1]) + csub(lazy_reduce(x1, Q), Q), Q);
      acc[jj][2] = csub((AP ? 0u : acc[jj][2]) + csub(x2, Q), Q);
      acc[jj][3] = csub((AP ? 0u : acc[jj][3]) + csub(x3, Q), Q);
#pragma unroll
      for (int i1 = 0; i1 < 4; i1++) {
        const u32 a = acc[jj][i1];
        accs[c * N + gt + 128 * jj + NB * i1] = ((a < (Q >> 1)) ? a : a - Q) + DIGIT_OFF;
      }
    }
    CLX_T(8);
  }

  // ---- epilogue: sample extraction (a14) and ModSwitch Q -> qKS (a15); CTA k writes the coefficients of block k ----
  {
    u32 *e = ext + gi * (N + 4);
    const u64 qKS = P.qKS;
    auto modswitch = [&](u32 v) -> u32 { return (qKS == Q) ? v : (u32)(((2 * (u64)v * qKS + Q) / (2 * (u64)Q)) % qKS); };
#pragma unroll
    for (int jj = 0; jj < 2; jj++)
#pragma unroll
      for (int i1 = 0; i1 < 4; i1++) {
        if ((u32)i1 != k) continue;
        const u32 j = gt + 128 * jj + NB * i1;
        if (acc_dbg) acc_dbg[(gi * 2 + c) * N + j] = acc[jj][i1];
        if (c == 0) {
          const u32 a = acc[jj][i1];
          const u32 v = (j == 0) ? a : (a == 0 ? 0 : Q - a); // Transpose: a'_0 = a_0, a'_k = -a_{N-k}
          e[(j == 0) ? 0 : N - j] = modswitch(v);
        } else if (j == 0) {
          e[N] = modswitch(csub(acc[jj][i1] + P.Q8, Q));
        }
      }
  }
#ifdef BFHE_PHASE_TIMING
  __syncwarp();
  bar_sync(BAR_DCT, 256); // the accumulator dump above is complete before the counters overwrite part of it
  if (acc_dbg && lane == 0 && (warp == 0 || warp == 4))
    for (int i = 0; i < 10; i++) {
      acc_dbg[(gi * 2 + 1) * N + NB * k + 32 + 16 * c + i] = (u32)(tph[i] / 1000); // kilo-cycles
      acc_dbg[(gi * 2 + 0) * N + NB * k + 32 + 16 * c + i] = tstamp[i];
    }
#endif
  cluster_sync_all(); // a CTA must not exit while its peers may still push into its shared memory
}

// key copy of this kernel: [step][rank][quad g][slot parity e][gt][4] <- evaluation-form key of kernels.cu ([chunk][lane][4] word order, slot
// P = 32 lane + 4 chunk + r holds the evaluation at psi^(2 bitrev(P) + 1)).  Quad g = (cc * 2 + sign) * 2 + half holds rows 4 half .. 4 half + 3
// of output component cc and key sign at slot t = 2 gt + e: one conflict-free LDS.128 per quad and slot in the product.
__global__ void bk_slice_clx_kernel(const u32 *__restrict__ src, u32 *__restrict__ dst, size_t nsteps) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nsteps * KEYPOLYS * N; i += (size_t)gridDim.x * blockDim.x) {
    const size_t step = i / ((size_t)KEYPOLYS * N), rem = i % ((size_t)KEYPOLYS * N);
    const int rk = (int)(rem / ((size_t)KEYPOLYS * NB)), g = (int)((rem / (NB * 4)) % 8), e = (int)((rem / (128 * 4)) % 2), gt = (int)((rem / 4) % 128),
              w4 = (int)(rem % 4);
    const int cc = g >> 2, sg = (g >> 1) & 1, hf = g & 1, rw = 4 * hf + w4, t = 2 * gt + e;
    const int pl = (sg * ROWS + rw) * 2 + cc; // polynomial index of kernels.cu's key: [sign][row][column]
    const int Ppos = slot_position(rk, t), sl = Ppos >> 5, j = Ppos & 31;
    dst[i] = src[(step * KEYPOLYS + pl) * N + ((j >> 2) * 32 + sl) * 4 + (j & 3)];
  }
}

// AP: one RGSW ciphertext (KEYPOLYS / 2 polynomials, [row][column]) per key; [key][rank][quad g = cc * 2 + half][slot parity e][gt][4]
__global__ void bk_slice_clx_ap_kernel(const u32 *__restrict__ src, u32 *__restrict__ dst, size_t nkeys) {
  constexpr int KP = KEYPOLYS / 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nkeys * KP * N; i += (size_t)gridDim.x * blockDim.x) {
    const size_t key = i / ((size_t)KP * N), rem = i % ((size_t)KP * N);
    const int rk = (int)(rem / ((size_t)KP * NB)), g = (int)((rem / (NB * 4)) % 4), e = (int)((rem / (128 * 4)) % 2), gt = (int)((rem / 4) % 128),
              w4 = (int)(rem % 4);
    const int cc = g >> 1, hf = g & 1, rw = 4 * hf + w4, t = 2 * gt + e;
    const int pl = rw * 2 + cc;
    const int Ppos = slot_position(rk, t), sl = Ppos >> 5, j = Ppos & 31;
    dst[i] = src[(key * KP + pl) * N + ((j >> 2) * 32 + sl) * 4 + (j & 3)];
  }
}

} // namespace clx

bool clx_supported(const DevConst &P, int method_ap) {
  return P.N == 1024 && P.dG == 4 && P.logBG == 7 && P.Q == SOLINAS_Q && P.n * (method_ap ? P.dR : 1u) <= (u32)clx::NSTEP_PAD;
}
size_t clx_tw_words() { return (size_t)clx::R * clx::TWR; }
int clx_set_attrs() {
  int rc = (int)cudaFuncSetAttribute(clx::blind_rotate_clx_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)clx::Smem::bytes);
  rc |= (int)cudaFuncSetAttribute(clx::blind_rotate_clx_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)clx::Smem::bytes);
  return rc;
}
static int clx_attrs_once() {
  static bool done[64];
  return once_per_device(done, clx_set_attrs);
}
int clx_max_gates() { // 4-CTA clusters of this kernel the device keeps co-resident, one CTA per SM; queried once per device, a 0 included
  static bool have[64];
  static int gates[64];
  const int d = device_slot();
  once_per_device(have, [&] {
    gates[d] = clx_attrs_once() ? 0 : max_active_clusters(clx::blind_rotate_clx_kernel<false>, clx::R, clx::THREADS, clx::Smem::bytes);
    return cudaSuccess;
  });
  return gates[d];
}
// The occupancy query is exact for this kernel (B200: 33 clusters; measured 1.02 ms per wave up to 33 gates, 2.03 ms -- a second round --
// from 34 on), so the whole co-resident maximum runs at full speed.
int clx_fast_gates() { return clx_max_gates(); }
int launch_bk_slice_clx(const u32 *d_src, u32 *d_dst, size_t npoly, int method_ap, void *stream) {
  if (npoly == 0) return 0;
  if (method_ap) clx::bk_slice_clx_ap_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_src, d_dst, npoly / (clx::KEYPOLYS / 2));
  else clx::bk_slice_clx_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(d_src, d_dst, npoly / clx::KEYPOLYS);
  return (int)cudaGetLastError();
}
int launch_blind_rotate_clx(const DevConst &P, int method_ap, const DevGate *d_gates, int count, const V2Bufs &vb, u32 *d_ext, u32 *d_acc_dbg,
                            void *stream, LaunchInfo *info) {
  if (count <= 0) return 0;
  if (int rc = clx_attrs_once()) return rc;
  if (info) { info->gates_per_cta = 1; info->ctas = clx::R * count; info->smem_bytes = clx::Smem::bytes; }
  if (method_ap)
    clx::blind_rotate_clx_kernel<true><<<clx::R * count, clx::THREADS, clx::Smem::bytes, (cudaStream_t)stream>>>(P, d_gates, count, vb.d_bkx, vb.d_twx,
                                                                                                           vb.d_F, d_ext, d_acc_dbg);
  else
    clx::blind_rotate_clx_kernel<false><<<clx::R * count, clx::THREADS, clx::Smem::bytes, (cudaStream_t)stream>>>(P, d_gates, count, vb.d_bkx, vb.d_twx,
                                                                                                            vb.d_F, d_ext, d_acc_dbg);
  return (int)cudaGetLastError();
}

} // namespace bfhe
