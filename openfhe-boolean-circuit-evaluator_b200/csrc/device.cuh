// device.cuh -- primitives shared by the kernel translation units (kernels.cu, kernels_v2.cu, kernels_cl.cu): modular arithmetic for the
// ring modulus, mbarrier / TMA bulk copy / cluster (DSMEM) helpers, named barriers, and the host-side per-device attribute and
// cluster-limit helpers of their launch functions.
#pragma once
#include "common.hpp"
#include <cuda_runtime.h>

namespace bfhe {

// Both parameter sets of the reference share Q = PreviousPrime(FirstPrime(27, 2N), 2N) = 2^27 - 2^11 + 1.  The kernels are specialised
// for it (lazy_reduce's quotient is a shift, mul_shoup<true> writes t*Q as shifts and adds); bfhe_create refuses any other modulus.
constexpr u32 SOLINAS_Q = (1u << 27) - (1u << 11) + 1;

// table of (psi^k - 1), k < 2N (cluster kernels): the lanes of a warp own slots whose exponents differ in bits 4..8, so entry k is stored at
// the 11-bit rotation of k by 5 (bank = bits 5..9 of k): 1.5 wavefronts per gather on average instead of 16
__host__ __device__ __forceinline__ u32 f_index(u32 k) { return ((k >> 5) & 63u) | ((k & 31u) << 6); }

// ------------------------------------------------------------------------------------------
// modular arithmetic
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 redc(u64 s, u32 Q, u32 qinv_neg) { // s * 2^-32 mod Q, lazy
  u32 m = (u32)s * qinv_neg;
  return (u32)((s + (u64)m * Q) >> 32);
}
__device__ __forceinline__ u32 lazy_reduce(u32 x, u32 Q) { // any x -> [0,2Q)
  const u32 t = x >> 27; // floor(2^32 / Q) = 32, so the Barrett quotient estimate is a shift
  return x - t * Q;
}
__device__ __forceinline__ u32 csub(u32 x, u32 Q) { return min(x, x - Q); } // [0,2Q) -> [0,Q)
// Shoup multiply x * w mod Q, lazy in [0,2Q).  SOL = true computes the t*Q term as three ALU-pipe instructions (t*Q = t - ((t - (t << 16))
// << 11) for Q = SOLINAS_Q) instead of one IMAD on the FMA-heavy pipe; both pipes issue 16 lanes/cycle per SM sub-partition.
template <bool SOL = false> __device__ __forceinline__ u32 mul_shoup(u32 x, u32 w, u32 ws, u32 Q) {
  const u32 t = __umulhi(x, ws);
  if constexpr (SOL) {
    const u32 s = t + (0u - (t << 16));
    return (x * w - t) + (s << 11);
  } else {
    return x * w - t * Q;
  }
}

// ------------------------------------------------------------------------------------------
// key-mask expansion (include/bfhe.h "compact key blob"): ChaCha20 block function (RFC 8439) with a 64-bit block counter and a 64-bit
// nonce, as the host's Rng (hostmath.hpp), and the reduction of four keystream words, read as one little-endian 128-bit integer, mod m
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void chacha20_block(const u32 (&key)[8], u64 nonce, u64 counter, u32 (&out)[16]) {
  u32 x[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
               (u32)counter, (u32)(counter >> 32), (u32)nonce, (u32)(nonce >> 32)};
  u32 s[16];
#pragma unroll
  for (int i = 0; i < 16; i++) s[i] = x[i];
#define BFHE_DQR(a, b, c, d)                                                                                           \
  x[a] += x[b]; x[d] = __funnelshift_l(x[d] ^ x[a], x[d] ^ x[a], 16); x[c] += x[d]; x[b] = __funnelshift_l(x[b] ^ x[c], x[b] ^ x[c], 12); \
  x[a] += x[b]; x[d] = __funnelshift_l(x[d] ^ x[a], x[d] ^ x[a], 8);  x[c] += x[d]; x[b] = __funnelshift_l(x[b] ^ x[c], x[b] ^ x[c], 7);
#pragma unroll
  for (int r = 0; r < 10; r++) {
    BFHE_DQR(0, 4, 8, 12) BFHE_DQR(1, 5, 9, 13) BFHE_DQR(2, 6, 10, 14) BFHE_DQR(3, 7, 11, 15)
    BFHE_DQR(0, 5, 10, 15) BFHE_DQR(1, 6, 11, 12) BFHE_DQR(2, 7, 8, 13) BFHE_DQR(3, 4, 9, 14)
  }
#undef BFHE_DQR
#pragma unroll
  for (int i = 0; i < 16; i++) out[i] = x[i] + s[i];
}
// (w0 + w1 2^32 + w2 2^64 + w3 2^96) mod m for any m < 2^32, by Horner steps of 32 bits
__device__ __forceinline__ u32 reduce128(u32 w0, u32 w1, u32 w2, u32 w3, u32 m) {
  u64 r = w3 % m;
  r = ((r << 32) | w2) % m;
  r = ((r << 32) | w1) % m;
  return (u32)(((r << 32) | w0) % m);
}

// ------------------------------------------------------------------------------------------
// mbarrier, TMA bulk copy, thread-block cluster
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count)); }
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(u64 *bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
  asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(
                   smem_u32(bar)),
               "r"(parity)
               : "memory");
}
__device__ __forceinline__ bool mbar_test(u64 *bar, u32 parity) { // one try, no loop
  u32 ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// global -> shared bulk copy (TMA) whose bytes are counted on `bar` (complete_tx)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, u32 bytes, u64 *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ u32 cluster_rank() { u32 r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ u32 dsmem_addr(const void *local, u32 rank) { // shared::cluster address of `local` in CTA `rank`
  u32 a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(local)), "r"(rank));
  return a;
}
// remote stores whose arrival is counted on the destination CTA's mbarrier (complete_tx): the receiver needs no cluster-scope fence, it
// just waits for the phase of its own barrier
__device__ __forceinline__ void st_async2(u32 dsmem, uint2 v, u32 dsmem_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];" ::"r"(dsmem), "r"(v.x), "r"(v.y), "r"(dsmem_bar)
               : "memory");
}
__device__ __forceinline__ void st_async4(u32 dsmem, uint4 v, u32 dsmem_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(dsmem), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w), "r"(dsmem_bar)
               : "memory");
}
// named barriers (id 0 is __syncthreads)
__device__ __forceinline__ void bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ------------------------------------------------------------------------------------------
// host side: function attributes and cluster limits are per DEVICE (one process may hold contexts on several GPUs), and attributes must
// not be set under stream capture, so the launch helpers establish them once per device, at first use
// ------------------------------------------------------------------------------------------
inline int device_slot() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < 64 ? dev : 0;
}
// runs set() (returns a cudaError_t) unless it has succeeded on this device before; done[] is marked only on success, so a failure is
// returned to the caller and retried at the next call
template <typename F> int once_per_device(bool (&done)[64], F set) {
  const int d = device_slot();
  if (done[d]) return 0;
  const int rc = (int)set();
  if (rc == 0) done[d] = true;
  return rc;
}
// clusters of `cluster` CTAs of `kern` (its shared-memory attribute already set) that this device keeps co-resident, capped at one CTA per
// SM: two co-resident CTAs of the cluster kernels would just share the pipe.  0 when the query fails.
template <typename K> int max_active_clusters(K kern, int cluster, int threads, size_t smem) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cluster * 148, 1, 1);
  cfg.blockDim = dim3(threads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); n = 0; }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return n < sms / cluster ? n : sms / cluster;
}

} // namespace bfhe
