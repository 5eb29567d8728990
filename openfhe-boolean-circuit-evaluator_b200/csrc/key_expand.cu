// key_expand.cu -- expansion of a compact key blob ("BFHEKEY2", include/bfhe.h) on the device: the public masks of the key-switching and
// bootstrapping keys are regenerated from the mask seed straight into the buffers the key upload already uses.
//
// Rule (one rule, a second implementation on the host in engine.cu): mask row r is the ChaCha20 stream with key = mask seed, nonce = r,
// block counter from 0; coefficient t of the row is stream words 4t..4t+3 as a little-endian 128-bit integer, reduced mod the row's modulus.
// So block b of a row gives coefficients 4b..4b+3, and every thread below computes one block.
#include "device.cuh"
#include <algorithm>

namespace bfhe {

// KSK: device layout [i][k][j][rowlen] (engine.cu ensure_device_keys), row (i, j, k) = mask row (i * baseKS + j) * dKS + k.  One thread per
// four columns of a padded row: mask words below n, the body at n, zeros up to rowlen.
template <typename T>
__global__ void __launch_bounds__(256) ksk_expand_kernel(const MaskKey key, const T *__restrict__ bodies, T *__restrict__ dksk, u32 baseKS,
                                                         u32 dKS, u32 n, u32 rowlen, u32 m, size_t total) {
  const u32 quads = rowlen / 4;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t drow = t / quads;
    const u32 c4 = (u32)(t % quads);
    const size_t i = drow / ((size_t)dKS * baseKS);
    const u32 rem = (u32)(drow % ((size_t)dKS * baseKS)), k = rem / baseKS, j = rem % baseKS;
    const size_t r = (i * baseKS + j) * dKS + k;
    T o[4];
    u32 w[16];
    if (4 * c4 < n) chacha20_block(key.k, r, c4, w);
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const u32 col = 4 * c4 + e;
      o[e] = col < n ? (T)reduce128(w[4 * e], w[4 * e + 1], w[4 * e + 2], w[4 * e + 3], m) : col == n ? bodies[r] : (T)0;
    }
    T *dst = dksk + drow * rowlen + 4 * (size_t)c4;
    if constexpr (sizeof(T) == 2) *reinterpret_cast<uint2 *>(dst) = make_uint2(o[0] | (u32)o[1] << 16, o[2] | (u32)o[3] << 16);
    else *reinterpret_cast<uint4 *>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

int launch_ksk_expand(const MaskKey &key, const void *d_bodies, void *d_ksk, int elem_bytes, u32 N, u32 baseKS, u32 dKS, u32 n, u32 rowlen,
                      u32 qKS, void *stream) {
  if (rowlen % 4 || rowlen < n + 1) return (int)cudaErrorInvalidValue;
  const size_t total = (size_t)N * baseKS * dKS * (rowlen / 4);
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 64);
  if (elem_bytes == 2)
    ksk_expand_kernel<u16><<<blocks, 256, 0, (cudaStream_t)stream>>>(key, (const u16 *)d_bodies, (u16 *)d_ksk, baseKS, dKS, n, rowlen, qKS, total);
  else
    ksk_expand_kernel<u32><<<blocks, 256, 0, (cudaStream_t)stream>>>(key, (const u32 *)d_bodies, (u32 *)d_ksk, baseKS, dKS, n, rowlen, qKS, total);
  return (int)cudaGetLastError();
}

// Fresh ciphertexts of a BFHECTS1 blob: with baseKS = dKS = 1 the KSK layout is `count` plain rows and row i is mask row i, so the same
// kernel writes them (mask words mod q below n, the body at n, zero padding up to the stride).
int launch_ct_expand(const MaskKey &key, const u32 *d_bodies, u32 *d_rows, size_t count, u32 n, u32 stride, u32 q, void *stream) {
  if (count == 0) return 0;
  if (count > 0xffffffffu) return (int)cudaErrorInvalidValue;
  return launch_ksk_expand(key, d_bodies, d_rows, 4, (u32)count, 1, 1, n, stride, q, stream);
}

// BK: `pairs` (mask, body) polynomial pairs of the coefficient-form key in BFHEKEY1 order, the first with mask number p_first (stream id
// 2^40 + p_first).  Polynomial 2s of the staging buffer gets mask p_first + s, polynomial 2s + 1 gets body s of d_bodies.
__global__ void __launch_bounds__(256) bk_mask_expand_kernel(const MaskKey key, const u32 *__restrict__ bodies, u32 *__restrict__ stage,
                                                             u64 p_first, u32 N, u32 Q, size_t total) {
  const u32 quads = N / 4;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t s = t / quads;
    const u32 b = (u32)(t % quads);
    u32 w[16];
    chacha20_block(key.k, BK_MASK_STREAM + p_first + s, b, w);
    uint4 mk;
    mk.x = reduce128(w[0], w[1], w[2], w[3], Q);
    mk.y = reduce128(w[4], w[5], w[6], w[7], Q);
    mk.z = reduce128(w[8], w[9], w[10], w[11], Q);
    mk.w = reduce128(w[12], w[13], w[14], w[15], Q);
    *reinterpret_cast<uint4 *>(stage + 2 * s * N + 4 * b) = mk;
    *reinterpret_cast<uint4 *>(stage + (2 * s + 1) * N + 4 * b) = *reinterpret_cast<const uint4 *>(bodies + s * N + 4 * b);
  }
}

int launch_bk_mask_expand(const MaskKey &key, const u32 *d_bodies, u32 *d_stage, u64 p_first, size_t pairs, u32 N, u32 Q, void *stream) {
  if (pairs == 0) return 0;
  if (N % 4) return (int)cudaErrorInvalidValue;
  const size_t total = pairs * (N / 4);
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 64);
  bk_mask_expand_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(key, d_bodies, d_stage, p_first, N, Q, total);
  return (int)cudaGetLastError();
}

} // namespace bfhe
