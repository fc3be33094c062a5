// Batched point (de)compression kernels — replaces G1Affine.Bytes()/SetBytes()
// (whisk/types.go:79-95, transcript/transcript.go:35, curdleproof.go:320-387).
#define CDL_FP_MUL_CALL 1  // one shared product body, as in k_elem.cu: inlined, decompression is ~84 k instructions
#include "codec.cuh"
#include "launch.h"

namespace cdl {

__global__ void k_compress(const G1Affine* __restrict__ in, uint8_t* __restrict__ out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1Affine p = in[i];
  g1_compress_dev(out + 48 * (size_t)i, p);
}

// Decompression: 64 threads per block, six blocks (12 warps) per SM.  ptxas then fits the kernel in 168 registers with
// 312 bytes of stack (540 B of spill stores); without the bound it needs 252
// registers and no stack, but only 8 warps fit per SM, and that measured slower on a B200 at 1 000 W
// from 2^17 points on (4 % at 2^19 .. 2^22; 2 % faster at 2^16; profiles/r11_decompress_chain.txt).
__global__ void __launch_bounds__(64, 6) k_decompress(const uint8_t* __restrict__ in,
                                                     G1Affine* __restrict__ out, uint8_t* __restrict__ status, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1Affine p;
  aff_set_inf(p);
  uint32_t st = g1_decompress_dev(p, in + 48 * (size_t)i);
  if (st) aff_set_inf(p);
  out[i] = p;
  status[i] = (uint8_t)st;
}


__global__ void k_compress_idx(const G1Affine* __restrict__ pool, const uint32_t* __restrict__ src,
                               uint8_t* __restrict__ out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1Affine p = pool[src[i]];
  g1_compress_dev(out + 48 * (size_t)i, p);
}

__global__ void __launch_bounds__(64, 6) k_decompress_idx(const uint8_t* __restrict__ in, G1Affine* __restrict__ pool,
                                 const uint32_t* __restrict__ dst, uint8_t* __restrict__ status, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  G1Affine p;
  aff_set_inf(p);
  uint32_t st = g1_decompress_dev(p, in + 48 * (size_t)i);
  if (st) aff_set_inf(p);
  pool[dst[i]] = p;
  status[i] = (uint8_t)st;
}

void launch_compress_idx(const G1Affine* pool, const uint32_t* src, uint8_t* out48, int n, cudaStream_t s) {
  k_compress_idx<<<(n + 127) / 128, 128, 0, s>>>(pool, src, out48, n);
}
void launch_decompress_idx(const uint8_t* in48, G1Affine* pool, const uint32_t* dst, uint8_t* status, int n,
                           cudaStream_t s) {
  k_decompress_idx<<<(n + 63) / 64, 64, 0, s>>>(in48, pool, dst, status, n);
}

void launch_compress(const G1Affine* in, uint8_t* out, int n, cudaStream_t s) {
  k_compress<<<(n + 127) / 128, 128, 0, s>>>(in, out, n);
}
void launch_decompress(const uint8_t* in, G1Affine* out, uint8_t* status, int n, cudaStream_t s) {
  k_decompress<<<(n + 63) / 64, 64, 0, s>>>(in, out, status, n);
}

}  // namespace cdl
