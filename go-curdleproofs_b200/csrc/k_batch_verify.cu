// Combined verifier check (engine_verify.cu): the tasks of the verifier's second MSM stage must each sum to
// the point at infinity.  All bases lie in the prime-order group G1, so with independent 128-bit weights
// rho_t the single sum  sum_t rho_t * MSM_t  is infinity only if every MSM_t is, except with probability
// <= 2^-128.  These kernels turn the stage into the term list of that one large MSM:
//   k_bv_weigh   thread per stage term: scalar * rho of its task, base index without the stage's flags
//   k_bv_crs     thread per CRS base: the weighted scalars of all its terms summed into one term at the end
//                of the list (and zeroed in place), so each shared base is gathered and bucketed once
//   k_bv_is_inf  the large MSM's Jacobian result: Z == 0
#include <cuda_runtime.h>
#include "fields.cuh"
#include "launch.h"

namespace cdl {

__global__ void __launch_bounds__(256)
k_bv_weigh(const uint32_t* __restrict__ idx, const Fr* __restrict__ sc, const MsmTask* __restrict__ tasks, uint32_t ntask,
           const Fr* __restrict__ rho, uint32_t nterm, uint32_t* __restrict__ cidx, Fr* __restrict__ csc) {
  const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nterm) return;
  // the task holding term j: the last one whose first term is <= j (tasks are contiguous and in order)
  uint32_t lo = 0, hi = ntask;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (tasks[mid].term_off <= j) lo = mid;
    else hi = mid;
  }
  Fr s = sc[j];
  FrM::mul(s, s, rho[lo]);
  csc[j] = s;
  cidx[j] = idx[j] & (kMsmIdxFixed - 1u);
}

__global__ void __launch_bounds__(128)
k_bv_crs(const uint32_t* __restrict__ off, const uint32_t* __restrict__ pos, uint32_t ncrs, uint32_t nterm,
         uint32_t* __restrict__ cidx, Fr* __restrict__ csc) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= ncrs) return;
  Fr acc, zero;
  FrM::set_zero(acc);
  FrM::set_zero(zero);
#pragma unroll 1
  for (uint32_t k = off[b]; k < off[b + 1]; k++) {
    const uint32_t p = pos[k];
    FrM::add(acc, acc, csc[p]);
    csc[p] = zero;
  }
  cidx[nterm + b] = b;
  csc[nterm + b] = acc;
}

__global__ void k_bv_is_inf(const G1Jac* __restrict__ r, uint32_t* __restrict__ flag) {
  if (threadIdx.x == 0 && blockIdx.x == 0) flag[0] = jac_is_inf(r[0]) ? 1u : 0u;
}

void launch_bv_assemble(const uint32_t* idx, const Fr* sc, const MsmTask* tasks, uint32_t ntask, const Fr* rho,
                        uint32_t nterm, const uint32_t* crs_off, const uint32_t* crs_pos, uint32_t ncrs, uint32_t* cidx,
                        Fr* csc, cudaStream_t st) {
  k_bv_weigh<<<(nterm + 255) / 256, 256, 0, st>>>(idx, sc, tasks, ntask, rho, nterm, cidx, csc);
  k_bv_crs<<<(ncrs + 127) / 128, 128, 0, st>>>(crs_off, crs_pos, ncrs, nterm, cidx, csc);
}

void launch_bv_is_inf(const G1Jac* r, uint32_t* flag, cudaStream_t st) { k_bv_is_inf<<<1, 32, 0, st>>>(r, flag); }

}  // namespace cdl
