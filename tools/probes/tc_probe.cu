// Stand-alone probe for the tcgen05 building blocks of the attention kernels (run on a B200):
//   S[128x128] = A[128x32] * B[128x32]^T   (SS MMA, K-major no-swizzle operands, 2 k-steps)  -> tcgen05.ld
//   P = bf16(S * 0.01) -> tcgen05.st (packed bf16x2) ; O[128x16] = P * V[128x16]  (TS MMA, A from TMEM)
// usage: tc_probe <variant>    bit0: swap LBO/SBO of the K-major operands
//                              bit1: swap LBO/SBO of the MN-major V operand
//                              bit2: stage V transposed and use a K-major descriptor instead of MN-major
// Prints max abs errors against a CPU reference.  Test infrastructure, not part of libpwa_b200.so.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "tc_common.cuh"

using namespace pwa::tc;

constexpr int M = 128, NK = 128, KD = 32, DV = 16;

__global__ void __launch_bounds__(128) probe_kernel(const __nv_bfloat16* A, const __nv_bfloat16* B, const __nv_bfloat16* V,
                                                    float* S_out, float* O_out, int variant) {
  __shared__ __align__(128) uint8_t sA[M * KD * 2];
  __shared__ __align__(128) uint8_t sB[NK * KD * 2];
  __shared__ __align__(128) uint8_t sV[NK * DV * 2];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5;

  // stage A, B: [k-chunk of 8][row][16 bytes]
  for (int i = tid; i < M * (KD / 8); i += 128) {
    int r = i % M, kc = i / M;
    *reinterpret_cast<uint4*>(sA + kc * (M * 16) + r * 16) = *reinterpret_cast<const uint4*>(A + r * KD + kc * 8);
    *reinterpret_cast<uint4*>(sB + kc * (NK * 16) + r * 16) = *reinterpret_cast<const uint4*>(B + r * KD + kc * 8);
  }
  if (variant & 4) {
    // V^T as a K-major operand: rows = d (16), K = keys: [key-chunk of 8][d][16 bytes]
    for (int i = tid; i < NK * DV; i += 128) {
      int key = i / DV, d = i % DV;
      *reinterpret_cast<__nv_bfloat16*>(sV + (key / 8) * (DV * 16) + d * 16 + (key % 8) * 2) = V[key * DV + d];
    }
  } else {
    // V as an MN-major operand: [key group of 8][d chunk of 8][key%8][16 bytes]
    for (int i = tid; i < NK * (DV / 8); i += 128) {
      int key = i / (DV / 8), dc = i % (DV / 8);
      *reinterpret_cast<uint4*>(sV + (key / 8) * ((DV / 8) * 128) + dc * 128 + (key % 8) * 16) =
          *reinterpret_cast<const uint4*>(V + key * DV + dc * 8);
    }
  }
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t lane_base = (uint32_t)(warp * 32) << 16;

  // ---- S = A * B^T
  if (tid == 0) {
    const uint32_t idesc = make_idesc_bf16(128, NK, 0, 0);
    for (int ks = 0; ks < KD / 16; ++ks) {
      uint32_t lboA = M * 16, lboB = NK * 16, sbo = 128;
      uint64_t da = (variant & 1) ? make_smem_desc(smem_u32(sA) + ks * 2 * M * 16, sbo, lboA)
                                  : make_smem_desc(smem_u32(sA) + ks * 2 * M * 16, lboA, sbo);
      uint64_t db = (variant & 1) ? make_smem_desc(smem_u32(sB) + ks * 2 * NK * 16, sbo, lboB)
                                  : make_smem_desc(smem_u32(sB) + ks * 2 * NK * 16, lboB, sbo);
      mma_ss(tmem, da, db, idesc, ks > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  tc_fence_after();
  const int row = tid;
  uint32_t r[32];
  for (int c = 0; c < NK / 32; ++c) {
    tmem_ld32(tmem + lane_base + c * 32, r);
    tmem_wait_ld();
    for (int j = 0; j < 32; ++j) S_out[row * NK + c * 32 + j] = __uint_as_float(r[j]);
  }
  // ---- P = bf16(0.01 * S) packed into columns [0, 64)
  for (int c = 0; c < NK / 32; ++c) {
    tmem_ld32(tmem + lane_base + c * 32, r);
    tmem_wait_ld();
    uint32_t pk[16];
    for (int j = 0; j < 16; ++j) pk[j] = pack_bf16(0.01f * __uint_as_float(r[2 * j]), 0.01f * __uint_as_float(r[2 * j + 1]));
    tmem_st16(tmem + lane_base + c * 16, pk);
  }
  tmem_wait_st();
  tc_fence_before();
  __syncthreads();
  // ---- O = P * V   (A from TMEM), D at column 128
  if (tid == 0) {
    tc_fence_after();
    for (int t = 0; t < NK / 16; ++t) {
      uint64_t dv;
      uint32_t idesc;
      if (variant & 4) {
        idesc = make_idesc_bf16(128, DV, 0, 0);
        dv = make_smem_desc(smem_u32(sV) + t * 2 * (DV * 16), DV * 16, 128);
      } else {
        idesc = make_idesc_bf16(128, DV, 0, 1);
        uint32_t lbo = (DV / 8) * 128, sbo = 128;
        uint32_t addr = smem_u32(sV) + t * 2 * (DV / 8) * 128;
        dv = (variant & 2) ? make_smem_desc(addr, sbo, lbo) : make_smem_desc(addr, lbo, sbo);
      }
      mma_ts(tmem + 128, tmem + t * 8, dv, idesc, t > 0);
    }
    mma_commit(&bar);
  }
  mbar_wait(&bar, 1);
  tc_fence_after();
  uint32_t o[16];
  tmem_ld16(tmem + lane_base + 128, o);
  tmem_wait_ld();
  for (int j = 0; j < DV; ++j) O_out[row * DV + j] = __uint_as_float(o[j]);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}

static float bf(float x) { return __bfloat162float(__float2bfloat16(x)); }

int main(int argc, char** argv) {
  int variant = argc > 1 ? atoi(argv[1]) : 0;
  std::vector<__nv_bfloat16> hA(M * KD), hB(NK * KD), hV(NK * DV);
  std::vector<float> fA(M * KD), fB(NK * KD), fV(NK * DV);
  srand(1);
  auto rnd = []() { return (float)(rand() % 2001 - 1000) / 1000.f; };
  for (int i = 0; i < M * KD; ++i) { fA[i] = bf(rnd()); hA[i] = __float2bfloat16(fA[i]); }
  for (int i = 0; i < NK * KD; ++i) { fB[i] = bf(rnd()); hB[i] = __float2bfloat16(fB[i]); }
  for (int i = 0; i < NK * DV; ++i) { fV[i] = bf(rnd()); hV[i] = __float2bfloat16(fV[i]); }
  __nv_bfloat16 *dA, *dB, *dV;
  float *dS, *dO;
  cudaMalloc(&dA, hA.size() * 2); cudaMalloc(&dB, hB.size() * 2); cudaMalloc(&dV, hV.size() * 2);
  cudaMalloc(&dS, M * NK * 4); cudaMalloc(&dO, M * DV * 4);
  cudaMemcpy(dA, hA.data(), hA.size() * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, hB.data(), hB.size() * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(dV, hV.data(), hV.size() * 2, cudaMemcpyHostToDevice);
  cudaMemset(dS, 0xff, M * NK * 4); cudaMemset(dO, 0xff, M * DV * 4);
  probe_kernel<<<1, 128>>>(dA, dB, dV, dS, dO, variant);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("variant %d: CUDA error %s\n", variant, cudaGetErrorString(e)); return 1; }
  std::vector<float> S(M * NK), O(M * DV);
  cudaMemcpy(S.data(), dS, S.size() * 4, cudaMemcpyDeviceToHost);
  cudaMemcpy(O.data(), dO, O.size() * 4, cudaMemcpyDeviceToHost);
  double es = 0, eo = 0, ms = 0, mo = 0;
  std::vector<float> Sref(M * NK);
  for (int i = 0; i < M; ++i)
    for (int j = 0; j < NK; ++j) {
      float s = 0;
      for (int k = 0; k < KD; ++k) s += fA[i * KD + k] * fB[j * KD + k];
      Sref[i * NK + j] = s;
      es = fmax(es, fabs(s - S[i * NK + j])); ms = fmax(ms, fabs(s));
    }
  for (int i = 0; i < M; ++i)
    for (int d = 0; d < DV; ++d) {
      float o = 0;
      for (int j = 0; j < NK; ++j) o += bf(0.01f * Sref[i * NK + j]) * fV[j * DV + d];
      eo = fmax(eo, fabs(o - O[i * DV + d])); mo = fmax(mo, fabs(o));
    }
  printf("variant %d: S max err %.4g (max |S| %.3g)   O max err %.4g (max |O| %.3g)   %s\n", variant, es, ms, eo, mo,
         (es < 1e-3 * ms && eo < 2e-2 * mo) ? "PASS" : "FAIL");
  return 0;
}
