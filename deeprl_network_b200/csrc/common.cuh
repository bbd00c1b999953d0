// common.cuh -- shared device helpers for libnmarl (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/nmarl.h"

#define NH NMARL_NH          // 64
#define NG (4 * NMARL_NH)    // 256 gate columns, order i,f,o,u (agents/utils.py:106,202)

void nmarl_set_error(const char* fmt, ...);

#define NMARL_CHECK(cond, ...)                         \
  do {                                                 \
    if (!(cond)) {                                     \
      nmarl_set_error(__VA_ARGS__);                    \
      return 1;                                        \
    }                                                  \
  } while (0)

#define NMARL_CUDA(call)                                                         \
  do {                                                                           \
    cudaError_t e_ = (call);                                                     \
    if (e_ != cudaSuccess) {                                                     \
      nmarl_set_error("%s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(e_));  \
      return 2;                                                                  \
    }                                                                            \
  } while (0)

#define NMARL_LAUNCH_CHECK()                                                      \
  do {                                                                            \
    cudaError_t e_ = cudaPeekAtLastError();                                       \
    if (e_ != cudaSuccess) {                                                      \
      nmarl_set_error("%s:%d: launch: %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
      return 3;                                                                   \
    }                                                                             \
  } while (0)

// debug aid: NMARL_DEBUG_SYNC=1 synchronises and reports after each stage of the backward pass
#include <stdlib.h>
#define NMARL_DBG_SYNC(st, name)                                                            \
  do {                                                                                      \
    static int dbg_ = -1;                                                                   \
    if (dbg_ < 0) dbg_ = (getenv("NMARL_DEBUG_SYNC") != nullptr);                           \
    if (dbg_) {                                                                             \
      fprintf(stderr, "[nmarl] %s ...", name); fflush(stderr);                              \
      cudaError_t e2_ = cudaStreamSynchronize(st);                                          \
      fprintf(stderr, " %s\n", cudaGetErrorString(e2_)); fflush(stderr);                    \
    }                                                                                       \
  } while (0)

// LSTM-state layout (nmarl_fwd_args / nmarl_bwd_args.state_fm) the kernels implement: feature-major on the
// tensor-core path, except DIAL, whose message kernels are env-major; env-major on the FFMA path
inline int nmarl_state_fm(const nmarl_model* m, bool tc) { return (tc && m->variant != NMARL_DIAL) ? 1 : 0; }

// ---- kernel launch with optional programmatic dependent launch (see tc.cuh: pdl_wait) ---------------------------
template <typename... KArgs, typename... Args>
inline cudaError_t nmarl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- cp.async (LDGSTS) staging ------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, int src_bytes) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float f4get(const float4& v, int k) {
  return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w));
}

// ---- FP32 FFMA tile GEMM: acc[TM][4*NGRP] += A_tile[BM x K] * W[K x 64*NGRP] ----------------
// Thread layout: 16 (tx) x TY (ty) threads; thread rows = ty + TY*q (q<TM), thread columns =
// g*64 + 4*tx + j (g<NGRP, j<4) -- for the LSTM gate GEMM (NGRP=4) a thread therefore owns all
// four gates i,f,o,u of 4 hidden units and the cell update is a pure register epilogue.
// A: shared memory, row-major [BM][lda] (lda % 4 == 0, columns [K, roundup4(K)) zeroed).
// W: global memory, k-major [K][ldw] (ldw % 4 == 0, 16B-aligned), streamed through a 2-stage
//    cp.async ring Ws[2][KC][64*NGRP]; rows >= K are zero-filled.
// Accumulation is k-ascending FFMA (fixed order -> run-to-run deterministic).
// Every thread of the CTA must call this (it contains __syncthreads()).
template <int TM, int NGRP, int TY, int KC>
__device__ __forceinline__ void gemm_rowA(float (&acc)[TM][4 * NGRP], const float* As, int lda, int K,
                                          const float* __restrict__ W, int ldw, float* Ws, int tid) {
  constexpr int NT = 16 * TY;
  constexpr int WROW = 64 * NGRP;
  constexpr int F4ROW = 16 * NGRP;
  const int tx = tid & 15, ty = tid >> 4;
  const int Kpad = (K + 3) & ~3;
  const int nch = (Kpad + KC - 1) / KC;
  auto load = [&](int ch, int st) {
    float* dst = Ws + st * KC * WROW;
    for (int idx = tid; idx < KC * F4ROW; idx += NT) {
      const int kk = idx / F4ROW, c4 = idx - kk * F4ROW;
      const int k = ch * KC + kk;
      const bool ok = k < K;
      cp_async16(dst + kk * WROW + 4 * c4, ok ? (W + (size_t)k * ldw + 4 * c4) : W, ok ? 16 : 0);
    }
    cp_async_commit();
  };
  if (nch > 0) load(0, 0);
  for (int ch = 0; ch < nch; ++ch) {
    if (ch + 1 < nch) {
      load(ch + 1, (ch + 1) & 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* Wst = Ws + (ch & 1) * KC * WROW;
    const int k0 = ch * KC;
    const int kend = min(KC, Kpad - k0);
    for (int k4 = 0; k4 < kend; k4 += 4) {
      float4 a[TM];
#pragma unroll
      for (int q = 0; q < TM; ++q) a[q] = *reinterpret_cast<const float4*>(As + (ty + TY * q) * lda + k0 + k4);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        float4 b[NGRP];
#pragma unroll
        for (int g = 0; g < NGRP; ++g)
          b[g] = *reinterpret_cast<const float4*>(Wst + (k4 + kk) * WROW + g * 64 + 4 * tx);
#pragma unroll
        for (int q = 0; q < TM; ++q) {
          const float av = f4get(a[q], kk);
#pragma unroll
          for (int g = 0; g < NGRP; ++g) {
            acc[q][4 * g + 0] = fmaf(av, b[g].x, acc[q][4 * g + 0]);
            acc[q][4 * g + 1] = fmaf(av, b[g].y, acc[q][4 * g + 1]);
            acc[q][4 * g + 2] = fmaf(av, b[g].z, acc[q][4 * g + 2]);
            acc[q][4 * g + 3] = fmaf(av, b[g].w, acc[q][4 * g + 3]);
          }
        }
      }
    }
    __syncthreads();
  }
}

// Philox4x32-10 (counter-based RNG; one call gives 4x32 random bits)
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
// 53-bit uniform in [0,1) from two words, numpy's random_sample recipe
__device__ __forceinline__ double u01_from_bits(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
}
__device__ __forceinline__ double philox_u01(uint64_t seed, uint64_t ctr, uint32_t lane_lo, uint32_t lane_hi) {
  uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), lane_lo, lane_hi};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return u01_from_bits(c[0], c[1]);
}
