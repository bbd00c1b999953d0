// train.cu -- K7 n-step returns, K8/K9 A2C loss + BPTT with message-gradient scatter + weight
// gradients, K10 global-norm clip + TF-semantics RMSProp.
//
// Backward structure (per update of T steps):
//   1. transposed copies of [wx;wh], w_msg, w_mfc (once per update; weights only change in K10)
//   2. T launches of the TRAIN-mode forward (cell_fwd.cu) saving activations + per-row
//      d(loss)/d(logits,v)                                              (policies.py:232-255)
//   3. T reverse launches of cell_bwd_kernel: gate derivatives -> dgrad GEMM dz [wx;wh]^T ->
//      encoder pre-activation grads -> message gradient dm = dpre_m W_msg^T written per
//      (receiver, slot) and GATHERED by the sender at step t-1 (deterministic; the transpose of
//      the forward neighbour gather, what tf.gradients does through tf.boolean_mask)
//   4. weight gradients as split-K "A^T D" GEMMs over all (t, env) rows + fixed-order reduce
#include "bwd_common.cuh"

int nmarl_check_model(const nmarl_model* m);
int nmarl_launch_train_fwd(const nmarl_model* m, const nmarl_fwd_args* a, const float* Rs, const float* Advs,
                           float* sv_xin, float* sv_sh, float* sv_gates, float* sv_enc, float* sv_dlv,
                           float* loss_part, float loss_scale, float v_coef, float e_coef, cudaStream_t st);
int nmarl_fwd_tiles(int B);

namespace {

// ============================ K7: returns ======================================================
struct RetK {
  int N, B, T, NR, zero_end;
  double gamma, rnorm, rclip, alpha;
  int n_pow;
};

__global__ void nstep_return_kernel(const RetK k, const double* __restrict__ reward, const float* __restrict__ value,
                                    const float* __restrict__ done_post, const float* __restrict__ R_end,
                                    const int32_t* __restrict__ dist, const double* __restrict__ alpha_pow,
                                    float* __restrict__ Rs, float* __restrict__ Advs) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= k.N * k.B) return;
  const int i = idx / k.B, b = idx - i * k.B;
  double R = (double)R_end[idx];
  if (k.zero_end && done_post[(size_t)(k.T - 1) * k.B + b] != 0.0f) R = 0.0;
  for (int t = k.T - 1; t >= 0; --t) {
    const double nd = 1.0 - (double)done_post[(size_t)t * k.B + b];
    const double* rt = reward + (size_t)t * k.NR * k.B;
    if (k.alpha < 0) {                          // _add_R_Adv (agents/utils.py:837-855)
      double r = rt[(size_t)(k.NR == 1 ? 0 : i) * k.B + b];
      if (k.rnorm > 0) r = r / k.rnorm;
      if (k.rclip > 0) r = fmin(fmax(r, -k.rclip), k.rclip);
      R = r + k.gamma * R * nd;
    } else {                                    // _add_s_R_Adv (agents/utils.py:888-912)
      R = k.gamma * R * nd;
      int maxd = 0;
      for (int j = 0; j < k.N; ++j) maxd = max(maxd, dist[i * k.N + j]);
      for (int d = 0; d <= maxd && d < k.n_pow; ++d) {
        double s = 0.0;                         // np.sum over the (short) masked vector: ascending j
        for (int j = 0; j < k.N; ++j) {
          if (dist[i * k.N + j] != d) continue;
          double r = rt[(size_t)j * k.B + b];
          if (k.rnorm > 0) r = r / k.rnorm;
          if (k.rclip > 0) r = fmin(fmax(r, -k.rclip), k.rclip);
          s += r;
        }
        R += alpha_pow[d] * s;
      }
    }
    const size_t o = ((size_t)t * k.N + i) * k.B + b;
    Rs[o] = (float)R;
    Advs[o] = (float)(R - (double)value[o]);
  }
}

// ============================ transposes =======================================================
__global__ void transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols) {
  // dst[c][r] = src[r][c]; small matrices, 32x32 smem tiles
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int r = r0 + y, c = c0 + threadIdx.x;
    tile[y][threadIdx.x] = (r < rows && c < cols) ? src[(size_t)r * cols + c] : 0.f;
  }
  __syncthreads();
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int c = c0 + y, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[(size_t)c * rows + r] = tile[threadIdx.x][y];
  }
}

// ============================ K9: one reverse step of the cell ==================================
template <int VAR, int BM, int TY>
__global__ void __launch_bounds__(16 * TY) cell_bwd_kernel(const __grid_constant__ nmarl_model m,
                                                          const __grid_constant__ BwdK k) {
  constexpr int NT = 16 * TY, TM = BM / TY, KC = 16;
  constexpr int NGRP = (VAR == NMARL_NC) ? 4 : 2;
  constexpr int LDZ = NG + 4, LDP = NH + 4;
  extern __shared__ __align__(16) float smem[];
  float* DZ = smem;                         // [BM][LDZ]
  float* Ws = smem + (size_t)BM * LDZ;      // 2*KC*64*NGRP
  float* DPm = smem;                        // aliases DZ after the dgrad GEMM
  const int i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  const int B = k.B, b0 = blockIdx.x * BM, rows = min(BM, B - b0);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n_a = m.n_a, SD = m.s_dim;
  const float* __restrict__ P = k.params;

  // ---- phase 0/1: total dh, gate derivatives ---------------------------------------------------
  float wpi[4][NMARL_MAX_NA];               // W_pi rows of this thread's 4 units, then W_v
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int c = 0; c < NMARL_MAX_NA; ++c) wpi[j][c] = 0.f;
    for (int c = 0; c < n_a; ++c) wpi[j][c] = __ldg(P + ag.o_pi_w + (4 * tx + j) * n_a + c);
    wpi[j][NMARL_MAX_NA - 1] = __ldg(P + ag.o_v_w + 4 * tx + j);
  }
#pragma unroll
  for (int q = 0; q < TM; ++q) {
    const int r = ty + TY * q;
    float dz[4][4];
#pragma unroll
    for (int g = 0; g < 4; ++g) dz[g][0] = dz[g][1] = dz[g][2] = dz[g][3] = 0.f;
    if (r < rows) {
      const int b = b0 + r;
      const size_t row = (size_t)i * B + b;
      const float4 d0 = *reinterpret_cast<const float4*>(k.sv_dlv + row * 8);
      const float4 d1 = *reinterpret_cast<const float4*>(k.sv_dlv + row * 8 + 4);
      const float dl[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      const float dv = dl[n_a];
      float dh[4], dc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float s = 0.f;
#pragma unroll
        for (int c = 0; c < NMARL_MAX_NA - 1; ++c) s = fmaf(c < n_a ? dl[c] : 0.f, wpi[j][c], s);
        dh[j] = fmaf(dv, wpi[j][NMARL_MAX_NA - 1], s);
      }
      if (k.has_next) {
        const float4 r4 = *reinterpret_cast<const float4*>(k.dh_in + row * NH + 4 * tx);
        dh[0] += r4.x; dh[1] += r4.y; dh[2] += r4.z; dh[3] += r4.w;
        if (VAR == NMARL_NC || VAR == NMARL_IC3) {
          for (int s = 0; s < ag.n_recv; ++s) {
            const float4 m4 = *reinterpret_cast<const float4*>(
                k.dmsg_in + (((size_t)ag.recv_agent[s] * NMARL_MAX_NBR + ag.recv_slot[s]) * B + b) * NH + 4 * tx);
            dh[0] += m4.x; dh[1] += m4.y; dh[2] += m4.z; dh[3] += m4.w;
          }
        }
        const float4 c4 = *reinterpret_cast<const float4*>(k.dc_in + row * NH + 4 * tx);
        dc[0] = c4.x; dc[1] = c4.y; dc[2] = c4.z; dc[3] = c4.w;
      }
      const float nd = 1.0f - k.done_pre[b];
      const float* gs = k.sv_gates + row * NG + 4 * tx;
      const float4 gi = *reinterpret_cast<const float4*>(gs), gf = *reinterpret_cast<const float4*>(gs + NH),
                   go = *reinterpret_cast<const float4*>(gs + 2 * NH), gu = *reinterpret_cast<const float4*>(gs + 3 * NH);
      const float4 cc = *reinterpret_cast<const float4*>(k.c_cur + row * NH + 4 * tx);
      const float4 cp = *reinterpret_cast<const float4*>(k.c_prev + row * NH + 4 * tx);
      float dcp[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float ig = f4get(gi, j), fg = f4get(gf, j), og = f4get(go, j), ug = f4get(gu, j);
        const float tc = tanhf(f4get(cc, j));
        const float cpm = f4get(cp, j) * nd;
        const float dct = dc[j] + dh[j] * og * (1.0f - tc * tc);
        dz[0][j] = dct * ug * ig * (1.0f - ig);
        dz[1][j] = dct * cpm * fg * (1.0f - fg);
        dz[2][j] = dh[j] * tc * og * (1.0f - og);
        dz[3][j] = dct * ig * (1.0f - ug * ug);
        dcp[j] = dct * fg * nd;
      }
      *reinterpret_cast<float4*>(k.dc_out + row * NH + 4 * tx) = make_float4(dcp[0], dcp[1], dcp[2], dcp[3]);
      float* zo = k.sv_dz + row * NG + 4 * tx;
#pragma unroll
      for (int g = 0; g < 4; ++g)
        *reinterpret_cast<float4*>(zo + g * NH) = make_float4(dz[g][0], dz[g][1], dz[g][2], dz[g][3]);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g)
      *reinterpret_cast<float4*>(DZ + r * LDZ + g * NH + 4 * tx) = make_float4(dz[g][0], dz[g][1], dz[g][2], dz[g][3]);
  }
  __syncthreads();

  // ---- phase 2: dgrad  d[s | h^] = dz [wx ; wh]^T ------------------------------------------------
  float acc[TM][4 * NGRP];
#pragma unroll
  for (int q = 0; q < TM; ++q)
#pragma unroll
    for (int c = 0; c < 4 * NGRP; ++c) acc[q][c] = 0.f;
  gemm_rowA<TM, NGRP, TY, KC>(acc, DZ, LDZ, NG, k.wt + ag.t_wxh, SD + NH, Ws, tid);
#pragma unroll
  for (int q = 0; q < TM; ++q) {
    const int r = ty + TY * q;
    float dpm[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < rows) {
      const int b = b0 + r;
      const size_t row = (size_t)i * B + b;
      const float nd = 1.0f - k.done_pre[b];
      constexpr int GH = 4 * (NGRP - 1);
      *reinterpret_cast<float4*>(k.dh_out + row * NH + 4 * tx) =
          make_float4(acc[q][GH] * nd, acc[q][GH + 1] * nd, acc[q][GH + 2] * nd, acc[q][GH + 3] * nd);
      float* dp = k.sv_dpre + row * 192 + 4 * tx;
      if (VAR == NMARL_NC) {
        const float* sp = k.sv_sh + row * (SD + NH) + 4 * tx;
#pragma unroll
        for (int g = 0; g < 3; ++g) {
          const float4 s4 = *reinterpret_cast<const float4*>(sp + g * NH);
          float o[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) o[j] = f4get(s4, j) > 0.f ? acc[q][4 * g + j] : 0.f;
          *reinterpret_cast<float4*>(dp + g * NH) = make_float4(o[0], o[1], o[2], o[3]);
          if (g == 2) { dpm[0] = o[0]; dpm[1] = o[1]; dpm[2] = o[2]; dpm[3] = o[3]; }
        }
      } else if (VAR == NMARL_IA2C) {
        const float4 s4 = *reinterpret_cast<const float4*>(k.sv_sh + row * (SD + NH) + 4 * tx);
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = f4get(s4, j) > 0.f ? acc[q][j] : 0.f;
        *reinterpret_cast<float4*>(dp) = make_float4(o[0], o[1], o[2], o[3]);
      } else if (VAR == NMARL_IC3) {
        const float4 hx = *reinterpret_cast<const float4*>(k.sv_enc + row * 128 + 4 * tx);
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float x = f4get(hx, j); o[j] = acc[q][j] * (1.0f - x * x); dpm[j] = acc[q][j]; }
        *reinterpret_cast<float4*>(dp) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(dp + NH) = make_float4(dpm[0], dpm[1], dpm[2], dpm[3]);
      } else {  // DIAL
        const float4 hx = *reinterpret_cast<const float4*>(k.sv_enc + row * 128 + 4 * tx);
        const float4 hm = *reinterpret_cast<const float4*>(k.sv_enc + row * 128 + NH + 4 * tx);
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[j] = f4get(hx, j) > 0.f ? acc[q][j] : 0.f;
          dpm[j] = f4get(hm, j) > 0.f ? acc[q][j] : 0.f;
        }
        *reinterpret_cast<float4*>(dp) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(dp + NH) = make_float4(dpm[0], dpm[1], dpm[2], dpm[3]);
      }
    }
    if (VAR != NMARL_IA2C) *reinterpret_cast<float4*>(DPm + r * LDP + 4 * tx) = make_float4(dpm[0], dpm[1], dpm[2], dpm[3]);
  }

  // ---- phase 3: message gradient  dm = dpre_m W_msg^T, one 64-wide block per neighbour slot ------
  if (VAR != NMARL_IA2C) {
    const int Km = (VAR == NMARL_IC3) ? NH : ag.n_nbr * NH;
    const int nblk = (VAR == NMARL_IC3) ? 1 : ag.n_nbr;
    for (int s = 0; s < nblk; ++s) {
      float a2[TM][4];
#pragma unroll
      for (int q = 0; q < TM; ++q) { a2[q][0] = a2[q][1] = a2[q][2] = a2[q][3] = 0.f; }
      gemm_rowA<TM, 1, TY, KC>(a2, DPm, LDP, NH, k.wt + ag.t_w_msg + s * NH, Km, Ws, tid);
#pragma unroll
      for (int q = 0; q < TM; ++q) {
        const int r = ty + TY * q;
        if (r >= rows) continue;
        const int b = b0 + r;
        if (VAR == NMARL_IC3) {                 // mean: every neighbour receives dm / n_m
          const float nn = (float)ag.n_nbr;
          const float4 o = make_float4(a2[q][0] / nn, a2[q][1] / nn, a2[q][2] / nn, a2[q][3] / nn);
          for (int s2 = 0; s2 < ag.n_nbr; ++s2)
            *reinterpret_cast<float4*>(k.dmsg_out + (((size_t)i * NMARL_MAX_NBR + s2) * B + b) * NH + 4 * tx) = o;
        } else {
          *reinterpret_cast<float4*>(k.dmsg_out + (((size_t)i * NMARL_MAX_NBR + s) * B + b) * NH + 4 * tx) =
              make_float4(a2[q][0], a2[q][1], a2[q][2], a2[q][3]);
        }
      }
    }
  }
}

// DIAL: sender-side message fc backward at step t (after cell_bwd(t)):
//   dmp = (sum over receivers of dmsg) * relu'(msg_t);  dh_rec += dmp W_mfc^T
template <int BM, int TY>
__global__ void __launch_bounds__(16 * TY) dial_msg_bwd_kernel(const __grid_constant__ nmarl_model m, int B,
                                                              const float* __restrict__ wt,
                                                              const float* __restrict__ msg_t,
                                                              const float* __restrict__ dmsg, float* __restrict__ sv_dmp,
                                                              float* __restrict__ dh_rec) {
  constexpr int NT = 16 * TY, TM = BM / TY, KC = 16, LDP = NH + 4;
  __shared__ __align__(16) float DM[BM * LDP];
  __shared__ __align__(16) float Ws[2 * KC * NH];
  const int i = blockIdx.y, b0 = blockIdx.x * BM, rows = min(BM, B - b0);
  const nmarl_agent& ag = m.agent[i];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int idx = tid; idx < BM * (NH / 4); idx += NT) {
    const int r = idx / (NH / 4), u4 = idx - r * (NH / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows) {
      const int b = b0 + r;
      for (int s = 0; s < ag.n_recv; ++s) {
        const float4 w = *reinterpret_cast<const float4*>(
            dmsg + (((size_t)ag.recv_agent[s] * NMARL_MAX_NBR + ag.recv_slot[s]) * B + b) * NH + 4 * u4);
        v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
      }
      const float4 mm = *reinterpret_cast<const float4*>(msg_t + ((size_t)i * B + b) * NH + 4 * u4);
      v.x = mm.x > 0.f ? v.x : 0.f; v.y = mm.y > 0.f ? v.y : 0.f; v.z = mm.z > 0.f ? v.z : 0.f; v.w = mm.w > 0.f ? v.w : 0.f;
      *reinterpret_cast<float4*>(sv_dmp + ((size_t)i * B + b) * NH + 4 * u4) = v;
    }
    *reinterpret_cast<float4*>(DM + r * LDP + 4 * u4) = v;
  }
  __syncthreads();
  float acc[TM][4];
#pragma unroll
  for (int q = 0; q < TM; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f; }
  gemm_rowA<TM, 1, TY, KC>(acc, DM, LDP, NH, wt + ag.t_mfc, NH, Ws, tid);
#pragma unroll
  for (int q = 0; q < TM; ++q) {
    const int r = ty + TY * q;
    if (r < rows) {
      float4* p = reinterpret_cast<float4*>(dh_rec + ((size_t)i * B + b0 + r) * NH + 4 * tx);
      float4 o = *p;
      o.x += acc[q][0]; o.y += acc[q][1]; o.z += acc[q][2]; o.w += acc[q][3];
      *p = o;
    }
  }
}

// ============================ weight gradients: C = A^T D over rows (t, env) =====================
struct WgK {
  int N, B, T, splits;
  const float* A; int lda; int a_col0;       // A[t][agent][env][lda], columns a_col0 + [0, Ka_i)
  const float* D; int ldd; int d_col0;       // D[t][agent][env][ldd], columns d_col0 + [0, 64*NGRP)
  int ka_max;                                // workspace row count per (split, agent) = ka_max + 1 (bias row)
  int Ka[NMARL_MAX_AGENT];
  float* ws;                                 // [splits][N][ka_max + 1][64*NGRP]
};

template <int NGRP>
__global__ void __launch_bounds__(256) wgrad_kernel(const __grid_constant__ WgK k) {
  constexpr int RC = 32, ND = 64 * NGRP;
  extern __shared__ __align__(16) float wg_smem[];
  float (*As)[RC][64] = reinterpret_cast<float (*)[RC][64]>(wg_smem);
  float (*Ds)[RC][ND] = reinterpret_cast<float (*)[RC][ND]>(wg_smem + 2 * RC * 64);
  const int sp = blockIdx.x, mt = blockIdx.y, i = blockIdx.z;
  const int Ka = k.Ka[i];
  if (mt * 64 >= Ka) return;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int R = k.T * k.B;
  const int per = ((R + k.splits - 1) / k.splits + RC - 1) / RC * RC;
  const int r_begin = sp * per, r_end = min(R, r_begin + per);
  float acc[4][4 * NGRP];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int c = 0; c < 4 * NGRP; ++c) acc[a][c] = 0.f;
  float bsum[4 * NGRP];
#pragma unroll
  for (int c = 0; c < 4 * NGRP; ++c) bsum[c] = 0.f;
  const int nch = r_end > r_begin ? (r_end - r_begin + RC - 1) / RC : 0;
  auto load = [&](int ch, int st) {
    const int rb = r_begin + ch * RC;
    for (int idx = tid; idx < RC * 16; idx += 256) {          // A chunk: RC x 64
      const int rr = idx >> 4, c4 = idx & 15;
      const int r = rb + rr;
      const int col = mt * 64 + 4 * c4;
      const bool ok = (r < r_end) && (col < Ka);
      const int t = ok ? r / k.B : 0, b = ok ? r - t * k.B : 0;
      const float* src = k.A + (((size_t)t * k.N + i) * k.B + b) * k.lda + k.a_col0 + col;
      cp_async16(&As[st][rr][4 * c4], ok ? src : k.A, ok ? 16 : 0);
    }
    for (int idx = tid; idx < RC * 16 * NGRP; idx += 256) {   // D chunk: RC x ND
      const int rr = idx / (16 * NGRP), c4 = idx - rr * (16 * NGRP);
      const int r = rb + rr;
      const bool ok = r < r_end;
      const int t = ok ? r / k.B : 0, b = ok ? r - t * k.B : 0;
      const float* src = k.D + (((size_t)t * k.N + i) * k.B + b) * k.ldd + k.d_col0 + 4 * c4;
      cp_async16(&Ds[st][rr][4 * c4], ok ? src : k.D, ok ? 16 : 0);
    }
    cp_async_commit();
  };
  if (nch > 0) load(0, 0);
  for (int ch = 0; ch < nch; ++ch) {
    if (ch + 1 < nch) { load(ch + 1, (ch + 1) & 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const int st = ch & 1;
#pragma unroll 8
    for (int rr = 0; rr < RC; ++rr) {
      const float4 a = *reinterpret_cast<const float4*>(&As[st][rr][4 * ty]);
      float4 d[NGRP];
#pragma unroll
      for (int g = 0; g < NGRP; ++g) d[g] = *reinterpret_cast<const float4*>(&Ds[st][rr][g * 64 + 4 * tx]);
#pragma unroll
      for (int g = 0; g < NGRP; ++g) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
          const float av = f4get(a, mi);
          acc[mi][4 * g + 0] = fmaf(av, d[g].x, acc[mi][4 * g + 0]);
          acc[mi][4 * g + 1] = fmaf(av, d[g].y, acc[mi][4 * g + 1]);
          acc[mi][4 * g + 2] = fmaf(av, d[g].z, acc[mi][4 * g + 2]);
          acc[mi][4 * g + 3] = fmaf(av, d[g].w, acc[mi][4 * g + 3]);
        }
      }
    }
    if (mt == 0) {                                            // bias = column sums of D (rows rr = ty, ty+16)
#pragma unroll
      for (int h2 = 0; h2 < RC / 16; ++h2) {
#pragma unroll
        for (int g = 0; g < NGRP; ++g) {
          const float4 d = *reinterpret_cast<const float4*>(&Ds[st][ty + 16 * h2][g * 64 + 4 * tx]);
          bsum[4 * g] += d.x; bsum[4 * g + 1] += d.y; bsum[4 * g + 2] += d.z; bsum[4 * g + 3] += d.w;
        }
      }
    }
    __syncthreads();
  }
  float* wsb = k.ws + ((size_t)sp * k.N + i) * (size_t)(k.ka_max + 1) * ND;
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int row = mt * 64 + 4 * ty + mi;
    if (row < Ka) {
#pragma unroll
      for (int g = 0; g < NGRP; ++g)
        *reinterpret_cast<float4*>(wsb + (size_t)row * ND + g * 64 + 4 * tx) =
            make_float4(acc[mi][4 * g], acc[mi][4 * g + 1], acc[mi][4 * g + 2], acc[mi][4 * g + 3]);
    }
  }
  if (mt == 0) {                                              // reduce bias partials over ty (fixed order)
    float* red = &Ds[0][0][0];                                // 2*RC*ND >= 16*ND floats
#pragma unroll
    for (int g = 0; g < NGRP; ++g)
      *reinterpret_cast<float4*>(red + ty * ND + g * 64 + 4 * tx) =
          make_float4(bsum[4 * g], bsum[4 * g + 1], bsum[4 * g + 2], bsum[4 * g + 3]);
    __syncthreads();
    for (int c = tid; c < ND; c += 256) {
      float s = 0.f;
      for (int y = 0; y < 16; ++y) s += red[y * ND + c];
      wsb[(size_t)k.ka_max * ND + c] = s;
    }
  }
}

struct WgRedK {
  int N, splits, ka_max, nd;
  int Ka[NMARL_MAX_AGENT];
  int o_w[NMARL_MAX_AGENT];
  int o_b[NMARL_MAX_AGENT];
  const float* ws;
  float* grads;
};

__global__ void wgrad_reduce_kernel(const __grid_constant__ WgRedK k) {
  const int i = blockIdx.y;
  const int Ka = k.Ka[i];
  const int total = (Ka + 1) * k.nd;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int row = e / k.nd, c = e - row * k.nd;
    const int wrow = (row == Ka) ? k.ka_max : row;
    float s = 0.f;
    for (int sp = 0; sp < k.splits; ++sp)
      s += k.ws[(((size_t)sp * k.N + i) * (size_t)(k.ka_max + 1) + wrow) * k.nd + c];
    if (row == Ka) { if (k.o_b[i] >= 0) k.grads[k.o_b[i] + c] = s; }
    else k.grads[k.o_w[i] + (size_t)row * k.nd + c] = s;
  }
}

// heads: dW_pi = h^T dlogits, db_pi, dW_v = [h, onehot(a_nbr)]^T dv, db_v   (skinny; own kernel)
struct HeadK {
  int N, B, T, splits, n_a, fm;
  const float* h1;           // h_seq + N*B*64  (h_t, t = 0..T-1)
  const float* dlv;          // [T][N][B][8]
  const int32_t* act;        // [T][N][B]
  float* ws;                 // [splits][N][HEAD_WS]
};
constexpr int HEAD_WS = 64 * 8 + 8 + NMARL_MAX_NBR * NMARL_MAX_NA;

__global__ void __launch_bounds__(256) head_wgrad_kernel(const __grid_constant__ nmarl_model m,
                                                        const __grid_constant__ HeadK k) {
  __shared__ float red[4][64][9];
  __shared__ float red2[256];
  const int sp = blockIdx.x, i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  const int tid = threadIdx.x, u = tid & 63, part = tid >> 6;
  const long R = (long)k.T * k.B;
  long r_begin, r_end;
  if (k.fm) {
    // feature-major h ([t][agent][unit][env]): the coalesced direction is env, so a warp covers 32 consecutive envs and
    // 8 of the 64 units; 8 x 8 accumulators per thread, one shuffle tree over the envs at the end.  (Reading it with
    // lanes = units touched 32 different 128-byte lines per load: 0.94 ms for 0.5 GB.)
    const long nb32 = R / 32, per32 = (nb32 + k.splits - 1) / k.splits;
    const long blk_begin = (long)sp * per32, blk_end = min(nb32, blk_begin + per32);
    r_begin = blk_begin * 32; r_end = blk_end * 32;
    const int lane = tid & 31, w = tid >> 5;
    float a[8][8];
#pragma unroll
    for (int uu = 0; uu < 8; ++uu)
#pragma unroll
      for (int c = 0; c < 8; ++c) a[uu][c] = 0.f;
    for (long blk = blk_begin; blk < blk_end; ++blk) {
      const long r = blk * 32 + lane, t = r / k.B, b = r - t * k.B;
      const size_t row = ((size_t)t * k.N + i) * k.B + b;
      const float4 d0 = *reinterpret_cast<const float4*>(k.dlv + row * 8);
      const float4 d1 = *reinterpret_cast<const float4*>(k.dlv + row * 8 + 4);
      const float dl[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      const float* hp = k.h1 + (((size_t)t * k.N + i) * NH + 8 * w) * k.B + b;
#pragma unroll
      for (int uu = 0; uu < 8; ++uu) {
        const float hv = hp[(size_t)uu * k.B];
#pragma unroll
        for (int c = 0; c < 8; ++c) a[uu][c] = fmaf(hv, dl[c], a[uu][c]);
      }
    }
#pragma unroll
    for (int uu = 0; uu < 8; ++uu)
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float x = a[uu][c];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) { red[0][8 * w + uu][c] = x; red[1][8 * w + uu][c] = 0.f; red[2][8 * w + uu][c] = 0.f; red[3][8 * w + uu][c] = 0.f; }
      }
  } else {
  const long per = (R + k.splits - 1) / k.splits;
  r_begin = (long)sp * per; r_end = min(R, r_begin + per);
  float acc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) acc[c] = 0.f;
  for (long r = r_begin + part; r < r_end; r += 4) {
    const long t = r / k.B, b = r - t * k.B;
    const size_t row = ((size_t)t * k.N + i) * k.B + b;
    const float hv = k.h1[row * NH + u];
    const float4 d0 = *reinterpret_cast<const float4*>(k.dlv + row * 8);
    const float4 d1 = *reinterpret_cast<const float4*>(k.dlv + row * 8 + 4);
    acc[0] = fmaf(hv, d0.x, acc[0]); acc[1] = fmaf(hv, d0.y, acc[1]); acc[2] = fmaf(hv, d0.z, acc[2]); acc[3] = fmaf(hv, d0.w, acc[3]);
    acc[4] = fmaf(hv, d1.x, acc[4]); acc[5] = fmaf(hv, d1.y, acc[5]); acc[6] = fmaf(hv, d1.z, acc[6]); acc[7] = fmaf(hv, d1.w, acc[7]);
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) red[part][u][c] = acc[c];
  }
  // bias sums (8) and one-hot sums (n_nbr x n_a): every thread strides over the rows, then a fixed-order
  // block reduction (warp shuffle tree + per-warp partials summed in warp order)
  constexpr int NX = 8 + NMARL_MAX_NBR * NMARL_MAX_NA;
  float ex[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) ex[c] = 0.f;
  const int n_extra = 8 + ag.n_nbr * k.n_a;
  for (long r = r_begin + tid; r < r_end; r += 256) {
    const long t = r / k.B, b = r - t * k.B;
    const size_t row = ((size_t)t * k.N + i) * k.B + b;
    const float4 d0 = *reinterpret_cast<const float4*>(k.dlv + row * 8);
    const float4 d1 = *reinterpret_cast<const float4*>(k.dlv + row * 8 + 4);
    const float dl[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
    for (int c = 0; c < 8; ++c) ex[c] += dl[c];
    const float dv = dl[k.n_a];
#pragma unroll
    for (int s = 0; s < NMARL_MAX_NBR; ++s) {
      if (s < ag.n_nbr) {
        const int a = k.act[((size_t)t * k.N + ag.nbr[s]) * k.B + b];
#pragma unroll
        for (int c = 0; c < NMARL_MAX_NA; ++c) ex[8 + s * NMARL_MAX_NA + c] += (c == a) ? dv : 0.f;
      }
    }
  }
  __shared__ float redx[8][NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) {
    float x = ex[c];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((tid & 31) == 0) redx[tid >> 5][c] = x;
  }
  __syncthreads();
  float extra = 0.f;
  if (tid < n_extra) {
    const int src = tid < 8 ? tid : 8 + ((tid - 8) / k.n_a) * NMARL_MAX_NA + (tid - 8) % k.n_a;
    for (int w2 = 0; w2 < 8; ++w2) extra += redx[w2][src];
  }
  red2[tid] = extra;
  __syncthreads();
  float* w = k.ws + ((size_t)sp * k.N + i) * HEAD_WS;
  for (int e = tid; e < 64 * 8; e += 256) {
    const int uu = e >> 3, c = e & 7;
    w[e] = ((red[0][uu][c] + red[1][uu][c]) + red[2][uu][c]) + red[3][uu][c];
  }
  if (tid < n_extra) w[64 * 8 + tid] = red2[tid];
}

struct HeadRedK { int N, splits, n_a; const float* ws; float* grads; };

__global__ void head_reduce_kernel(const __grid_constant__ nmarl_model m, const __grid_constant__ HeadRedK k) {
  const int i = blockIdx.x;
  const nmarl_agent& ag = m.agent[i];
  const int n_extra = 8 + ag.n_nbr * k.n_a;
  for (int e = threadIdx.x; e < 64 * 8 + n_extra; e += blockDim.x) {
    float s = 0.f;
    for (int sp = 0; sp < k.splits; ++sp) s += k.ws[((size_t)sp * k.N + i) * HEAD_WS + e];
    if (e < 64 * 8) {
      const int u = e >> 3, c = e & 7;
      if (c < k.n_a) k.grads[ag.o_pi_w + u * k.n_a + c] = s;
      else if (c == k.n_a) k.grads[ag.o_v_w + u] = s;
    } else {
      const int x = e - 64 * 8;
      if (x < k.n_a) k.grads[ag.o_pi_b + x] = s;
      else if (x == k.n_a) k.grads[ag.o_v_b] = s;
      else if (x >= 8) k.grads[ag.o_v_w + NH + (x - 8)] = s;
    }
  }
}

// ============================ K10: clip + RMSProp ================================================
struct OptK {
  int n_groups, nblk;
  int g_begin[NMARL_MAX_AGENT], g_end[NMARL_MAX_AGENT];
  float clip, rho, eps;
};

__global__ void __launch_bounds__(256) sumsq_kernel(const __grid_constant__ OptK k, const float* __restrict__ g,
                                                   float* __restrict__ scratch) {
  __shared__ float red[8];
  const int grp = blockIdx.y;
  const int beg = k.g_begin[grp], end = k.g_end[grp];
  float s = 0.f;
  for (int e = beg + blockIdx.x * 256 + threadIdx.x; e < end; e += gridDim.x * 256) { const float x = g[e]; s = fmaf(x, x, s); }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    scratch[grp * k.nblk + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) rmsprop_kernel(const __grid_constant__ OptK k, float* __restrict__ w,
                                                     const float* __restrict__ g, float* __restrict__ ms,
                                                     const float* __restrict__ lr_p, const float* __restrict__ scratch,
                                                     float* __restrict__ norm_out) {
  const int grp = blockIdx.y;
  double tot = 0.0;
  for (int x = 0; x < k.nblk; ++x) tot += (double)scratch[grp * k.nblk + x];
  const float gn = (float)sqrt(tot);
  if (blockIdx.x == 0 && threadIdx.x == 0) norm_out[grp] = gn;
  const float scale = (k.clip > 0.f) ? k.clip / fmaxf(gn, k.clip) : 1.0f;
  const float lr = *lr_p;
  const int beg = k.g_begin[grp], end = k.g_end[grp];
  for (int e = beg + blockIdx.x * 256 + threadIdx.x; e < end; e += gridDim.x * 256) {
    const float gg = g[e] * scale;
    const float m2 = k.rho * ms[e] + (1.0f - k.rho) * gg * gg;
    ms[e] = m2;
    w[e] = w[e] - lr * gg / sqrtf(m2 + k.eps);
  }
}

// Heads + A2C loss terms + d(loss)/d(logits, v) from the saved h sequence (thread == env row); used when the
// rollout already saved the cell activations.  Same arithmetic as the TRAIN epilogue of the forward kernels.
struct HeadFwdK {                 // pointers are for step 0; t = t0 + blockIdx.z strides them
  int B, N, loss_tiles, fm, t0;
  const float* params; const float* h1; const int32_t* act; const float* Rs; const float* Advs;
  float* sv_dlv; float* loss_part;
  float loss_scale, v_coef, e_coef;
};

__global__ void __launch_bounds__(128) train_heads_kernel(const __grid_constant__ nmarl_model m, const __grid_constant__ HeadFwdK k) {
  __shared__ float red[3][4];
  const int i = blockIdx.y, b = blockIdx.x * 128 + threadIdx.x, B = k.B, t = k.t0 + blockIdx.z;
  const nmarl_agent& ag = m.agent[i];
  const int n_a = m.n_a;
  const float* __restrict__ P = k.params;
  float l_pol = 0.f, l_val = 0.f, l_ent = 0.f;
  const size_t tb = (size_t)t * k.N * B;                    // step offset in rows
  if (b < B) {
    const size_t row = tb + (size_t)i * B + b;
    float logit[NMARL_MAX_NA];
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc) logit[cc] = 0.f;
    float v = 0.f;
#pragma unroll 4
    for (int q = 0; q < NH / 4; ++q) {
      float4 h4;
      if (k.fm) {
        const float* hp = k.h1 + ((tb / B + i) * NH + 4 * q) * (size_t)B + b;      // [t][agent][unit][env]
        h4 = make_float4(hp[0], hp[(size_t)B], hp[2 * (size_t)B], hp[3 * (size_t)B]);
      } else {
        h4 = *reinterpret_cast<const float4*>(k.h1 + row * NH + 4 * q);
      }
      const float4 vw = __ldg(reinterpret_cast<const float4*>(P + ag.o_v_w) + q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float hv = f4get(h4, j);
        const int u = 4 * q + j;
        if (n_a == 4) {                                   // one 16-byte load per unit instead of four scalar ones
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(P + ag.o_pi_w) + u);
          logit[0] = fmaf(hv, w4.x, logit[0]); logit[1] = fmaf(hv, w4.y, logit[1]);
          logit[2] = fmaf(hv, w4.z, logit[2]); logit[3] = fmaf(hv, w4.w, logit[3]);
        } else {
#pragma unroll
          for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
            if (cc < n_a) logit[cc] = fmaf(hv, __ldg(P + ag.o_pi_w + u * n_a + cc), logit[cc]);
        }
        v = fmaf(hv, f4get(vw, j), v);
      }
    }
    float pi[NMARL_MAX_NA];
    float mx = -3.0e38f;
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
      if (cc < n_a) { logit[cc] += __ldg(P + ag.o_pi_b + cc); mx = fmaxf(mx, logit[cc]); }
    float se = 0.f;
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
      if (cc < n_a) { pi[cc] = expf(logit[cc] - mx); se += pi[cc]; } else pi[cc] = 0.f;
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc) if (cc < n_a) pi[cc] = pi[cc] / se;
    for (int s = 0; s < ag.n_nbr; ++s) v += __ldg(P + ag.o_v_w + NH + s * n_a + k.act[tb + (size_t)ag.nbr[s] * B + b]);
    v += __ldg(P + ag.o_v_b);
    const int act = k.act[row];
    const float R = k.Rs[row], Adv = k.Advs[row], cs = k.loss_scale;
    float g[NMARL_MAX_NA];
    float ent = 0.f, dot = 0.f, lpa = 0.f;
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc) {
      g[cc] = 0.f;
      if (cc < n_a) {
        const float pc = fminf(fmaxf(pi[cc], 1e-10f), 1.0f);
        const float in_rng = (pi[cc] >= 1e-10f && pi[cc] <= 1.0f) ? 1.0f : 0.0f;
        const float lp = logf(pc);
        ent -= pi[cc] * lp;
        g[cc] = k.e_coef * cs * (lp + in_rng);
        if (cc == act) { g[cc] += -cs * Adv * in_rng / pc; lpa = lp; }
        dot += pi[cc] * g[cc];
      }
    }
    float dl[8];
#pragma unroll
    for (int cc = 0; cc < 8; ++cc) dl[cc] = (cc < n_a) ? pi[cc] * (g[cc] - dot) : 0.f;
    const float dvv = -k.v_coef * cs * (R - v);
#pragma unroll
    for (int cc = 0; cc < 8; ++cc) if (cc == n_a) dl[cc] = dvv;
    *reinterpret_cast<float4*>(k.sv_dlv + row * 8) = make_float4(dl[0], dl[1], dl[2], dl[3]);
    *reinterpret_cast<float4*>(k.sv_dlv + row * 8 + 4) = make_float4(dl[4], dl[5], dl[6], dl[7]);
    l_pol = -lpa * Adv; l_val = (R - v) * (R - v); l_ent = ent;
  }
  float vals[3] = {l_pol, l_val, l_ent};
#pragma unroll
  for (int cc = 0; cc < 3; ++cc) {
    float x = vals[cc];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) == 0) red[cc][threadIdx.x >> 5] = x;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const float s = ((red[threadIdx.x][0] + red[threadIdx.x][1]) + red[threadIdx.x][2]) + red[threadIdx.x][3];
    float* lp = k.loss_part + (((size_t)t * k.N + i) * k.loss_tiles + 2 * blockIdx.x) * 4;
    lp[threadIdx.x] = s;
    if (2 * blockIdx.x + 1 < k.loss_tiles) lp[4 + threadIdx.x] = 0.f;
  }
}

constexpr int BWD_BM = 64, BWD_TY = 16;

template <int VAR>
int launch_bwd(const nmarl_model* m, const BwdK& k, cudaStream_t st) {
  constexpr int NGRP = (VAR == NMARL_NC) ? 4 : 2;
  auto kern = cell_bwd_kernel<VAR, BWD_BM, BWD_TY>;
  const size_t smem = ((size_t)BWD_BM * (NG + 4) + 2 * 16 * 64 * NGRP) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    NMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  dim3 grid((k.B + BWD_BM - 1) / BWD_BM, m->n_agent);
  kern<<<grid, 16 * BWD_TY, smem, st>>>(*m, k);
  NMARL_LAUNCH_CHECK();
  return 0;
}

int wgrad_splits(long R) {
  long s = R / 4096;
  if (s < 1) s = 1;
  if (s > 32) s = 32;
  return (int)s;
}

int head_splits(long R) {
  long s = R / 1024;
  if (s < 1) s = 1;
  if (s > 512) s = 512;
  return (int)s;
}

int run_wgrad(const nmarl_model* m, const nmarl_bwd_args* a, int ngrp, const float* A, int lda, int a_col0,
              const float* D, int ldd, int d_col0, const int* Ka, const int* o_w, const int* o_b, cudaStream_t st) {
  WgK k{};
  k.N = m->n_agent; k.B = a->B; k.T = a->T;
  k.splits = wgrad_splits((long)a->B * a->T);
  k.A = A; k.lda = lda; k.a_col0 = a_col0; k.D = D; k.ldd = ldd; k.d_col0 = d_col0;
  int kmax = 0;
  for (int i = 0; i < m->n_agent; ++i) { k.Ka[i] = Ka[i]; kmax = Ka[i] > kmax ? Ka[i] : kmax; }
  if (kmax == 0) return 0;
  k.ka_max = kmax; k.ws = a->ws;
  const int nd = 64 * ngrp;
  NMARL_CHECK((int64_t)k.splits * k.N * (kmax + 1) * nd <= a->ws_floats, "wgrad: workspace too small");
  dim3 grid(k.splits, (kmax + 63) / 64, m->n_agent);
  const size_t smem = (size_t)(2 * 32 * 64 + 2 * 32 * nd) * sizeof(float);
  static bool configured = false;
  if (!configured) {
    NMARL_CUDA(cudaFuncSetAttribute(wgrad_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((2 * 32 * 64 + 2 * 32 * 256) * sizeof(float))));
    configured = true;
  }
  if (ngrp == 4) wgrad_kernel<4><<<grid, 256, smem, st>>>(k);
  else wgrad_kernel<1><<<grid, 256, smem, st>>>(k);
  NMARL_LAUNCH_CHECK();
  WgRedK r{};
  r.N = k.N; r.splits = k.splits; r.ka_max = kmax; r.nd = nd; r.ws = a->ws; r.grads = a->grads;
  for (int i = 0; i < m->n_agent; ++i) { r.Ka[i] = Ka[i]; r.o_w[i] = o_w[i]; r.o_b[i] = o_b[i]; }
  dim3 rg(((kmax + 1) * nd + 255) / 256, m->n_agent);
  wgrad_reduce_kernel<<<rg, 256, 0, st>>>(r);
  NMARL_LAUNCH_CHECK();
  return 0;
}

int check_bwd_args(const nmarl_model* m, const nmarl_bwd_args* a) {
  if (nmarl_check_model(m)) return 1;
  NMARL_CHECK(a && a->B > 0 && a->T > 0 && a->B_total >= a->B, "a2c_backward: bad sizes");
  NMARL_CHECK(a->params && a->obs && a->act && a->done_pre && a->Rs && a->Advs && a->h_seq && a->c_seq,
              "a2c_backward: missing rollout buffers");
  NMARL_CHECK(a->sv_xin && a->sv_sh && a->sv_gates && a->sv_dlv && a->sv_dz && a->sv_dpre && a->dh_rec && a->dc_rec &&
                  a->wt && a->ws && a->loss_part && a->grads,
              "a2c_backward: missing scratch buffers");
  NMARL_CHECK(m->variant == NMARL_IA2C || a->dmsg, "a2c_backward: dmsg buffer required");
  NMARL_CHECK((m->variant != NMARL_IC3 && m->variant != NMARL_DIAL) || a->sv_enc, "a2c_backward: sv_enc required");
  NMARL_CHECK(m->variant != NMARL_DIAL || (a->msg_seq && a->sv_dmp), "a2c_backward: DIAL buffers required");
  const int fm = nmarl_state_fm(m, a->wpack != nullptr && nmarl_tc_supported(m, a->B));
  NMARL_CHECK(a->state_fm == fm, "a2c_backward: state_fm must be %d for this variant and path, got %d", fm, a->state_fm);
  NMARL_CHECK((m->variant != NMARL_NC && m->variant != NMARL_DIAL) || a->fp, "a2c_backward: fp required");
  return 0;
}

}  // namespace

extern "C" int nmarl_loss_tiles(const nmarl_model* m, int B) { (void)m; return nmarl_fwd_tiles(B); }

extern "C" int64_t nmarl_ws_floats(const nmarl_model* m, int B, int T) {
  const int splits = wgrad_splits((long)B * T);
  int64_t gate = (int64_t)splits * m->n_agent * (m->s_dim + NH + 1) * NG;
  int64_t enc = (int64_t)splits * m->n_agent * (m->km_pad + m->kx_pad + 1) * NH;
  int64_t head = (int64_t)head_splits((long)B * T) * m->n_agent * HEAD_WS;
  int64_t r = gate > enc ? gate : enc;
  r = r > head ? r : head;
  const int64_t tcw = nmarl_tc_wgrad_ws_floats(m);
  return r > tcw ? r : tcw;
}

extern "C" int nmarl_nstep_return_adv(int n_agent, int B, int T, int NR, const double* reward, const float* value,
                                      const float* done_post, const float* R_end, int zero_end_if_done, double gamma,
                                      double reward_norm, double reward_clip, double alpha, const int32_t* dist,
                                      const double* alpha_pow, int n_pow, float* Rs, float* Advs, void* stream) {
  NMARL_CHECK(n_agent > 0 && B > 0 && T > 0 && reward && value && done_post && R_end && Rs && Advs, "nstep_return_adv: bad arguments");
  NMARL_CHECK(alpha < 0 || (dist && alpha_pow && n_pow > 0 && NR == n_agent), "nstep_return_adv: spatial variant needs dist/alpha_pow and per-agent rewards");
  NMARL_CHECK(NR == 1 || NR == n_agent, "nstep_return_adv: NR must be 1 or n_agent");
  RetK k{n_agent, B, T, NR, zero_end_if_done, gamma, reward_norm, reward_clip, alpha, n_pow};
  const int n = n_agent * B;
  nstep_return_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(k, reward, value, done_post, R_end, dist,
                                                                          alpha_pow, Rs, Advs);
  NMARL_LAUNCH_CHECK();
  return 0;
}

extern "C" int nmarl_a2c_train_forward(const nmarl_model* m, const nmarl_bwd_args* a, void* stream) {
  if (check_bwd_args(m, a)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = m->n_agent, B = a->B, T = a->T;
  const size_t nb = (size_t)N * B;
  const int LDI = m->kx_pad + m->kp_pad + m->km_pad;
  const int tiles = nmarl_fwd_tiles(B);
  const float scale = 1.0f / ((float)T * (float)a->B_total);
  for (int t = 0; t < T; ++t) {
    nmarl_fwd_args f{};
    f.B = B; f.params = a->params;
    f.obs = a->obs + (size_t)t * nb * m->obs_stride;
    f.fp = a->fp ? a->fp + (size_t)t * nb * m->n_a : nullptr;
    f.done = a->done_pre + (size_t)t * B;
    f.c_in = a->c_seq + (size_t)t * nb * NH;       f.h_in = a->h_seq + (size_t)t * nb * NH;
    f.c_out = a->c_seq + (size_t)(t + 1) * nb * NH; f.h_out = a->h_seq + (size_t)(t + 1) * nb * NH;
    if (m->variant == NMARL_DIAL) { f.msg_in = a->msg_seq + (size_t)t * nb * NH; f.msg_out = a->msg_seq + (size_t)(t + 1) * nb * NH; }
    f.act_in = a->act + (size_t)t * nb;
    f.wpack = a->wpack; f.tc_err = a->tc_err; f.state_fm = a->state_fm;
    int rc = nmarl_launch_train_fwd(m, &f, a->Rs + (size_t)t * nb, a->Advs + (size_t)t * nb,
                                    a->sv_xin + (size_t)t * nb * LDI, a->sv_sh + (size_t)t * nb * (m->s_dim + NH),
                                    a->sv_gates + (size_t)t * nb * NG, a->sv_enc ? a->sv_enc + (size_t)t * nb * 128 : nullptr,
                                    a->sv_dlv + (size_t)t * nb * 8, a->loss_part + (size_t)t * N * tiles * 4, scale,
                                    a->v_coef, a->e_coef, st);
    if (rc) return rc;
  }
  return 0;
}

// heads + loss partials + d(loss)/d(logits, v) of time steps [t0, t0 + nt) from h_seq
static int launch_train_heads(const nmarl_model* m, const nmarl_bwd_args* a, int t0, int nt, cudaStream_t st) {
  if (nt <= 0) return 0;
  const int N = m->n_agent, B = a->B, T = a->T;
  const size_t nb = (size_t)N * B;
  HeadFwdK k{};
  k.B = B; k.N = N; k.loss_tiles = nmarl_fwd_tiles(B); k.params = a->params; k.fm = a->state_fm; k.t0 = t0;
  k.h1 = a->h_seq + nb * NH;                                  // h after step t = h_seq[t + 1]
  k.act = a->act; k.Rs = a->Rs; k.Advs = a->Advs;
  k.sv_dlv = a->sv_dlv; k.loss_part = a->loss_part;
  k.loss_scale = 1.0f / ((float)T * (float)a->B_total); k.v_coef = a->v_coef; k.e_coef = a->e_coef;
  train_heads_kernel<<<dim3((B + 127) / 128, N, nt), 128, 0, st>>>(*m, k);
  NMARL_LAUNCH_CHECK();
  return 0;
}

extern "C" int nmarl_a2c_train_heads(const nmarl_model* m, const nmarl_bwd_args* a, void* stream) {
  if (check_bwd_args(m, a)) return 1;
  return launch_train_heads(m, a, 0, a->T, (cudaStream_t)stream);
}

extern "C" int nmarl_a2c_bptt(const nmarl_model* m, const nmarl_bwd_args* a, void* stream) {
  if (check_bwd_args(m, a)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  const int N = m->n_agent, B = a->B, T = a->T, SD = m->s_dim;
  const size_t nb = (size_t)N * B;
  // 0. gradients of padding slots stay zero
  NMARL_CUDA(cudaMemsetAsync(a->grads, 0, (size_t)m->n_param * sizeof(float), st));
  // tensor-core path (reverse steps and weight gradients) or FFMA path, as in the forward (nmarl_tc_fwd_supported)
  const bool tc = a->wpack != nullptr && nmarl_tc_supported(m, B);
  // 1. transposed weights for the FFMA backward kernels and DIAL's message-gradient kernel (the tensor-core cell
  //    kernels read their own packed transposed operands, refreshed by nmarl_pack_weights)
  if (!tc || m->variant == NMARL_DIAL)
  for (int i = 0; i < N; ++i) {
    const nmarl_agent& ag = m->agent[i];
    dim3 blk(32, 8);
    {
      const int rows = SD + NH, cols = NG;
      transpose_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), blk, 0, st>>>(a->params + ag.o_wxh, a->wt + ag.t_wxh, rows, cols);
    }
    if (m->variant != NMARL_IA2C) {
      const int rows = (m->variant == NMARL_IC3) ? NH : ag.n_nbr * NH, cols = NH;
      if (rows > 0) transpose_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), blk, 0, st>>>(a->params + ag.o_w_msg, a->wt + ag.t_w_msg, rows, cols);
    }
    if (m->variant == NMARL_DIAL)
      transpose_kernel<<<dim3(2, 2), blk, 0, st>>>(a->params + ag.o_mfc_w, a->wt + ag.t_mfc, NH, NH);
  }
  NMARL_LAUNCH_CHECK();
  // 1b. policy/value head weight gradients need only sv_dlv and h_seq: they run on a forked stream
  //     beside the BPTT chain (whose 256-CTA launches leave SMs idle in their second wave) and join
  //     before the weight-gradient phase, which shares the workspace.
  //     The helper stream and its two events live in the caller's nmarl_ctx.
  NMARL_CHECK(a->ctx != nullptr, "a2c_bptt: nmarl_bwd_args.ctx is NULL (nmarl_create)");
  cudaStream_t side = a->ctx->side;
  cudaEvent_t ev_fork = a->ctx->fork, ev_join = a->ctx->join;
  // fused_heads (saved-rollout path): the heads / loss kernel (nmarl_a2c_train_heads) is folded in.  Only the last
  // HEAD_LEAD time steps are computed on the caller's stream before the reverse chain starts; the remaining steps run
  // on the side stream beside the first reverse steps (the chain reaches step T-1-HEAD_LEAD long after they are done).
  constexpr int HEAD_LEAD = 6;
  const int lead = a->fused_heads ? (T < HEAD_LEAD ? T : HEAD_LEAD) : 0;
  if (a->fused_heads && launch_train_heads(m, a, T - lead, lead, st)) return 1;
  NMARL_CUDA(cudaEventRecord(ev_fork, st));
  NMARL_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
  if (a->fused_heads) {
    if (launch_train_heads(m, a, 0, T - lead, side)) return 1;
    NMARL_CUDA(cudaEventRecord(a->ctx->heads, side));
  }
  {
    HeadK h{};
    h.N = N; h.B = B; h.T = T; h.splits = head_splits((long)B * T); h.n_a = m->n_a; h.fm = a->state_fm;
    h.h1 = a->h_seq + nb * NH; h.dlv = a->sv_dlv; h.act = a->act; h.ws = a->ws;
    NMARL_CHECK((int64_t)h.splits * N * HEAD_WS <= a->ws_floats, "head wgrad: workspace too small");
    head_wgrad_kernel<<<dim3(h.splits, N), 256, 0, side>>>(*m, h);
    NMARL_LAUNCH_CHECK();
    HeadRedK r{N, h.splits, m->n_a, a->ws, a->grads};
    head_reduce_kernel<<<N, 256, 0, side>>>(*m, r);
    NMARL_LAUNCH_CHECK();
  }
  NMARL_CUDA(cudaEventRecord(ev_join, side));
  // 2. reverse time
  for (int t = T - 1; t >= 0; --t) {
    BwdK k{};
    k.B = B; k.t = t; k.has_next = (t < T - 1);
    k.params = a->params; k.wt = a->wt;
    k.done_pre = a->done_pre + (size_t)t * B;
    k.sv_gates = a->sv_gates + (size_t)t * nb * NG;
    k.sv_sh = a->sv_sh + (size_t)t * nb * (SD + NH);
    k.sv_enc = a->sv_enc ? a->sv_enc + (size_t)t * nb * 128 : nullptr;
    k.sv_dlv = a->sv_dlv + (size_t)t * nb * 8;
    k.c_prev = a->c_seq + (size_t)t * nb * NH;
    k.c_cur = a->c_seq + (size_t)(t + 1) * nb * NH;
    const int pin = (t + 1) & 1, pout = t & 1;
    k.dh_in = a->dh_rec + (size_t)pin * nb * NH;  k.dh_out = a->dh_rec + (size_t)pout * nb * NH;
    k.dc_in = a->dc_rec + (size_t)pin * nb * NH;  k.dc_out = a->dc_rec + (size_t)pout * nb * NH;
    if (a->dmsg) {
      k.dmsg_in = a->dmsg + (size_t)pin * nb * NMARL_MAX_NBR * NH;
      k.dmsg_out = a->dmsg + (size_t)pout * nb * NMARL_MAX_NBR * NH;
    }
    k.sv_dpre = a->sv_dpre + (size_t)t * nb * 192;
    k.wpack = a->wpack; k.tc_err = a->tc_err;
    // tensor-core path: sv_dz holds the per-tile gate-bias partial sums [T][N][B/128][256]; FFMA path: dz [T][N][B][256]
    k.sv_dz = tc ? a->sv_dz + (size_t)t * N * (B / 128) * NG : a->sv_dz + (size_t)t * nb * NG;
    k.ndp = nmarl_tc_ndp(m);
    k.dzT = (tc && a->sv_dzT) ? a->sv_dzT + t * nmarl_tc_tile_step_floats(N, B, 256) : nullptr;
    k.dpT = (tc && a->sv_dpT) ? a->sv_dpT + t * nmarl_tc_tile_step_floats(N, B, k.ndp) : nullptr;
    int rc = 0;
    if (a->fused_heads && t == T - 1 - lead) NMARL_CUDA(cudaStreamWaitEvent(st, a->ctx->heads, 0));   // dlv of steps < T - lead
    if (a->ev_step) NMARL_CUDA(cudaEventRecord((cudaEvent_t)a->ev_step[2 * t], st));
    if (tc) rc = nmarl_tc_launch_bwd(m, k, st);
    else
    switch (m->variant) {
      case NMARL_IA2C: rc = launch_bwd<NMARL_IA2C>(m, k, st); break;
      case NMARL_NC: rc = launch_bwd<NMARL_NC>(m, k, st); break;
      case NMARL_IC3: rc = launch_bwd<NMARL_IC3>(m, k, st); break;
      case NMARL_DIAL: rc = launch_bwd<NMARL_DIAL>(m, k, st); break;
    }
    if (rc) return rc;
    if (a->ev_step) NMARL_CUDA(cudaEventRecord((cudaEvent_t)a->ev_step[2 * t + 1], st));
    NMARL_DBG_SYNC(st, "cell_bwd");
    if (m->variant == NMARL_DIAL) {
      dim3 grid((B + 63) / 64, N);
      dial_msg_bwd_kernel<64, 16><<<grid, 256, 0, st>>>(*m, B, a->wt, a->msg_seq + (size_t)t * nb * NH, k.dmsg_out,
                                                        a->sv_dmp + (size_t)t * nb * NH, k.dh_out);
      NMARL_LAUNCH_CHECK();
    }
  }
  // 3. weight gradients
  NMARL_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
  int Ka[NMARL_MAX_AGENT], ow[NMARL_MAX_AGENT], ob[NMARL_MAX_AGENT];
  const int LDI = m->kx_pad + m->kp_pad + m->km_pad;
  if (tc) {
    NMARL_CHECK(a->sv_dzT && a->sv_dpT, "a2c_bptt: tensor-core path needs sv_dzT / sv_dpT");
    NMARL_CHECK(nmarl_tc_wgrad_ws_floats(m) <= a->ws_floats, "tc wgrad: workspace too small");
    // the gate-bias column sums only read sv_dz: second fork, beside the GEMM jobs
    NMARL_CUDA(cudaEventRecord(ev_fork, st));
    NMARL_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
    if (nmarl_tc_launch_wgrads(m, B, T, a->sv_sh, a->sv_xin, a->sv_dzT, a->sv_dpT, a->sv_dz, a->ws, a->grads, a->tc_err, st, side, a->ev_wgrad,
                               a->state_fm ? a->h_seq : nullptr, a->done_pre)) return 1;
    NMARL_CUDA(cudaEventRecord(ev_join, side));
    NMARL_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
    NMARL_DBG_SYNC(st, "tc_wgrads");
  } else {
    for (int i = 0; i < N; ++i) { Ka[i] = SD + NH; ow[i] = m->agent[i].o_wxh; ob[i] = m->agent[i].o_b; }
    if (run_wgrad(m, a, 4, a->sv_sh, SD + NH, 0, a->sv_dz, NG, 0, Ka, ow, ob, st)) return 1;
    for (int i = 0; i < N; ++i) { Ka[i] = m->agent[i].x_nsrc * m->agent[i].x_w; ow[i] = m->agent[i].o_w_ob; ob[i] = m->agent[i].o_b_ob; }
    if (run_wgrad(m, a, 1, a->sv_xin, LDI, 0, a->sv_dpre, 192, 0, Ka, ow, ob, st)) return 1;
    if (m->variant == NMARL_NC) {
      for (int i = 0; i < N; ++i) { Ka[i] = m->agent[i].n_nbr * m->n_a; ow[i] = m->agent[i].o_w_fp; ob[i] = m->agent[i].o_b_fp; }
      if (run_wgrad(m, a, 1, a->sv_xin, LDI, m->kx_pad, a->sv_dpre, 192, NH, Ka, ow, ob, st)) return 1;
    }
    if (m->variant != NMARL_IA2C) {
      for (int i = 0; i < N; ++i) {
        Ka[i] = (m->variant == NMARL_IC3) ? NH : m->agent[i].n_nbr * NH;
        ow[i] = m->agent[i].o_w_msg; ob[i] = m->agent[i].o_b_msg;
      }
      if (run_wgrad(m, a, 1, a->sv_xin, LDI, m->kx_pad + m->kp_pad, a->sv_dpre, 192, (m->variant == NMARL_NC) ? 2 * NH : NH,
                    Ka, ow, ob, st)) return 1;
    }
  }
  if (m->variant == NMARL_DIAL) {
    for (int i = 0; i < N; ++i) { Ka[i] = NH; ow[i] = m->agent[i].o_mfc_w; ob[i] = m->agent[i].o_mfc_b; }
    if (run_wgrad(m, a, 1, a->h_seq, NH, 0, a->sv_dmp, NH, 0, Ka, ow, ob, st)) return 1;
  }
  (void)0;
  return 0;
}

extern "C" int nmarl_a2c_backward(const nmarl_model* m, const nmarl_bwd_args* a, void* stream) {
  int rc = nmarl_a2c_train_forward(m, a, stream);
  if (rc) return rc;
  return nmarl_a2c_bptt(m, a, stream);
}

extern "C" int nmarl_clip_rmsprop_step(const nmarl_model* m, float* params, float* grads, float* ms, const float* lr,
                                       float max_grad_norm, float rho, float eps, float* norm_out, float* scratch,
                                       void* stream) {
  if (nmarl_check_model(m)) return 1;
  NMARL_CHECK(params && grads && ms && lr && norm_out && scratch, "clip_rmsprop_step: missing buffers");
  OptK k{};
  k.clip = max_grad_norm; k.rho = rho; k.eps = eps;
  if (m->per_agent_norm) {
    k.n_groups = m->n_agent;
    for (int i = 0; i < m->n_agent; ++i) { k.g_begin[i] = m->agent[i].p_begin; k.g_end[i] = m->agent[i].p_end; }
  } else {
    k.n_groups = 1; k.g_begin[0] = 0; k.g_end[0] = m->n_param;
  }
  k.nblk = (k.n_groups == 1) ? 256 : 32;       // n_groups * nblk <= 1024 scratch floats
  cudaStream_t st = (cudaStream_t)stream;
  sumsq_kernel<<<dim3(k.nblk, k.n_groups), 256, 0, st>>>(k, grads, scratch);
  NMARL_LAUNCH_CHECK();
  rmsprop_kernel<<<dim3(k.nblk, k.n_groups), 256, 0, st>>>(k, params, grads, ms, lr, scratch, norm_out);
  NMARL_LAUNCH_CHECK();
  return 0;
}

// ---- consensus update of the LSTM blocks (ma2c_cu) -------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) consensus_mean_kernel(const __grid_constant__ nmarl_model m, const float* __restrict__ params,
                                                            float* __restrict__ scratch, int n) {
  const int i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
    float s = params[ag.o_wxh + e];                      // own block first, then neighbours ascending
    for (int k = 0; k < ag.n_nbr; ++k) s += params[m.agent[ag.nbr[k]].o_wxh + e];
    scratch[(size_t)i * n + e] = s / (float)(1 + ag.n_nbr);
  }
}
__global__ void __launch_bounds__(256) consensus_store_kernel(const __grid_constant__ nmarl_model m, float* __restrict__ params,
                                                             const float* __restrict__ scratch, int n) {
  const int i = blockIdx.y;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x)
    params[m.agent[i].o_wxh + e] = scratch[(size_t)i * n + e];
}
}  // namespace

extern "C" int nmarl_consensus_update(const nmarl_model* m, float* params, float* scratch, void* stream) {
  if (nmarl_check_model(m)) return 1;
  NMARL_CHECK(params && scratch, "consensus_update: missing buffers");
  const int n = (m->s_dim + NH) * NG + NG;
  for (int i = 0; i < m->n_agent; ++i)
    NMARL_CHECK(m->agent[i].o_b == m->agent[i].o_wxh + (m->s_dim + NH) * NG, "consensus_update: LSTM block of agent %d is not contiguous", i);
  cudaStream_t st = (cudaStream_t)stream;
  consensus_mean_kernel<<<dim3(32, m->n_agent), 256, 0, st>>>(*m, params, scratch, n);
  NMARL_LAUNCH_CHECK();
  consensus_store_kernel<<<dim3(32, m->n_agent), 256, 0, st>>>(*m, params, scratch, n);
  NMARL_LAUNCH_CHECK();
  return 0;
}
