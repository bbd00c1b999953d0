// cell_fwd.cu -- K2..K6 fused: neighbour gather -> encoders -> LSTM gate GEMM -> cell update ->
// actor / critic heads -> action sampling, for one env step of every agent.
//
// Grid: (env tiles, agents).  One CTA owns BM envs of ONE agent (weights are per agent, never
// shared: agents/utils.py:141-162), so each GEMM below is one group of a grouped GEMM with
// M = BM rows.  FP32 FFMA, k-ascending (the 1e-5 parity budget on logits/values rules out
// plain TF32; see DESIGN.md).  Shared memory: IN tile [BM][kx+kp+km] (gathered x~|p~|m~),
// SH tile [BM][s_dim+64] (encoder outputs s | done-masked own h) and a cp.async weight ring.
//
// Restates (per agent i, gate order i,f,o,u, state [c|h]):
//   lstm_comm  agents/utils.py:163-217      lstm_ic3  :378-417      lstm_dial :555-599
//   lstm (IA2C) :87-115 + fc policies.py:145   heads policies.py:50-77   sampling utils.py:135-141
//   A2C loss terms policies.py:236-255 (TRAIN mode: per-row loss + d/dlogits, d/dv)
#include "cell_common.cuh"

namespace {

template <int BM, int KC>
__host__ __device__ inline size_t fwd_region0_floats(const nmarl_model& m) {
  const size_t in = (size_t)BM * (m.kx_pad + m.kp_pad + m.km_pad);
  const size_t ring = (size_t)2 * KC * NG;
  const size_t hs = (size_t)BM * (NH + 4);
  size_t r = in > ring ? in : ring;
  return r > hs ? r : hs;
}
template <int BM, int KC>
__host__ __device__ inline size_t fwd_smem_floats(const nmarl_model& m) {
  return fwd_region0_floats<BM, KC>(m) + (size_t)BM * (m.s_dim + NH + 4) + (size_t)2 * KC * NH;
}

template <int VAR, int MODE, int BM, int TY>
__global__ void __launch_bounds__(16 * TY) cell_fwd_kernel(const __grid_constant__ nmarl_model m,
                                                          const __grid_constant__ FwdK k) {
  constexpr int NT = 16 * TY, TM = BM / TY, KC = 16;
  static_assert(BM % TY == 0 && NT >= BM, "tile/thread mismatch");
  extern __shared__ __align__(16) float smem[];
  const nmarl_fwd_args& a = k.a;
  const int i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  const int B = a.B, b0 = blockIdx.x * BM;
  const int rows = min(BM, B - b0);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n_a = m.n_a, SD = m.s_dim;
  const int LDI = m.kx_pad + m.kp_pad + m.km_pad, PO = m.kx_pad, MO = m.kx_pad + m.kp_pad;
  const int LDS = SD + NH + 4;
  float* IN = smem;
  float* SH = smem + fwd_region0_floats<BM, KC>(m);
  float* WsE = SH + (size_t)BM * LDS;
  float* WsG = smem;                     // gate-weight ring aliases IN (dead after the encoders)
  float* Hs = smem;                      // new-h tile aliases the ring (dead after the gate GEMM)
  constexpr int LDH = NH + 4;
  const float* __restrict__ P = a.params;

  // ---- phase 0: gather inputs (agent-major global -> row-major smem) ------------------------
  const int Kx = ag.x_nsrc * ag.x_w;
  for (int idx = tid; idx < BM * m.kx_pad; idx += NT) {
    const int r = idx / m.kx_pad, kk = idx - r * m.kx_pad;
    float v = 0.f;
    if (r < rows && kk < Kx) {
      const int s = kk / ag.x_w, f = kk - s * ag.x_w;
      v = a.obs[((size_t)ag.x_src[s] * B + b0 + r) * m.obs_stride + f];
    }
    IN[r * LDI + kk] = v;
  }
  if (VAR == NMARL_NC) {
    const int Kp = ag.n_nbr * n_a;
    for (int idx = tid; idx < BM * m.kp_pad; idx += NT) {
      const int r = idx / m.kp_pad, kk = idx - r * m.kp_pad;
      float v = 0.f;
      if (r < rows && kk < Kp) {
        const int s = kk / n_a, f = kk - s * n_a;
        v = a.fp[((size_t)ag.nbr[s] * B + b0 + r) * n_a + f];
      }
      IN[r * LDI + PO + kk] = v;
    }
  }
  if (VAR == NMARL_NC || VAR == NMARL_DIAL) {
    const float* src = (VAR == NMARL_NC) ? a.h_in : a.msg_in;      // messages: UN-masked (utils.py:182-183)
    const int q4 = m.km_pad / 4;
    for (int idx = tid; idx < BM * q4; idx += NT) {
      const int r = idx / q4, c4 = idx - r * q4;
      const int s = c4 / (NH / 4), u4 = c4 - s * (NH / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows && s < ag.n_nbr)
        v = *reinterpret_cast<const float4*>(src + ((size_t)ag.nbr[s] * B + b0 + r) * NH + 4 * u4);
      *reinterpret_cast<float4*>(IN + r * LDI + MO + 4 * c4) = v;
    }
  }
  if (VAR == NMARL_IC3) {                                             // mean of neighbours' h (utils.py:395)
    for (int idx = tid; idx < BM * (NH / 4); idx += NT) {
      const int r = idx / (NH / 4), u4 = idx - r * (NH / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows) {
        for (int s = 0; s < ag.n_nbr; ++s) {
          const float4 w = *reinterpret_cast<const float4*>(a.h_in + ((size_t)ag.nbr[s] * B + b0 + r) * NH + 4 * u4);
          v.x += w.x; v.y += w.y; v.z += w.z; v.w += w.w;
        }
        const float nn = (float)ag.n_nbr;
        v.x /= nn; v.y /= nn; v.z /= nn; v.w /= nn;
      }
      *reinterpret_cast<float4*>(IN + r * LDI + MO + 4 * u4) = v;
    }
  }
  for (int idx = tid; idx < BM * (NH / 4); idx += NT) {                // own h, done-masked (utils.py:189-190)
    const int r = idx / (NH / 4), u4 = idx - r * (NH / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows) {
      v = *reinterpret_cast<const float4*>(a.h_in + ((size_t)i * B + b0 + r) * NH + 4 * u4);
      const float nd = 1.0f - a.done[b0 + r];
      v.x *= nd; v.y *= nd; v.z *= nd; v.w *= nd;
    }
    *reinterpret_cast<float4*>(SH + r * LDS + SD + 4 * u4) = v;
  }
  __syncthreads();
  if (MODE == MODE_TRAIN) {                                            // save gathered inputs for wgrad
    const int q4 = LDI / 4;
    for (int idx = tid; idx < rows * q4; idx += NT) {
      const int r = idx / q4, c4 = idx - r * q4;
      *reinterpret_cast<float4*>(k.sv_xin + ((size_t)i * B + b0 + r) * LDI + 4 * c4) =
          *reinterpret_cast<const float4*>(IN + r * LDI + 4 * c4);
    }
  }

  // ---- phase 1: encoders -> s (columns [0, s_dim) of SH) -------------------------------------
  float sv[TM][4];
  {
    float acc[TM][4];
#pragma unroll
    for (int q = 0; q < TM; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f; }
    gemm_rowA<TM, 1, TY, KC>(acc, IN, LDI, Kx, P + ag.o_w_ob, NH, WsE, tid);
    const float4 bb = *reinterpret_cast<const float4*>(P + ag.o_b_ob + 4 * tx);
#pragma unroll
    for (int q = 0; q < TM; ++q) {
      const float z0 = acc[q][0] + bb.x, z1 = acc[q][1] + bb.y, z2 = acc[q][2] + bb.z, z3 = acc[q][3] + bb.w;
      if (VAR == NMARL_IC3) { sv[q][0] = tanhf(z0); sv[q][1] = tanhf(z1); sv[q][2] = tanhf(z2); sv[q][3] = tanhf(z3); }
      else { sv[q][0] = fmaxf(z0, 0.f); sv[q][1] = fmaxf(z1, 0.f); sv[q][2] = fmaxf(z2, 0.f); sv[q][3] = fmaxf(z3, 0.f); }
      const int r = ty + TY * q;
      if (VAR == NMARL_NC || VAR == NMARL_IA2C)
        *reinterpret_cast<float4*>(SH + r * LDS + 4 * tx) = make_float4(sv[q][0], sv[q][1], sv[q][2], sv[q][3]);
      if (MODE == MODE_TRAIN && (VAR == NMARL_IC3 || VAR == NMARL_DIAL) && r < rows)
        *reinterpret_cast<float4*>(k.sv_enc + ((size_t)i * B + b0 + r) * 128 + 4 * tx) =
            make_float4(sv[q][0], sv[q][1], sv[q][2], sv[q][3]);
    }
  }
  if (VAR == NMARL_NC) {
    float acc[TM][4];
#pragma unroll
    for (int q = 0; q < TM; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f; }
    gemm_rowA<TM, 1, TY, KC>(acc, IN + PO, LDI, ag.n_nbr * n_a, P + ag.o_w_fp, NH, WsE, tid);
    const float4 bb = *reinterpret_cast<const float4*>(P + ag.o_b_fp + 4 * tx);
#pragma unroll
    for (int q = 0; q < TM; ++q) {
      const int r = ty + TY * q;
      *reinterpret_cast<float4*>(SH + r * LDS + NH + 4 * tx) =
          make_float4(fmaxf(acc[q][0] + bb.x, 0.f), fmaxf(acc[q][1] + bb.y, 0.f), fmaxf(acc[q][2] + bb.z, 0.f),
                      fmaxf(acc[q][3] + bb.w, 0.f));
    }
  }
  if (VAR != NMARL_IA2C) {
    float acc[TM][4];
#pragma unroll
    for (int q = 0; q < TM; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f; }
    const int Km = (VAR == NMARL_IC3) ? NH : ag.n_nbr * NH;
    gemm_rowA<TM, 1, TY, KC>(acc, IN + MO, LDI, Km, P + ag.o_w_msg, NH, WsE, tid);
    const float4 bb = *reinterpret_cast<const float4*>(P + ag.o_b_msg + 4 * tx);
#pragma unroll
    for (int q = 0; q < TM; ++q) {
      const int r = ty + TY * q;
      float z[4] = {acc[q][0] + bb.x, acc[q][1] + bb.y, acc[q][2] + bb.z, acc[q][3] + bb.w};
      if (VAR == NMARL_NC) {
        *reinterpret_cast<float4*>(SH + r * LDS + 2 * NH + 4 * tx) =
            make_float4(fmaxf(z[0], 0.f), fmaxf(z[1], 0.f), fmaxf(z[2], 0.f), fmaxf(z[3], 0.f));
      } else if (VAR == NMARL_IC3) {                                    // s = tanh(..) + m W_msg + b  (utils.py:400)
        *reinterpret_cast<float4*>(SH + r * LDS + 4 * tx) =
            make_float4(sv[q][0] + z[0], sv[q][1] + z[1], sv[q][2] + z[2], sv[q][3] + z[3]);
      } else {                                                          // DIAL: relu + relu + onehot(argmax p_i)
        float hm[4] = {fmaxf(z[0], 0.f), fmaxf(z[1], 0.f), fmaxf(z[2], 0.f), fmaxf(z[3], 0.f)};
        int am = 0;
        if (r < rows) {
          const float* pr = a.fp + ((size_t)i * B + b0 + r) * n_a;
          float best = pr[0];
          for (int c = 1; c < n_a; ++c) { const float pv = pr[c]; if (pv > best) { best = pv; am = c; } }
        }
        float o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = (sv[q][j] + hm[j]) + ((4 * tx + j) == am ? 1.0f : 0.0f);
        *reinterpret_cast<float4*>(SH + r * LDS + 4 * tx) = make_float4(o[0], o[1], o[2], o[3]);
        if (MODE == MODE_TRAIN && r < rows)
          *reinterpret_cast<float4*>(k.sv_enc + ((size_t)i * B + b0 + r) * 128 + NH + 4 * tx) =
              make_float4(hm[0], hm[1], hm[2], hm[3]);
      }
    }
  }
  __syncthreads();   // SH complete; IN dead from here on (ring WsG aliases it)

  // ---- phase 2: gates  z = [s | h] [wx ; wh] + b,  cell update in registers ------------------
  float acc[TM][16];
#pragma unroll
  for (int q = 0; q < TM; ++q)
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[q][c] = 0.f;
  gemm_rowA<TM, 4, TY, KC>(acc, SH, LDS, SD + NH, P + ag.o_wxh, NG, WsG, tid);
  if (MODE == MODE_TRAIN) {                                             // save [s | h^] for wgrad
    const int q4 = (SD + NH) / 4;
    for (int idx = tid; idx < rows * q4; idx += NT) {
      const int r = idx / q4, c4 = idx - r * q4;
      *reinterpret_cast<float4*>(k.sv_sh + ((size_t)i * B + b0 + r) * (SD + NH) + 4 * c4) =
          *reinterpret_cast<const float4*>(SH + r * LDS + 4 * c4);
    }
  }
  {
    float4 bg[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) bg[g] = *reinterpret_cast<const float4*>(P + ag.o_b + g * NH + 4 * tx);
#pragma unroll
    for (int q = 0; q < TM; ++q) {
      const int r = ty + TY * q;
      float hn[4] = {0.f, 0.f, 0.f, 0.f};
      if (r < rows) {
        const size_t row = (size_t)i * B + b0 + r;
        const float nd = 1.0f - a.done[b0 + r];
        const float4 cp4 = *reinterpret_cast<const float4*>(a.c_in + row * NH + 4 * tx);
        const float cp[4] = {cp4.x * nd, cp4.y * nd, cp4.z * nd, cp4.w * nd};
        float cn[4], gi[4], gf[4], go[4], gu[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          gi[j] = sigmoidf_(acc[q][0 + j] + f4get(bg[0], j));
          gf[j] = sigmoidf_(acc[q][4 + j] + f4get(bg[1], j));
          go[j] = sigmoidf_(acc[q][8 + j] + f4get(bg[2], j));
          gu[j] = tanhf(acc[q][12 + j] + f4get(bg[3], j));
          cn[j] = gf[j] * cp[j] + gi[j] * gu[j];
          hn[j] = go[j] * tanhf(cn[j]);
        }
        if (MODE != MODE_V) {
          *reinterpret_cast<float4*>(a.c_out + row * NH + 4 * tx) = make_float4(cn[0], cn[1], cn[2], cn[3]);
          *reinterpret_cast<float4*>(a.h_out + row * NH + 4 * tx) = make_float4(hn[0], hn[1], hn[2], hn[3]);
        }
        if (MODE == MODE_TRAIN) {
          float* gs = k.sv_gates + row * NG + 4 * tx;
          *reinterpret_cast<float4*>(gs + 0 * NH) = make_float4(gi[0], gi[1], gi[2], gi[3]);
          *reinterpret_cast<float4*>(gs + 1 * NH) = make_float4(gf[0], gf[1], gf[2], gf[3]);
          *reinterpret_cast<float4*>(gs + 2 * NH) = make_float4(go[0], go[1], go[2], go[3]);
          *reinterpret_cast<float4*>(gs + 3 * NH) = make_float4(gu[0], gu[1], gu[2], gu[3]);
        }
      }
      *reinterpret_cast<float4*>(Hs + r * LDH + 4 * tx) = make_float4(hn[0], hn[1], hn[2], hn[3]);
    }
  }
  __syncthreads();

  // ---- phase 3: heads (one thread per env row) ------------------------------------------------
  float l_pol = 0.f, l_val = 0.f, l_ent = 0.f;
  if (tid < rows) {
    const int r = tid, b = b0 + r;
    const size_t row = (size_t)i * B + b;
    float h[NH];
#pragma unroll
    for (int u4 = 0; u4 < NH / 4; ++u4) {
      const float4 t4 = *reinterpret_cast<const float4*>(Hs + r * LDH + 4 * u4);
      h[4 * u4] = t4.x; h[4 * u4 + 1] = t4.y; h[4 * u4 + 2] = t4.z; h[4 * u4 + 3] = t4.w;
    }
    float pi[NMARL_MAX_NA];
    if (MODE != MODE_V) {
      float mx = -3.0e38f;
      for (int c = 0; c < n_a; ++c) {
        float l = 0.f;
#pragma unroll
        for (int u = 0; u < NH; ++u) l = fmaf(h[u], __ldg(P + ag.o_pi_w + u * n_a + c), l);
        l += __ldg(P + ag.o_pi_b + c);
        pi[c] = l;
        mx = fmaxf(mx, l);
      }
      float se = 0.f;
      for (int c = 0; c < n_a; ++c) { pi[c] = expf(pi[c] - mx); se += pi[c]; }
      for (int c = 0; c < n_a; ++c) pi[c] = pi[c] / se;
      if (a.pi != nullptr)
        for (int c = 0; c < n_a; ++c) a.pi[row * n_a + c] = pi[c];
    }
    if (MODE == MODE_P && a.action != nullptr && a.sample_mode != NMARL_SAMPLE_NONE) {
      int act = 0;
      if (a.sample_mode == NMARL_SAMPLE_GREEDY) {                       // np.argmax: first maximum
        float best = pi[0];
        for (int c = 1; c < n_a; ++c) if (pi[c] > best) { best = pi[c]; act = c; }
      } else {                                                          // np.random.choice(p=pi): cdf.searchsorted(u,'right')
        double u;
        if (a.sample_mode == NMARL_SAMPLE_UNIFORM) u = a.uniforms[row];
        else u = philox_u01(a.rng[0], a.rng[1] + a.rng_offset, (uint32_t)row, 0x41435431u);
        double cdf[NMARL_MAX_NA];
        double s = 0.0;
        for (int c = 0; c < n_a; ++c) { s += (double)pi[c]; cdf[c] = s; }
        for (int c = 0; c < n_a; ++c) act += ((cdf[c] / s) <= u) ? 1 : 0;
        act = min(act, n_a - 1);
      }
      a.action[row] = act;
    }
    float v = 0.f;
    if (MODE != MODE_P) {                                               // v = [h, onehot(a_j)] W_v + b  (policies.py:59-77)
#pragma unroll
      for (int u = 0; u < NH; ++u) v = fmaf(h[u], __ldg(P + ag.o_v_w + u), v);
      for (int s = 0; s < ag.n_nbr; ++s) v += __ldg(P + ag.o_v_w + NH + s * n_a + a.act_in[(size_t)ag.nbr[s] * B + b]);
      v += __ldg(P + ag.o_v_b);
      if (a.v != nullptr) a.v[row] = v;
    }
    if (MODE == MODE_TRAIN) {
      const int act = a.act_in[row];
      const float R = k.Rs[row], Adv = k.Advs[row];
      const float cs = k.loss_scale;
      float lp[NMARL_MAX_NA], g[NMARL_MAX_NA];
      float ent = 0.f, dot = 0.f;
      for (int c = 0; c < n_a; ++c) {
        const float pc = fminf(fmaxf(pi[c], 1e-10f), 1.0f);
        const float in_rng = (pi[c] >= 1e-10f && pi[c] <= 1.0f) ? 1.0f : 0.0f;
        lp[c] = logf(pc);
        ent -= pi[c] * lp[c];
        g[c] = k.e_coef * cs * (lp[c] + in_rng);
        if (c == act) g[c] += -cs * Adv * in_rng / pc;
      }
      for (int c = 0; c < n_a; ++c) dot += pi[c] * g[c];
      float* dl = k.sv_dlv + row * 8;
      for (int c = 0; c < 8; ++c) dl[c] = (c < n_a) ? pi[c] * (g[c] - dot) : 0.f;
      dl[n_a] = -k.v_coef * cs * (R - v);
      l_pol = -lp[act] * Adv;
      l_val = (R - v) * (R - v);
      l_ent = ent;
    }
  }
  if (MODE == MODE_TRAIN) {                                             // deterministic per-CTA loss partials
    __shared__ float red[3][32];
    float vals[3] = {l_pol, l_val, l_ent};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float x = vals[c];
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if ((tid & 31) == 0) red[c][tid >> 5] = x;
    }
    __syncthreads();
    if (tid < 3) {
      float s = 0.f;
      for (int w = 0; w < NT / 32; ++w) s += red[tid][w];
      k.loss_part[((size_t)i * k.loss_tiles + blockIdx.x) * 4 + tid] = s;
    }
  }
  if (VAR == NMARL_DIAL && MODE != MODE_V) {                            // sender-side message of the NEW h (utils.py:563-566)
    float macc[TM][4];
#pragma unroll
    for (int q = 0; q < TM; ++q) { macc[q][0] = macc[q][1] = macc[q][2] = macc[q][3] = 0.f; }
    gemm_rowA<TM, 1, TY, KC>(macc, Hs, LDH, NH, P + ag.o_mfc_w, NH, WsE, tid);
    const float4 bb = *reinterpret_cast<const float4*>(P + ag.o_mfc_b + 4 * tx);
#pragma unroll
    for (int q = 0; q < TM; ++q) {
      const int r = ty + TY * q;
      if (r < rows)
        *reinterpret_cast<float4*>(a.msg_out + ((size_t)i * B + b0 + r) * NH + 4 * tx) =
            make_float4(fmaxf(macc[q][0] + bb.x, 0.f), fmaxf(macc[q][1] + bb.y, 0.f), fmaxf(macc[q][2] + bb.z, 0.f),
                        fmaxf(macc[q][3] + bb.w, 0.f));
    }
  }
}

// stand-alone DIAL message kernel (after a reset / state load): msg = relu(h W_mfc + b)
template <int BM, int TY>
__global__ void __launch_bounds__(16 * TY) dial_msg_kernel(const __grid_constant__ nmarl_model m, int B,
                                                          const float* __restrict__ P, const float* __restrict__ h,
                                                          float* __restrict__ msg) {
  constexpr int NT = 16 * TY, TM = BM / TY, KC = 16, LDH = NH + 4;
  __shared__ __align__(16) float Hs[BM * LDH];
  __shared__ __align__(16) float Ws[2 * KC * NH];
  const int i = blockIdx.y, b0 = blockIdx.x * BM, rows = min(BM, B - b0);
  const nmarl_agent& ag = m.agent[i];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  for (int idx = tid; idx < BM * (NH / 4); idx += NT) {
    const int r = idx / (NH / 4), u4 = idx - r * (NH / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows) v = *reinterpret_cast<const float4*>(h + ((size_t)i * B + b0 + r) * NH + 4 * u4);
    *reinterpret_cast<float4*>(Hs + r * LDH + 4 * u4) = v;
  }
  __syncthreads();
  float acc[TM][4];
#pragma unroll
  for (int q = 0; q < TM; ++q) { acc[q][0] = acc[q][1] = acc[q][2] = acc[q][3] = 0.f; }
  gemm_rowA<TM, 1, TY, KC>(acc, Hs, LDH, NH, P + ag.o_mfc_w, NH, Ws, tid);
  const float4 bb = *reinterpret_cast<const float4*>(P + ag.o_mfc_b + 4 * tx);
#pragma unroll
  for (int q = 0; q < TM; ++q) {
    const int r = ty + TY * q;
    if (r < rows)
      *reinterpret_cast<float4*>(msg + ((size_t)i * B + b0 + r) * NH + 4 * tx) =
          make_float4(fmaxf(acc[q][0] + bb.x, 0.f), fmaxf(acc[q][1] + bb.y, 0.f), fmaxf(acc[q][2] + bb.z, 0.f),
                      fmaxf(acc[q][3] + bb.w, 0.f));
  }
}

__global__ void rng_advance_kernel(uint64_t* rng, uint64_t n) {
  if (threadIdx.x == 0 && blockIdx.x == 0) rng[1] += n;
}

constexpr int FWD_BM = 64, FWD_TY = 16;

template <int VAR, int MODE>
int launch_fwd(const nmarl_model* m, const FwdK& k, cudaStream_t st) {
  auto kern = cell_fwd_kernel<VAR, MODE, FWD_BM, FWD_TY>;
  const size_t smem = fwd_smem_floats<FWD_BM, 16>(*m) * sizeof(float);
  NMARL_CHECK(smem <= 227 * 1024, "policy_step: shared memory %zu B exceeds 227 KB", smem);
  static size_t configured = 0;     // per instantiation
  if (smem > configured) {
    NMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  dim3 grid((k.a.B + FWD_BM - 1) / FWD_BM, m->n_agent);
  kern<<<grid, 16 * FWD_TY, smem, st>>>(*m, k);
  NMARL_LAUNCH_CHECK();
  return 0;
}

template <int MODE>
int dispatch_fwd(const nmarl_model* m, const FwdK& k, cudaStream_t st) {
  if (nmarl_tc_fwd_supported(m, &k.a)) return nmarl_tc_launch_fwd(m, k, MODE, st);
  switch (m->variant) {
    case NMARL_IA2C: return launch_fwd<NMARL_IA2C, MODE>(m, k, st);
    case NMARL_NC: return launch_fwd<NMARL_NC, MODE>(m, k, st);
    case NMARL_IC3: return launch_fwd<NMARL_IC3, MODE>(m, k, st);
    case NMARL_DIAL: return launch_fwd<NMARL_DIAL, MODE>(m, k, st);
  }
  nmarl_set_error("unknown variant %d", m->variant);
  return 1;
}

int check_model(const nmarl_model* m) {
  NMARL_CHECK(m != nullptr, "model is NULL");
  NMARL_CHECK(m->n_agent > 0 && m->n_agent <= NMARL_MAX_AGENT, "n_agent %d out of range", m->n_agent);
  NMARL_CHECK(m->n_a > 0 && m->n_a < NMARL_MAX_NA, "n_a %d out of range (max %d)", m->n_a, NMARL_MAX_NA - 1);
  NMARL_CHECK(m->s_dim == ((m->variant == NMARL_NC) ? 3 * NH : NH), "s_dim %d does not match variant", m->s_dim);
  NMARL_CHECK(m->kx_pad % 4 == 0 && m->kp_pad % 4 == 0 && m->km_pad % 4 == 0, "segment pads must be multiples of 4");
  for (int i = 0; i < m->n_agent; ++i) {
    const nmarl_agent& ag = m->agent[i];
    NMARL_CHECK(ag.n_nbr >= 0 && ag.n_nbr <= NMARL_MAX_NBR, "agent %d: n_nbr %d", i, ag.n_nbr);
    NMARL_CHECK(ag.x_nsrc * ag.x_w <= m->kx_pad, "agent %d: obs width exceeds kx_pad", i);
    NMARL_CHECK((m->variant != NMARL_NC && m->variant != NMARL_DIAL) || ag.n_nbr * NH <= m->km_pad,
                "agent %d: message width exceeds km_pad", i);
    NMARL_CHECK(m->variant != NMARL_IC3 || m->km_pad >= NH, "CommNet needs km_pad >= 64");
    NMARL_CHECK(m->variant != NMARL_NC || ag.n_nbr * m->n_a <= m->kp_pad, "agent %d: fingerprint width exceeds kp_pad", i);
    NMARL_CHECK(m->variant != NMARL_IC3 || ag.n_nbr > 0, "agent %d: CommNet needs >= 1 neighbour", i);
  }
  return 0;
}

}  // namespace

int nmarl_check_model(const nmarl_model* m) { return check_model(m); }
int nmarl_fwd_tiles(int B) { return (B + 64 - 1) / 64; }

int nmarl_fwd_tiles(int B);
// entry used by train.cu for the TRAIN-mode forward of one time step
int nmarl_launch_train_fwd(const nmarl_model* m, const nmarl_fwd_args* a, const float* Rs, const float* Advs,
                           float* sv_xin, float* sv_sh, float* sv_gates, float* sv_enc, float* sv_dlv,
                           float* loss_part, float loss_scale, float v_coef, float e_coef, cudaStream_t st) {
  FwdK k{};
  k.a = *a;
  k.Rs = Rs; k.Advs = Advs;
  k.sv_xin = sv_xin; k.sv_sh = sv_sh; k.sv_gates = sv_gates; k.sv_enc = sv_enc; k.sv_dlv = sv_dlv;
  k.loss_part = loss_part; k.loss_tiles = nmarl_fwd_tiles(a->B); k.loss_scale = loss_scale; k.v_coef = v_coef; k.e_coef = e_coef;
  return dispatch_fwd<MODE_TRAIN>(m, k, st);
}



extern "C" int nmarl_policy_step_p(const nmarl_model* m, const nmarl_fwd_args* a, void* stream) {
  if (check_model(m)) return 1;
  NMARL_CHECK(a && a->B > 0 && a->params && a->obs && a->done && a->c_in && a->h_in && a->c_out && a->h_out,
              "policy_step_p: missing buffers");
  NMARL_CHECK(a->c_in != a->c_out && a->h_in != a->h_out, "policy_step_p: state in/out must not alias");
  NMARL_CHECK((m->variant != NMARL_NC && m->variant != NMARL_DIAL) || a->fp, "policy_step_p: fp required");
  NMARL_CHECK(m->variant != NMARL_DIAL || (a->msg_in && a->msg_out), "policy_step_p: DIAL needs msg_in/msg_out");
  NMARL_CHECK(a->sample_mode != NMARL_SAMPLE_UNIFORM || a->uniforms, "policy_step_p: uniforms required");
  NMARL_CHECK(a->sample_mode != NMARL_SAMPLE_PHILOX || a->rng, "policy_step_p: rng state required");
  const int fm = nmarl_state_fm(m, nmarl_tc_fwd_supported(m, a));
  NMARL_CHECK(a->state_fm == fm, "policy_step_p: state_fm must be %d for this variant and path, got %d", fm, a->state_fm);
  FwdK k{};
  k.a = *a;
  if (a->sv_sh != nullptr) {                 // rollout p-call that also saves activations for BPTT
    NMARL_CHECK(nmarl_tc_fwd_supported(m, a), "policy_step_p: activation saving needs the tensor-core path (B %% 128 == 0, wpack)");
    NMARL_CHECK(a->sv_xin && a->sv_gates, "policy_step_p: sv_xin / sv_gates missing");
    NMARL_CHECK((m->variant != NMARL_IC3 && m->variant != NMARL_DIAL) || a->sv_enc, "policy_step_p: sv_enc missing");
    k.sv_xin = a->sv_xin; k.sv_sh = a->sv_sh; k.sv_gates = a->sv_gates; k.sv_enc = a->sv_enc;
    return nmarl_tc_launch_fwd(m, k, MODE_PS, (cudaStream_t)stream);
  }
  return dispatch_fwd<MODE_P>(m, k, (cudaStream_t)stream);
}

extern "C" int nmarl_policy_step_v(const nmarl_model* m, const nmarl_fwd_args* a, void* stream) {
  if (check_model(m)) return 1;
  NMARL_CHECK(a && a->B > 0 && a->params && a->obs && a->done && a->c_in && a->h_in && a->act_in && a->v,
              "policy_step_v: missing buffers");
  NMARL_CHECK((m->variant != NMARL_NC && m->variant != NMARL_DIAL) || a->fp, "policy_step_v: fp required");
  NMARL_CHECK(m->variant != NMARL_DIAL || a->msg_in, "policy_step_v: DIAL needs msg_in");
  const int fm = nmarl_state_fm(m, nmarl_tc_fwd_supported(m, a));
  NMARL_CHECK(a->state_fm == fm, "policy_step_v: state_fm must be %d for this variant and path, got %d", fm, a->state_fm);
  FwdK k{};
  k.a = *a;
  return dispatch_fwd<MODE_V>(m, k, (cudaStream_t)stream);
}

extern "C" int nmarl_dial_msg(const nmarl_model* m, int B, const float* params, const float* h, float* msg, void* stream) {
  if (check_model(m)) return 1;
  NMARL_CHECK(m->variant == NMARL_DIAL, "dial_msg: model is not DIAL");
  dim3 grid((B + 63) / 64, m->n_agent);
  dial_msg_kernel<64, 16><<<grid, 256, 0, (cudaStream_t)stream>>>(*m, B, params, h, msg);
  NMARL_LAUNCH_CHECK();
  return 0;
}

extern "C" int nmarl_rng_advance(uint64_t* rng, uint64_t n, void* stream) {
  rng_advance_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rng, n);
  NMARL_LAUNCH_CHECK();
  return 0;
}
