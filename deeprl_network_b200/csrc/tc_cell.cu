// tc_cell.cu -- tcgen05 (5th-gen tensor core) version of the fused forward cell (K2..K6):
// every GEMM of the step (obs / fingerprint / message encoders and the LSTM gate GEMM) runs as
// 3xTF32 tcgen05.mma with FP32 accumulators in TMEM; CUDA cores only do the elementwise epilogues.
//
// One CTA = 128 envs of one agent (UMMA M = 128).  576 threads:
//   warps 0-15 "row threads": 4 warp-sets x 4 warps; a thread of set s in TMEM-lane quarter w owns env
//              row r = 32 w + lane (TMEM lane r) and the column slice s of it.  They gather the row's
//              inputs, split them hi/lo and tcgen05.st them as the A operand (A lives in TMEM, so no
//              shared memory is spent on activations), read encoder results back with tcgen05.ld, apply
//              bias/activation, feed them to the gate GEMM, and finally run the LSTM cell update, the
//              heads, softmax and sampling for their row.
//   warp 16    B producer: one cp.async.bulk (TMA engine) per 32-wide k-block of pre-packed,
//              128B-swizzled [hi | lo] weight tiles into a 3-stage shared-memory ring (mbarrier tx).
//   warp 17    MMA issuer: a single elected thread issues tcgen05.mma kind::tf32 (3 per k-step:
//              hi*hi + hi*lo + lo*hi) and tcgen05.commit's completion onto the ring barriers.
// TMEM (512 columns): [0,256) accumulators (the encoder GEMMs land in 64-column blocks of it and are consumed
// before the gate GEMM overwrites it), [256,512) A-operand ring (4 slots x (hi 32 | lo 32)).
//
// Same math, same argument block and same outputs as cell_fwd.cu (FP32 FFMA); used when
// B % 128 == 0 and packed weights are supplied.  Restates the same reference lines as cell_fwd.cu.
#include "cell_common.cuh"
#include "tc_row.cuh"

int nmarl_launch_pack_b(const float* W, int ldw, int K, int n0, int nrows, float* out, cudaStream_t st);

namespace {

using namespace tcrow;

template <int VAR, int MODE, bool FM>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_cell_fwd_kernel(const __grid_constant__ nmarl_model m,
                                                                    const __grid_constant__ FwdK k) {
  constexpr bool SAVE = (MODE == MODE_TRAIN || MODE == MODE_PS);   // store activations for BPTT
  constexpr bool SAMPLE = (MODE == MODE_P || MODE == MODE_PS);     // p-call: sample actions
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* bst = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S_STAGES * STAGE_BYTES);
  uint64_t* b_full = bars, *b_empty = bars + S_STAGES, *a_full = bars + 2 * S_STAGES, *a_empty = a_full + A_SLOTS;
  uint64_t* enc_full = a_empty + A_SLOTS, *acc_full = enc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  int* n_kb_s = reinterpret_cast<int*>(tmem_slot + 1);
  KbEnt* sched = reinterpret_cast<KbEnt*>(tmem_slot + 4);
  float* hpart = reinterpret_cast<float*>(sched + MAX_KB);       // [NSET][128][8] head partial sums
  __shared__ float red[3][4];

  const nmarl_fwd_args& a = k.a;
  const int i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  const int B = a.B, b0 = blockIdx.x * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_a = m.n_a, SD = m.s_dim;
  const float* __restrict__ P = a.params;
  const int Kx = ag.x_nsrc * ag.x_w;

  if (tid == 0) {
    for (int s = 0; s < S_STAGES; ++s) { tc::mbar_init(&b_full[s], 1); tc::mbar_init(&b_empty[s], 1); }
    for (int s = 0; s < A_SLOTS; ++s) { tc::mbar_init(&a_full[s], ROW_THREADS); tc::mbar_init(&a_empty[s], 1); }
    tc::mbar_init(enc_full, 1);
    tc::mbar_init(acc_full, 1);
    tc::fence_barrier_init();
    // ---- k-block schedule shared by the three roles: all encoder GEMMs first (each into its own 64-column
    // block of the accumulator region, one completion barrier), then the gate GEMM over [s | h^] ----------------
    int n = 0;
    const int KG = SD + NH, nG = KG / 32;
    sched[n++] = make_kb(ag.tp_x, 64, Kx, 0, ACC_COL, 1, VAR == NMARL_IA2C, 0);          // X (Kx <= 32 on this path)
    if (VAR == NMARL_NC) sched[n++] = make_kb(ag.tp_p, 64, ag.n_nbr * n_a, 0, ACC_COL + 64, 1, 0, 0);
    if (VAR != NMARL_IA2C) {
      const int nM = (VAR == NMARL_IC3) ? 2 : 2 * ag.n_nbr;
      const int KM = (VAR == NMARL_IC3) ? NH : NH * ag.n_nbr;
      const int mcol = (VAR == NMARL_NC) ? ACC_COL + 128 : ACC_COL + 64;
      for (int j = 0; j < nM; ++j) sched[n++] = make_kb(ag.tp_m, 64, KM, j, mcol, j == 0, j == nM - 1, 0);
    }
    for (int g = 0; g < nG; ++g) sched[n++] = make_kb(ag.tp_g, 256, KG, g, ACC_COL, g == 0, 0, g == nG - 1);
    if (VAR == NMARL_DIAL && MODE != MODE_V)
      for (int j = 0; j < 2; ++j) sched[n++] = make_kb(ag.tp_mfc, 64, NH, j, ACC_COL, j == 0, j == 1, 0);
    *n_kb_s = n;
  }
  if (warp == ROW_THREADS / 32 + 1) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const int n_kb = *n_kb_s;
  // PDL: the prologue above overlapped the tail of the previous kernel of the stream; from here on the kernel reads
  // what that kernel (env step / previous cell call) wrote.
  tc::pdl_launch_dependents();
  tc::pdl_wait();

  if (warp < ROW_THREADS / 32) {
    // =================================== row threads ===================================================
    RowCtx c;
    const int set = warp >> 2, quarter = warp & 3, r = quarter * 32 + lane;
    c.tmem = tmem; c.lane_base = (uint32_t)(quarter * 32) << 16;
    c.a_full = a_full; c.a_empty = a_empty; c.enc_full = enc_full; c.q = 0; c.e = 0; c.set = set; c.err = a.tc_err;
    const int b = b0 + r;
    const size_t row = (size_t)i * B + b;
    const float nd = 1.0f - a.done[b];
    const int LDI = m.kx_pad + m.kp_pad + m.km_pad;
    // saved activations are feature-major on this path: [agent][feature][env]
    float* xin_fm = SAVE ? k.sv_xin + (size_t)i * LDI * B : nullptr;
    float* sh_fm = SAVE ? k.sv_sh + (size_t)i * (SD + NH) * B : nullptr;
    float* enc_fm = (SAVE && k.sv_enc) ? k.sv_enc + (size_t)i * 128 * B : nullptr;
    float* gates_fm = SAVE ? k.sv_gates + (size_t)i * NG * B : nullptr;
    long long* prof = (k.prof != nullptr && blockIdx.x == 0 && blockIdx.y == 1 && tid == 0) ? k.prof : nullptr;
    int pi_ = 0;
#define STAMP() do { if (prof) prof[pi_++] = clock64(); } while (0)
    STAMP();
    const int c0 = set * W;             // this thread's columns inside every 32-wide input k-block
    const int e0 = set * EW;            // this thread's hidden units / encoder columns

    // ---- gather every encoder input of this thread up front (all loads in flight together) ------------------
    const int inv_xw = 65536 / ag.x_w + 1, inv_na = 65536 / n_a + 1;    // exact floor(kk / d) for kk < 32, d <= 32
    float xv[W];
#pragma unroll
    for (int j = 0; j < W; ++j) {
      const int kk = c0 + j;
      float val = 0.f;
      if (kk < Kx) {
        const int s = (kk * inv_xw) >> 16, f = kk - s * ag.x_w;     // kk / x_w for kk < 32 without an integer division
        val = a.obs[((size_t)ag.x_src[s] * B + b) * m.obs_stride + f];
      }
      xv[j] = val;
    }
    float pv[W];
    if (VAR == NMARL_NC) {
      const int Kp = ag.n_nbr * n_a;
#pragma unroll
      for (int j = 0; j < W; ++j) {
        const int kk = c0 + j;
        float val = 0.f;
        if (kk < Kp) {
          const int s = (kk * inv_na) >> 16, f = kk - s * n_a;
          val = a.fp[((size_t)ag.nbr[s] * B + b) * n_a + f];
        }
        pv[j] = val;
      }
    }
    constexpr int NPRE = 2;                      // neighbours whose messages are prefetched into registers
    float mv[NPRE][2][W];
    if (VAR == NMARL_NC || VAR == NMARL_DIAL) {
      const float* src = (VAR == NMARL_NC) ? a.h_in : a.msg_in;          // messages: UN-masked (utils.py:182-183)
#pragma unroll
      for (int s = 0; s < NPRE; ++s) {
        if (s < ag.n_nbr) {
#pragma unroll
          for (int hb = 0; hb < 2; ++hb) ld_state<FM, W>(src, (size_t)ag.nbr[s], b, hb * 32 + c0, B, mv[s][hb]);
        }
      }
    }
    if (VAR == NMARL_IC3) {                                               // mean of the neighbours' h (utils.py:395)
      const float nn = (float)ag.n_nbr;
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
        for (int j = 0; j < W; ++j) mv[0][hb][j] = 0.f;
        for (int s = 0; s < ag.n_nbr; ++s) {
          float w8[W];
          ld_state<FM, W>(a.h_in, (size_t)ag.nbr[s], b, hb * 32 + c0, B, w8);
#pragma unroll
          for (int j = 0; j < W; ++j) mv[0][hb][j] += w8[j];
        }
#pragma unroll
        for (int j = 0; j < W; ++j) mv[0][hb][j] /= nn;
      }
    }
    float hv[2][W];                                                       // own h, done-masked (utils.py:189-190)
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
      ld_state<FM, W>(a.h_in, (size_t)i, b, hb * 32 + c0, B, hv[hb]);
#pragma unroll
      for (int j = 0; j < W; ++j) hv[hb][j] *= nd;
    }
    STAMP();
    // ---- encoder GEMMs: A chunks back to back, one completion wait ----------------------------------------------
    const int xm0 = m.kx_pad + m.kp_pad;
    if (SAVE && c0 < m.kx_pad) st_fm<W>(xin_fm, c0, B, b, xv);
    produce_in(c, xv);
    if (VAR == NMARL_NC) {
      if (SAVE && c0 < m.kp_pad) st_fm<W>(xin_fm, m.kx_pad + c0, B, b, pv);
      produce_in(c, pv);
    }
    if (VAR == NMARL_IC3) {
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
        if (SAVE) st_fm<W>(xin_fm, xm0 + hb * 32 + c0, B, b, mv[0][hb]);
        produce_in(c, mv[0][hb]);
      }
    } else if (VAR != NMARL_IA2C) {
      const float* src = (VAR == NMARL_NC) ? a.h_in : a.msg_in;
      for (int s = 0; s < ag.n_nbr; ++s) {
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {
          float t[W];
          if (s < NPRE) {
#pragma unroll
            for (int j = 0; j < W; ++j) t[j] = (s == 0) ? mv[0][hb][j] : mv[NPRE - 1][hb][j];
          } else {
            ld_state<FM, W>(src, (size_t)ag.nbr[s], b, hb * 32 + c0, B, t);
          }
          // NeurComm with feature-major state: m~ is a plain copy of the neighbours' h_seq[t]; the weight-gradient
          // kernel reads it from there (tc_wgrad.cu), so it is not saved a second time
          if (SAVE && !(FM && VAR == NMARL_NC)) st_fm<W>(xin_fm, xm0 + s * NH + hb * 32 + c0, B, b, t);
          produce_in(c, t);
        }
      }
      if (SAVE && !(FM && VAR == NMARL_NC)) {
        float z[W];
#pragma unroll
        for (int j = 0; j < W; ++j) z[j] = 0.f;
        for (int q = ag.n_nbr * 2; q < m.km_pad / 32; ++q) st_fm<W>(xin_fm, xm0 + q * 32 + c0, B, b, z);
      }
    }
    STAMP();
    enc_wait(c);
    STAMP();
    // ---- encoder epilogues -> s, fed to the gate GEMM ---------------------------------------------------------------
    float s0[EW];
    enc_load(c, ACC_COL, s0);
    bias_act(s0, P + ag.o_b_ob + e0, VAR == NMARL_IC3 ? 1 : 0);
    if (SAVE && (VAR == NMARL_IC3 || VAR == NMARL_DIAL)) st_fm<EW>(enc_fm, e0, B, b, s0);
    if (VAR == NMARL_NC) {
      float s1[EW], s2[EW];
      enc_load(c, ACC_COL + 64, s1);
      enc_load(c, ACC_COL + 128, s2);
      bias_act(s1, P + ag.o_b_fp + e0, 0);
      bias_act(s2, P + ag.o_b_msg + e0, 0);
      if (SAVE) { st_fm<EW>(sh_fm, e0, B, b, s0); st_fm<EW>(sh_fm, NH + e0, B, b, s1); st_fm<EW>(sh_fm, 2 * NH + e0, B, b, s2); }
      produce_act(c, s0);
      produce_act(c, s1);
      produce_act(c, s2);
    } else if (VAR == NMARL_IA2C) {
      if (SAVE) st_fm<EW>(sh_fm, e0, B, b, s0);
      produce_act(c, s0);
    } else {
      float s1[EW];
      enc_load(c, ACC_COL + 64, s1);
      if (VAR == NMARL_IC3) {                                            // s = tanh(..) + m W_msg + b  (utils.py:400)
        bias_act(s1, P + ag.o_b_msg + e0, 2);
#pragma unroll
        for (int j = 0; j < EW; ++j) s0[j] += s1[j];
      } else {                                                           // DIAL: relu + relu + onehot(argmax p_i)
        bias_act(s1, P + ag.o_b_msg + e0, 0);
        if (SAVE) st_fm<EW>(enc_fm, NH + e0, B, b, s1);
        int am = 0;
        {
          const float* pr = a.fp + row * n_a;
          float best = pr[0];
          for (int cc = 1; cc < n_a; ++cc) { const float pvv = pr[cc]; if (pvv > best) { best = pvv; am = cc; } }
        }
#pragma unroll
        for (int j = 0; j < EW; ++j) s0[j] = (s0[j] + s1[j]) + ((e0 + j) == am ? 1.0f : 0.0f);
      }
      if (SAVE) st_fm<EW>(sh_fm, e0, B, b, s0);
      produce_act(c, s0);
    }
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
      if (SAVE && !FM) st_fm<W>(sh_fm, SD + hb * 32 + c0, B, b, hv[hb]);   // FM: h^ = (1 - done) * h_seq[t], re-derived by tc_wgrad
      produce_in(c, hv[hb]);
    }
    STAMP();
    // ---- LSTM cell update for hidden units [e0, e0 + EW), 8 at a time; partial head sums -----------------------
    tc::mbar_wait(acc_full, 0, a.tc_err, 13);
    tc::fence_after_sync();
    STAMP();
    float logit[NMARL_MAX_NA];
#pragma unroll
    for (int cc = 0; cc < NMARL_MAX_NA; ++cc) logit[cc] = 0.f;
    float v = 0.f;
#pragma unroll 1
    for (int u0 = e0; u0 < e0 + EW; u0 += 8) {
      float gi[8], gf[8], go[8], gu[8];
      tc::tmem_ld8(tmem + c.lane_base + ACC_COL + 0 * NH + u0, gi);
      tc::tmem_ld8(tmem + c.lane_base + ACC_COL + 1 * NH + u0, gf);
      tc::tmem_ld8(tmem + c.lane_base + ACC_COL + 2 * NH + u0, go);
      tc::tmem_ld8(tmem + c.lane_base + ACC_COL + 3 * NH + u0, gu);
      tc::wait_ld();
      STAMP();
      float cn[8], hn[8], cpv[8];
      ld_state<FM, 8>(a.c_in, (size_t)i, b, u0, B, cpv);
      // MUFU budget: the SFU (16 lanes/clk/SM) bounds this loop, so reciprocals are shared pairwise:
      // 1/(1+a), 1/(1+b) from ONE rcp of (1+a)(1+b)  ->  5 ex2 + 2.5 rcp per hidden unit instead of 5 + 5
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const float4 bi = __ldg(reinterpret_cast<const float4*>(P + ag.o_b + 0 * NH + u0) + q);
        const float4 bf = __ldg(reinterpret_cast<const float4*>(P + ag.o_b + 1 * NH + u0) + q);
        const float4 bo = __ldg(reinterpret_cast<const float4*>(P + ag.o_b + 2 * NH + u0) + q);
        const float4 bu = __ldg(reinterpret_cast<const float4*>(P + ag.o_b + 3 * NH + u0) + q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int x = 4 * q + j;
          const float di = 1.0f + __expf(fminf(-(gi[x] + f4get(bi, j)), 40.0f));
          const float df = 1.0f + __expf(fminf(-(gf[x] + f4get(bf, j)), 40.0f));
          const float dO = 1.0f + __expf(fminf(-(go[x] + f4get(bo, j)), 40.0f));
          const float du = 1.0f + __expf(fminf(-2.0f * (gu[x] + f4get(bu, j)), 40.0f));
          const float r1 = frcp_(di * df), r2 = frcp_(dO * du);
          gi[x] = r1 * df;                          // sigmoid(i)
          gf[x] = r1 * di;                          // sigmoid(f)
          go[x] = r2 * du;                          // sigmoid(o)
          gu[x] = fmaf(2.0f, r2 * dO, -1.0f);       // tanh(u)
          cn[x] = gf[x] * (cpv[x] * nd) + gi[x] * gu[x];
        }
      }
#pragma unroll
      for (int x = 0; x < 8; x += 2) {              // tanh(c) for two units from one reciprocal
        const float d0 = 1.0f + __expf(fminf(-2.0f * cn[x], 40.0f)), d1 = 1.0f + __expf(fminf(-2.0f * cn[x + 1], 40.0f));
        const float r = frcp_(d0 * d1);
        hn[x] = go[x] * fmaf(2.0f, r * d1, -1.0f);
        hn[x + 1] = go[x + 1] * fmaf(2.0f, r * d0, -1.0f);
      }
      STAMP();
      if (MODE != MODE_V) {
        st_state<FM, 8>(a.c_out, (size_t)i, b, u0, B, cn);
        st_state<FM, 8>(a.h_out, (size_t)i, b, u0, B, hn);
      }
      if (SAVE) {
        st_fm<8>(gates_fm, 0 * NH + u0, B, b, gi); st_fm<8>(gates_fm, 1 * NH + u0, B, b, gf);
        st_fm<8>(gates_fm, 2 * NH + u0, B, b, go); st_fm<8>(gates_fm, 3 * NH + u0, B, b, gu);
      }
      STAMP();
      if (MODE != MODE_V) {
        if (n_a == 4) {
#pragma unroll
          for (int x = 0; x < 8; ++x) {
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(P + ag.o_pi_w) + u0 + x);
            logit[0] = fmaf(hn[x], w4.x, logit[0]); logit[1] = fmaf(hn[x], w4.y, logit[1]);
            logit[2] = fmaf(hn[x], w4.z, logit[2]); logit[3] = fmaf(hn[x], w4.w, logit[3]);
          }
        } else {
#pragma unroll
          for (int x = 0; x < 8; ++x)
#pragma unroll
            for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
              if (cc < n_a) logit[cc] = fmaf(hn[x], __ldg(P + ag.o_pi_w + (u0 + x) * n_a + cc), logit[cc]);
        }
      }
      if (!SAMPLE) {
        const float4 v0 = __ldg(reinterpret_cast<const float4*>(P + ag.o_v_w + u0)), v1 = __ldg(reinterpret_cast<const float4*>(P + ag.o_v_w + u0) + 1);
        v = fmaf(hn[0], v0.x, v); v = fmaf(hn[1], v0.y, v); v = fmaf(hn[2], v0.z, v); v = fmaf(hn[3], v0.w, v);
        v = fmaf(hn[4], v1.x, v); v = fmaf(hn[5], v1.y, v); v = fmaf(hn[6], v1.z, v); v = fmaf(hn[7], v1.w, v);
      }
      STAMP();
      if (VAR == NMARL_DIAL && MODE != MODE_V) {          // stash h' for the sender-side message fc below
#pragma unroll
        for (int x = 0; x < 8; ++x) s0[(u0 - e0) + x] = hn[x];
      }
    }
    tc::fence_before_sync();
    if (VAR == NMARL_DIAL && MODE != MODE_V) produce_act(c, s0);

    // ---- heads: combine the NSET partial sums of a row in fixed order, then softmax / sampling / loss -------
    {
      float* hp = hpart + ((size_t)set * 128 + r) * 8;
#pragma unroll
      for (int cc = 0; cc < NMARL_MAX_NA - 1; ++cc) hp[cc] = logit[cc];
      hp[NMARL_MAX_NA - 1] = v;
    }
    STAMP();
    row_barrier();
    STAMP();
    float l_pol = 0.f, l_val = 0.f, l_ent = 0.f;
    if (set == 0) {
#pragma unroll
      for (int cc = 0; cc < NMARL_MAX_NA; ++cc) logit[cc] = 0.f;
      v = 0.f;
#pragma unroll
      for (int s = 0; s < NSET; ++s) {
        const float* hp = hpart + ((size_t)s * 128 + r) * 8;
#pragma unroll
        for (int cc = 0; cc < NMARL_MAX_NA - 1; ++cc) logit[cc] += hp[cc];
        v += hp[NMARL_MAX_NA - 1];
      }
      float pi[NMARL_MAX_NA];
      if (MODE != MODE_V) {
        float mx = -3.0e38f;
#pragma unroll
        for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
          if (cc < n_a) { logit[cc] += __ldg(P + ag.o_pi_b + cc); mx = fmaxf(mx, logit[cc]); }
        float se = 0.f;
#pragma unroll
        for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
          if (cc < n_a) { pi[cc] = expf(logit[cc] - mx); se += pi[cc]; } else pi[cc] = 0.f;
#pragma unroll
        for (int cc = 0; cc < NMARL_MAX_NA; ++cc)
          if (cc < n_a) { pi[cc] = pi[cc] / se; if (a.pi != nullptr) a.pi[row * n_a + cc] = pi[cc]; }
      }
      if (SAMPLE && a.action != nullptr && a.sample_mode != NMARL_SAMPLE_NONE) {
        int act = 0;
        if (a.sample_mode == NMARL_SAMPLE_GREEDY) {
          float best = pi[0];
#pragma unroll
          for (int cc = 1; cc < NMARL_MAX_NA; ++cc) if (cc < n_a && pi[cc] > best) { best = pi[cc]; act = cc; }
        } else {
          double u;
          if (a.sample_mode == NMARL_SAMPLE_UNIFORM) u = a.uniforms[row];
          else u = philox_u01(a.rng[0], a.rng[1] + a.rng_offset, (uint32_t)row, 0x41435431u);
          double cdf[NMARL_MAX_NA];
          double s = 0.0;
#pragma unroll
          for (int cc = 0; cc < NMARL_MAX_NA; ++cc) { if (cc < n_a) s += (double)pi[cc]; cdf[cc] = s; }
          if (a.sample_mode == NMARL_SAMPLE_UNIFORM) {
            // host-supplied uniforms: np.random.choice's rule verbatim (cdf /= cdf[-1]; searchsorted(cdf, u, 'right'))
#pragma unroll
            for (int cc = 0; cc < NMARL_MAX_NA; ++cc) if (cc < n_a) act += ((cdf[cc] / s) <= u) ? 1 : 0;
          } else {
            // device Philox stream (no NumPy stream to reproduce): the same inverse-cdf draw without the four fp64
            // divisions -- they are the longest dependent chain of the kernel's tail
            const double us = u * s;
#pragma unroll
            for (int cc = 0; cc < NMARL_MAX_NA; ++cc) if (cc < n_a) act += (cdf[cc] <= us) ? 1 : 0;
          }
          act = min(act, n_a - 1);
        }
        a.action[row] = act;
      }
      if (!SAMPLE) {
        for (int s = 0; s < ag.n_nbr; ++s) v += __ldg(P + ag.o_v_w + NH + s * n_a + a.act_in[(size_t)ag.nbr[s] * B + b]);
        v += __ldg(P + ag.o_v_b);
        if (a.v != nullptr) a.v[row] = v;
      }
      if (MODE == MODE_TRAIN) {
        const int act = a.act_in[row];
        const float R = k.Rs[row], Adv = k.Advs[row];
        const float cs = k.loss_scale;
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
    }
    if (VAR == NMARL_DIAL && MODE != MODE_V) {            // msg' = relu(h' W_mfc + b)   (utils.py:563-566)
      float mo[EW];
      enc_wait(c);
      enc_load(c, ACC_COL, mo);
      bias_act(mo, P + ag.o_mfc_b + e0, 0);
      st_state<FM, EW>(a.msg_out, (size_t)i, b, e0, B, mo);
    }
    STAMP();
    if (prof) prof[31] = pi_;
    if (MODE == MODE_TRAIN && set == 0) {
      float vals[3] = {l_pol, l_val, l_ent};
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) {
        float x = vals[cc];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) red[cc][quarter] = x;
      }
    }
  } else if (warp == ROW_THREADS / 32) {
    // =================================== B producer ======================================================
    if (tc::elect_one()) producer_loop(sched, n_kb, bst, b_full, b_empty, a.wpack, a.tc_err);
  } else {
    // =================================== MMA issuer ======================================================
    if (tc::elect_one()) mma_loop(sched, n_kb, bst, b_full, b_empty, a_full, a_empty, enc_full, acc_full, tmem, a.tc_err,
                            (k.prof != nullptr && blockIdx.x == 0 && blockIdx.y == 1) ? k.prof : nullptr);
  }
  __syncthreads();
  if (MODE == MODE_TRAIN && tid < 3) {
    const float s = ((red[tid][0] + red[tid][1]) + red[tid][2]) + red[tid][3];
    float* lp = k.loss_part + ((size_t)i * k.loss_tiles + 2 * blockIdx.x) * 4;
    lp[tid] = s;
    lp[4 + tid] = 0.f;                 // the second 64-row slot of this 128-row tile
  }
  if (warp == ROW_THREADS / 32 + 1) { tc::fence_after_sync(); tc::tmem_dealloc(tmem, 512); }
}


// one state layout per variant: feature-major except DIAL, whose message kernels are env-major
template <int VAR, int MODE>
int launch_tc(const nmarl_model* m, const FwdK& k, cudaStream_t st) {
  auto kern = tc_cell_fwd_kernel<VAR, MODE, VAR != NMARL_DIAL>;
  static bool configured = false;
  if (!configured) {
    NMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM));
    configured = true;
  }
  dim3 grid(k.a.B / 128, m->n_agent);
  FwdK k2 = k;
  k2.prof = g_nmarl_prof;
  NMARL_CUDA(nmarl_launch(kern, grid, dim3(TC_THREADS), TC_SMEM, st, true, *m, k2));
  NMARL_LAUNCH_CHECK();
  return 0;
}

template <int VAR>
int launch_tc_mode(const nmarl_model* m, const FwdK& k, int mode, cudaStream_t st) {
  switch (mode) {
    case MODE_P: return launch_tc<VAR, MODE_P>(m, k, st);
    case MODE_V: return launch_tc<VAR, MODE_V>(m, k, st);
    case MODE_PS: return launch_tc<VAR, MODE_PS>(m, k, st);
    default: return launch_tc<VAR, MODE_TRAIN>(m, k, st);
  }
}

}  // namespace

extern "C" int nmarl_tc_supported(const nmarl_model* m, int B) {
  if (B % 128 != 0 || m->kx_pad > 32 || m->kp_pad > 32) return 0;
  for (int i = 0; i < m->n_agent; ++i)
    if (m->agent[i].tp_g < 0 || m->agent[i].tp_x < 0) return 0;
  return 1;
}

bool nmarl_tc_fwd_supported(const nmarl_model* m, const nmarl_fwd_args* a) {
  return a->wpack != nullptr && nmarl_tc_supported(m, a->B);
}

int nmarl_tc_launch_fwd(const nmarl_model* m, const FwdK& k, int mode, cudaStream_t st) {
  switch (m->variant) {
    case NMARL_IA2C: return launch_tc_mode<NMARL_IA2C>(m, k, mode, st);
    case NMARL_NC: return launch_tc_mode<NMARL_NC>(m, k, mode, st);
    case NMARL_IC3: return launch_tc_mode<NMARL_IC3>(m, k, mode, st);
    case NMARL_DIAL: return launch_tc_mode<NMARL_DIAL>(m, k, mode, st);
  }
  nmarl_set_error("unknown variant %d", m->variant);
  return 1;
}

namespace {
__global__ void tc_transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int r = r0 + y, cidx = c0 + threadIdx.x;
    tile[y][threadIdx.x] = (r < rows && cidx < cols) ? src[(size_t)r * cols + cidx] : 0.f;
  }
  __syncthreads();
  for (int y = threadIdx.y; y < 32; y += blockDim.y) {
    const int cidx = c0 + y, r = r0 + threadIdx.x;
    if (r < rows && cidx < cols) dst[(size_t)cidx * rows + r] = tile[threadIdx.x][y];
  }
}
}  // namespace

namespace {
// One launch packs every tensor-core operand of every agent: per 32-deep k-block a [hi | lo] pair of 128B-swizzled
// K-major tiles (see tc.cuh).  Job j of agent i (blockIdx.y = i * PACK_JOBS + j) is one matrix; the backward
// operands (transposed weights) are gathered straight from the parameters with transposed indexing, so no
// transposed copy is needed on this path.
enum { PJ_X = 0, PJ_P, PJ_M, PJ_G, PJ_GT, PJ_MT, PJ_MFC, PJ_MFCT, PACK_JOBS };
struct PackJob { int src, ld, K, N, transposed, dst; };     // operand element (k, n) = transposed ? W[n * ld + k] : W[k * ld + n]

__device__ __forceinline__ PackJob pack_job(const nmarl_model& m, int i, int j) {
  const nmarl_agent& ag = m.agent[i];
  const int SD = m.s_dim, Kx = ag.x_nsrc * ag.x_w;
  const int Km = (m.variant == NMARL_IC3) ? NH : ag.n_nbr * NH;
  PackJob p{0, 0, 0, 0, 0, -1};
  switch (j) {
    case PJ_X: p = PackJob{ag.o_w_ob, NH, Kx, NH, 0, ag.tp_x}; break;
    case PJ_P: if (m.variant == NMARL_NC) p = PackJob{ag.o_w_fp, NH, ag.n_nbr * m.n_a, NH, 0, ag.tp_p}; break;
    case PJ_M: if (m.variant != NMARL_IA2C && Km > 0) p = PackJob{ag.o_w_msg, NH, Km, NH, 0, ag.tp_m}; break;
    case PJ_G: p = PackJob{ag.o_wxh, NG, SD + NH, NG, 0, ag.tp_g}; break;
    case PJ_GT: p = PackJob{ag.o_wxh, NG, NG, SD + NH, 1, ag.tp_gT}; break;
    case PJ_MT: if (m.variant != NMARL_IA2C && Km > 0) p = PackJob{ag.o_w_msg, NH, NH, Km, 1, ag.tp_mT}; break;
    case PJ_MFC: if (m.variant == NMARL_DIAL) p = PackJob{ag.o_mfc_w, NH, NH, NH, 0, ag.tp_mfc}; break;
    case PJ_MFCT: if (m.variant == NMARL_DIAL) p = PackJob{ag.o_mfc_w, NH, NH, NH, 1, ag.tp_mfcT}; break;
  }
  return p;
}

__global__ void __launch_bounds__(256) pack_all_kernel(const __grid_constant__ nmarl_model m, const float* __restrict__ params,
                                                       float* __restrict__ wpack) {
  const int i = blockIdx.y / PACK_JOBS, j = blockIdx.y % PACK_JOBS;
  const PackJob p = pack_job(m, i, j);
  if (p.dst < 0 || p.K <= 0 || p.N <= 0) return;
  const float* W = params + p.src;
  const int nkb = (p.K + 31) / 32;
  const int total = nkb * p.N * 32;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    int n, kk, kb;
    if (p.transposed) { kk = idx & 31; n = (idx >> 5) % p.N; kb = idx / (32 * p.N); }      // consecutive threads -> consecutive k
    else { n = idx % p.N; kk = (idx / p.N) & 31; kb = idx / (p.N * 32); }                  // consecutive threads -> consecutive n
    const int k = kb * 32 + kk;
    float x = 0.f;
    if (k < p.K) x = p.transposed ? W[(size_t)n * p.ld + k] : W[(size_t)k * p.ld + n];
    float hi, lo;
    tc::split_tf32(x, hi, lo);
    char* tile = reinterpret_cast<char*>(wpack + p.dst) + (size_t)kb * 2 * p.N * 128;
    const uint32_t off = tc::sw128_offset((uint32_t)n, (uint32_t)kk);
    *reinterpret_cast<float*>(tile + off) = hi;
    *reinterpret_cast<float*>(tile + (size_t)p.N * 128 + off) = lo;
  }
}
}  // namespace

extern "C" int nmarl_pack_weights(const nmarl_model* m, const float* params, float* wt, float* wpack, void* stream) {
  NMARL_CHECK(m && params && wt && wpack, "pack_weights: missing buffers");
  cudaStream_t st = (cudaStream_t)stream;
  pack_all_kernel<<<dim3(16, m->n_agent * PACK_JOBS), 256, 0, st>>>(*m, params, wpack);
  NMARL_LAUNCH_CHECK();
  if (m->variant == NMARL_DIAL) {          // DIAL's message-gradient kernel reads the plain transposed copies
    dim3 blk(32, 8);
    for (int i = 0; i < m->n_agent; ++i) {
      const nmarl_agent& ag = m->agent[i];
      const int Km = ag.n_nbr * NH;
      if (Km > 0) tc_transpose_kernel<<<dim3(2, (Km + 31) / 32), blk, 0, st>>>(params + ag.o_w_msg, wt + ag.t_w_msg, Km, NH);
      tc_transpose_kernel<<<dim3(2, 2), blk, 0, st>>>(params + ag.o_mfc_w, wt + ag.t_mfc, NH, NH);
    }
    NMARL_LAUNCH_CHECK();
  }
  return 0;
}
