// tc_bwd.cu -- tcgen05 version of one reverse BPTT step of the cell (K9): gate derivatives on CUDA
// cores, then the dgrad GEMM  d[s | h^] = dz [wx;wh]^T  and the message-gradient GEMM
// dm = dpre_m W_msg^T  as 3xTF32 tcgen05.mma with the A operand (dz, dpre_m) written straight from
// registers into TMEM and the pre-packed transposed weights bulk-copied into swizzled shared memory.
// Same CTA structure as tc_cell.cu (128 env rows x one agent, 4 warp-sets of row threads + producer +
// MMA issuer); same inputs/outputs as cell_bwd_kernel (train.cu).
#include "bwd_common.cuh"
#include "tc_row.cuh"

namespace {
using namespace tcrow;

// The operand tiles for the weight-gradient GEMMs (dzT, dpT) are stored once as raw fp32; the weight-gradient kernel
// derives the 3xTF32 lo part in shared memory (tc_wgrad.cu).
template <int VAR, bool FM>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_cell_bwd_kernel(const __grid_constant__ nmarl_model m,
                                                                    const __grid_constant__ BwdK k) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* bst = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S_STAGES * STAGE_BYTES);
  uint64_t* b_full = bars, *b_empty = bars + S_STAGES, *a_full = bars + 2 * S_STAGES, *a_empty = a_full + A_SLOTS;
  uint64_t* enc_full = a_empty + A_SLOTS, *acc_full = enc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  int* n_kb_s = reinterpret_cast<int*>(tmem_slot + 1);
  KbEnt* sched = reinterpret_cast<KbEnt*>(tmem_slot + 4);
  float* bsum = reinterpret_cast<float*>(sched + MAX_KB);         // [4 quarters][256] gate-bias partial sums

  const int i = blockIdx.y;
  const nmarl_agent& ag = m.agent[i];
  const int B = k.B, b0 = blockIdx.x * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_a = m.n_a, SD = m.s_dim;
  const float* __restrict__ P = k.params;
  constexpr int NGRP = (VAR == NMARL_NC) ? 4 : 2;
  const int Km = (VAR == NMARL_IC3) ? NH : ag.n_nbr * NH;

  if (tid == 0) {
    for (int s = 0; s < S_STAGES; ++s) { tc::mbar_init(&b_full[s], 1); tc::mbar_init(&b_empty[s], 1); }
    for (int s = 0; s < A_SLOTS; ++s) { tc::mbar_init(&a_full[s], ROW_THREADS); tc::mbar_init(&a_empty[s], 1); }
    tc::mbar_init(enc_full, 1);
    tc::mbar_init(acc_full, 1);
    tc::fence_barrier_init();
    int n = 0;
    // dgrad k-blocks in the order the row threads produce dz: gate o first (its inputs are already in registers from
    // the dc computation), then i and u (which share their two loads), then f
    const int korder[8] = {4, 5, 0, 1, 6, 7, 2, 3};
    for (int q = 0; q < 8; ++q) sched[n++] = make_kb(ag.tp_gT, SD + NH, NG, korder[q], 0, q == 0, 0, q == 7);
    if (VAR != NMARL_IA2C && Km > 0)
      for (int kb = 0; kb < 2; ++kb) sched[n++] = make_kb(ag.tp_mT, Km, NH, kb, 0, kb == 0, 0, kb == 1);
    *n_kb_s = n;
  }
  if (warp == ROW_THREADS / 32 + 1) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const int n_kb = *n_kb_s;
  tc::pdl_launch_dependents();       // PDL (tc.cuh): the prologue overlapped the previous reverse step's tail
  tc::pdl_wait();

  if (warp < ROW_THREADS / 32) {
    RowCtx c;
    const int set = warp >> 2, quarter = warp & 3, r = quarter * 32 + lane;
    c.tmem = tmem; c.lane_base = (uint32_t)(quarter * 32) << 16;
    c.a_full = a_full; c.a_empty = a_empty; c.enc_full = enc_full; c.q = 0; c.e = 0; c.set = set; c.err = k.tc_err;
    const int b = b0 + r;
    const size_t row = (size_t)i * B + b;
    const float nd = 1.0f - k.done_pre[b];
    const int e0 = set * EW;                       // this thread's 16 hidden units
    // saved activations are feature-major on this path ([agent][feature][env])
    const float* gates_fm = k.sv_gates + (size_t)i * NG * B;
    const float* sh_fm = k.sv_sh + (size_t)i * (SD + NH) * B;
    const float* enc_fm = k.sv_enc ? k.sv_enc + (size_t)i * 128 * B : nullptr;

    // ---- total dh and dc for the thread's units --------------------------------------------------------------
    float dh[EW], dct[EW], dzo[EW];
    {
      const float4 d0 = *reinterpret_cast<const float4*>(k.sv_dlv + row * 8);
      const float4 d1 = *reinterpret_cast<const float4*>(k.sv_dlv + row * 8 + 4);
      const float dl[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      float dv = 0.f;
#pragma unroll
      for (int cc = 0; cc < 8; ++cc) if (cc == n_a) dv = dl[cc];
      float4 vw[EW / 4];
#pragma unroll
      for (int q4 = 0; q4 < EW / 4; ++q4) vw[q4] = __ldg(reinterpret_cast<const float4*>(P + ag.o_v_w + e0) + q4);
#pragma unroll
      for (int j = 0; j < EW; ++j) {
        float s = 0.f;
        if (n_a == 4) {                       // one 16-byte (warp-uniform) load per hidden unit instead of four scalar ones
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(P + ag.o_pi_w) + e0 + j);
          s = fmaf(dl[0], w4.x, s); s = fmaf(dl[1], w4.y, s); s = fmaf(dl[2], w4.z, s); s = fmaf(dl[3], w4.w, s);
        } else {
#pragma unroll
          for (int cc = 0; cc < NMARL_MAX_NA - 1; ++cc)
            if (cc < n_a) s = fmaf(dl[cc], __ldg(P + ag.o_pi_w + (e0 + j) * n_a + cc), s);
        }
        dh[j] = fmaf(dv, f4get(vw[j >> 2], j & 3), s);
        dct[j] = 0.f;
      }
      if (k.has_next) {
        float t16[EW];
        ld_state<FM, EW>(k.dh_in, (size_t)i, b, e0, B, t16);
#pragma unroll
        for (int j = 0; j < EW; ++j) dh[j] += t16[j];
        ld_state<FM, EW>(k.dc_in, (size_t)i, b, e0, B, dct);
        if (VAR == NMARL_NC || VAR == NMARL_IC3) {
          for (int s = 0; s < ag.n_recv; ++s) {
            ld_state<FM, EW>(k.dmsg_in, (size_t)ag.recv_agent[s] * NMARL_MAX_NBR + ag.recv_slot[s], b, e0, B, t16);
#pragma unroll
            for (int j = 0; j < EW; ++j) dh[j] += t16[j];
          }
        }
      }
      // dc_t += dh * o * (1 - tanh(c_t)^2)
      float gov[EW], ccv[EW];
      ld_fm<EW>(gates_fm, 2 * NH + e0, B, b, gov);
      ld_state<FM, EW>(k.c_cur, (size_t)i, b, e0, B, ccv);
#pragma unroll
      for (int j = 0; j < EW; ++j) {
        const float tcv = ftanh(ccv[j]);
        dct[j] += dh[j] * gov[j] * (1.0f - tcv * tcv);
        dzo[j] = dh[j] * tcv * gov[j] * (1.0f - gov[j]);          // dz of gate o, produced first below
      }
    }
    // ---- gate derivatives: per gate the bias partial sums, the dz^T operand tile for the weight-gradient GEMM and the
    // two dgrad A k-blocks.  Order o, i, u, f (see the k-block schedule above): every saved gate is loaded once.
    auto emit = [&](const int g, const float (&dz)[EW]) {
      {   // gate-bias gradient = column sums of dz: sum over this warp's 32 rows by recursive halving (16 shuffles per
          // gate instead of a feature-major copy of dz in HBM + a separate column-sum kernel)
        float a[EW];
#pragma unroll
        for (int j = 0; j < EW; ++j) a[j] = dz[j];
#pragma unroll
        for (int half = EW / 2, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
          const bool up = (lane & bit) != 0;
#pragma unroll
          for (int j = 0; j < half; ++j) {
            const float send = up ? a[j] : a[j + half];
            const float keep = up ? a[j + half] : a[j];
            a[j] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
          }
        }
        a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
        const int col = (((lane >> 4) & 1) << 3) | (((lane >> 3) & 1) << 2) | (((lane >> 2) & 1) << 1) | ((lane >> 1) & 1);
        if ((lane & 1) == 0) bsum[quarter * NG + g * NH + e0 + col] = a[0];
      }
      if (k.dzT != nullptr) {                 // dz^T tile for the tensor-core wgrad: K-major over rows, raw fp32
        uint8_t* tile = reinterpret_cast<uint8_t*>(k.dzT) + ((size_t)i * (B / 32) + (b0 / 32) + quarter) * (size_t)(256 * 128);
#pragma unroll
        for (int j = 0; j < EW; ++j) {
          const uint32_t off = tc::sw128_offset((uint32_t)(g * NH + e0 + j), (uint32_t)lane);
          __stcs(reinterpret_cast<float*>(tile + off), dz[j]);                      // read once, by the wgrad kernel
        }
      }
      produce_act(c, dz);                      // the gate's two k-blocks of the 256-deep dgrad contraction
    };
    emit(2, dzo);
    {
      float gi[EW], gu[EW], dz[EW];
      ld_fm<EW>(gates_fm, 0 * NH + e0, B, b, gi);
      ld_fm<EW>(gates_fm, 3 * NH + e0, B, b, gu);
#pragma unroll
      for (int j = 0; j < EW; ++j) dz[j] = dct[j] * gu[j] * gi[j] * (1.0f - gi[j]);
      emit(0, dz);
#pragma unroll
      for (int j = 0; j < EW; ++j) dz[j] = dct[j] * gi[j] * (1.0f - gu[j] * gu[j]);
      emit(3, dz);
    }
    {
      float gf[EW], cpv[EW], dcp[EW], dz[EW];
      ld_fm<EW>(gates_fm, 1 * NH + e0, B, b, gf);
      ld_state<FM, EW>(k.c_prev, (size_t)i, b, e0, B, cpv);
#pragma unroll
      for (int j = 0; j < EW; ++j) {
        dz[j] = dct[j] * (cpv[j] * nd) * gf[j] * (1.0f - gf[j]);
        dcp[j] = dct[j] * gf[j] * nd;
      }
      st_state<FM, EW>(k.dc_out, (size_t)i, b, e0, B, dcp);
      emit(1, dz);
    }

    // per-tile gate-bias partial sums (fixed order over the four row quarters), reduced over (t, tile) afterwards
    row_barrier();
    if (tid < NG) {
      const float sm = ((bsum[tid] + bsum[NG + tid]) + bsum[2 * NG + tid]) + bsum[3 * NG + tid];
      k.sv_dz[((size_t)i * gridDim.x + blockIdx.x) * NG + tid] = sm;
    }
    // ---- dgrad result: d[s | h^] -------------------------------------------------------------------------------
    tc::mbar_wait(acc_full, 0, k.tc_err, 13);
    tc::fence_after_sync();
    float dpm[EW];
#pragma unroll
    for (int j = 0; j < EW; ++j) dpm[j] = 0.f;
    uint8_t* dptile = (k.dpT != nullptr)
        ? reinterpret_cast<uint8_t*>(k.dpT) + ((size_t)i * (B / 32) + (b0 / 32) + quarter) * (size_t)(k.ndp * 128) : nullptr;
    auto put_dp = [&](int n0, const float (&vals)[EW]) {        // encoder pre-activation grads as K-major tiles
      if (dptile == nullptr) return;
#pragma unroll
      for (int j = 0; j < EW; ++j) {
        const uint32_t off = tc::sw128_offset((uint32_t)(n0 + j), (uint32_t)lane);
        __stcs(reinterpret_cast<float*>(dptile + off), vals[j]);
      }
    };
#pragma unroll
    for (int gp = 0; gp < NGRP; ++gp) {
      float d[EW];
#pragma unroll
      for (int p = 0; p < EW / 8; ++p) {
        float t[8];
        tc::tmem_ld8(tmem + c.lane_base + ACC_COL + gp * NH + e0 + 8 * p, t);
        tc::wait_ld();
#pragma unroll
        for (int j = 0; j < 8; ++j) d[8 * p + j] = t[j];
      }
      if (gp == NGRP - 1) {                    // own recurrent gradient, done-masked
#pragma unroll
        for (int j = 0; j < EW; ++j) d[j] *= nd;
        st_state<FM, EW>(k.dh_out, (size_t)i, b, e0, B, d);
      } else if (VAR == NMARL_NC || VAR == NMARL_IA2C) {
        float sv[EW];
        ld_fm<EW>(sh_fm, gp * NH + e0, B, b, sv);
#pragma unroll
        for (int j = 0; j < EW; ++j) d[j] = sv[j] > 0.f ? d[j] : 0.f;
        put_dp(gp * NH + e0, d);
        if (VAR == NMARL_NC && gp == 2) {
#pragma unroll
          for (int j = 0; j < EW; ++j) dpm[j] = d[j];
        }
      } else {                                  // IC3 / DIAL: one 64-wide s
        float hx[EW], hm[EW], o[EW];
        ld_fm<EW>(enc_fm, e0, B, b, hx);
        if (VAR == NMARL_DIAL) ld_fm<EW>(enc_fm, NH + e0, B, b, hm);
#pragma unroll
        for (int j = 0; j < EW; ++j) {
          if (VAR == NMARL_IC3) { o[j] = d[j] * (1.0f - hx[j] * hx[j]); dpm[j] = d[j]; }
          else { o[j] = hx[j] > 0.f ? d[j] : 0.f; dpm[j] = hm[j] > 0.f ? d[j] : 0.f; }
        }
        put_dp(e0, o);
        put_dp(NH + e0, dpm);
      }
    }
    tc::fence_before_sync();
    // ---- message gradient dm = dpre_m W_msg^T, one 64-wide block per neighbour slot --------------------------
    if (VAR != NMARL_IA2C && Km > 0) {
      produce_act(c, dpm);
      tc::mbar_wait(acc_full, 1, k.tc_err, 14);
      tc::fence_after_sync();
      const int nblk = (VAR == NMARL_IC3) ? 1 : ag.n_nbr;
      for (int s = 0; s < nblk; ++s) {
        float d[EW];
#pragma unroll
        for (int p = 0; p < EW / 8; ++p) {
          float t[8];
          tc::tmem_ld8(tmem + c.lane_base + ACC_COL + s * NH + e0 + 8 * p, t);
          tc::wait_ld();
#pragma unroll
          for (int j = 0; j < 8; ++j) d[8 * p + j] = t[j];
        }
        if (VAR == NMARL_IC3) {
          const float nn = (float)ag.n_nbr;
#pragma unroll
          for (int j = 0; j < EW; ++j) d[j] /= nn;
          for (int s2 = 0; s2 < ag.n_nbr; ++s2) st_state<FM, EW>(k.dmsg_out, (size_t)i * NMARL_MAX_NBR + s2, b, e0, B, d);
        } else {
          st_state<FM, EW>(k.dmsg_out, (size_t)i * NMARL_MAX_NBR + s, b, e0, B, d);
        }
      }
      tc::fence_before_sync();
    }
  } else if (warp == ROW_THREADS / 32) {
    if (tc::elect_one()) producer_loop(sched, n_kb, bst, b_full, b_empty, k.wpack, k.tc_err);
  } else {
    if (tc::elect_one()) mma_loop(sched, n_kb, bst, b_full, b_empty, a_full, a_empty, enc_full, acc_full, tmem, k.tc_err);
  }
  __syncthreads();
  if (warp == ROW_THREADS / 32 + 1) { tc::fence_after_sync(); tc::tmem_dealloc(tmem, 512); }
}

// one state layout per variant: feature-major except DIAL, whose message kernels are env-major
template <int VAR>
int launch_tc_bwd(const nmarl_model* m, const BwdK& k, cudaStream_t st) {
  auto kern = tc_cell_bwd_kernel<VAR, VAR != NMARL_DIAL>;
  static bool configured = false;
  if (!configured) {
    NMARL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM));
    configured = true;
  }
  dim3 grid(k.B / 128, m->n_agent);
  NMARL_CUDA(nmarl_launch(kern, grid, dim3(TC_THREADS), TC_SMEM, st, true, *m, k));
  NMARL_LAUNCH_CHECK();
  return 0;
}

}  // namespace

int nmarl_tc_launch_bwd(const nmarl_model* m, const BwdK& k, cudaStream_t st) {
  switch (m->variant) {
    case NMARL_IA2C: return launch_tc_bwd<NMARL_IA2C>(m, k, st);
    case NMARL_NC: return launch_tc_bwd<NMARL_NC>(m, k, st);
    case NMARL_IC3: return launch_tc_bwd<NMARL_IC3>(m, k, st);
    case NMARL_DIAL: return launch_tc_bwd<NMARL_DIAL>(m, k, st);
  }
  nmarl_set_error("unknown variant %d", m->variant);
  return 1;
}
