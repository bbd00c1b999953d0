// tc_wgrad.cu -- tcgen05 weight gradients of every GEMM of the cell (gate matrix and the obs / fingerprint /
// message encoders):   dW[ka][n] = sum over all (t, env) rows r of  A[r][ka] * D[r][n]
// as 3xTF32 GEMMs with M = ka (one 128-lane tile per job), the contraction over rows split across CTAs and a
// fixed-order reduce afterwards.
//   A operand: the saved activations are feature-major ([t][agent][feature][env]); TMEM lane = feature ka, so
//              a thread reads 8 consecutive envs (32 contiguous bytes), splits hi/lo and tcgen05.st's them.
//   B operand: D^T, K-major over rows, was written by the backward cell kernel as raw fp32 128B-swizzled tiles
//              (dz: 256 rows, encoder pre-activation grads: 192/128/64 rows); the producer bulk-copies the needed
//              row range of the tile per 32 env rows, and the 3xTF32 lo part is derived in shared memory.
//   Biases:    the obs-encoder job carries an extra all-ones lane and spans every column of the dpre tile, which
//              yields all encoder bias gradients for free; the gate bias is a coalesced column sum of dz.
#include "bwd_common.cuh"
#include "tc_row.cuh"

extern long long* g_nmarl_prof;          // api.cu: debug hook (nmarl_debug_set_prof)

namespace {
using namespace tcrow;

enum { J_GATE0 = 0, J_GATE1, J_ENC_X, J_ENC_M0, J_ENC_M1, J_COUNT };
// Row-thread roles: warp-sets 0,1 produce the A operand (16 of the 32 columns of a k-block each), warp-sets 2,3 derive
// the `lo` half of the raw B tiles in shared memory; the two dependent chains (global load -> split -> tcgen05.st
// and TMA wait -> lds/sts -> proxy fence) run side by side instead of back to back in every thread.
constexpr int A_SETS = 2, A_THREADS = 128 * A_SETS, WA = 32 / A_SETS;
// Shared-memory rings: WG_STAGES raw 32 KB B tiles (bulk-copied, deep enough to cover the DRAM latency of a 32 KB copy
// at one k-block per ~0.8 us) + WG_LO_BUFS derived `lo` tiles.
constexpr int WG_STAGES = 5, WG_LO_BUFS = 2;
constexpr uint32_t WG_TILE_BYTES = 256 * 128;
constexpr size_t WG_SMEM = (size_t)(WG_STAGES + WG_LO_BUFS) * WG_TILE_BYTES + 1024 + 32 * 8 + 64;
static_assert(WG_SMEM <= 232448, "wgrad ring exceeds the 227 KB of dynamic shared memory");
constexpr int SEG_KB = 20;       // k-blocks (of 32 rows) accumulated in TMEM before the accumulator is drained (see flush)

struct TcWgK {
  int B, T, splits, ndp;
  const float* sv_sh; const float* sv_xin; const float* dzT; const float* dpT;
  const float* h_seq; const float* done_pre;   // feature-major state path: h^ / m~ operand rows come from the state sequence
  float* ws;
  long long ws_off[J_COUNT];     // float offset of each job's partial block [splits][N_agents][128][N_job]
  int jobs[J_COUNT]; int n_jobs; // job kinds present
  int* err;
  long long* prof;               // debug: clock64 stamps of CTA (split 1, job 0, agent 1) or NULL (tools/wg_prof.py)
};

struct JobDesc {
  const float* A; int F_A, a_feat0, ka_cnt, ones;
  int p_feat0, p_cnt;             // obs-encoder job only: fingerprint features ride on the lanes behind the ones lane
  const float* BT; int tile_rows, n_row0, N;
};

__device__ __forceinline__ JobDesc job_desc(const nmarl_model& m, const TcWgK& k, int kind, int i) {
  const nmarl_agent& ag = m.agent[i];
  JobDesc d;
  d.p_feat0 = 0; d.p_cnt = 0;
  const int SD = m.s_dim, LDI = m.kx_pad + m.kp_pad + m.km_pad;
  const int Km = (m.variant == NMARL_IC3) ? NH : ag.n_nbr * NH;
  if (kind == J_GATE0 || kind == J_GATE1) {
    const int mt = kind - J_GATE0;
    d.A = k.sv_sh; d.F_A = SD + NH; d.a_feat0 = 128 * mt; d.ka_cnt = max(0, min(128, SD + NH - 128 * mt)); d.ones = 0;
    d.BT = k.dzT; d.tile_rows = 256; d.n_row0 = 0; d.N = 256;
  } else if (kind == J_ENC_X) {
    d.A = k.sv_xin; d.F_A = LDI; d.a_feat0 = 0; d.ka_cnt = ag.x_nsrc * ag.x_w; d.ones = 1;
    if (m.variant == NMARL_NC) { d.p_feat0 = m.kx_pad; d.p_cnt = ag.n_nbr * m.n_a; }
    d.BT = k.dpT; d.tile_rows = k.ndp; d.n_row0 = 0; d.N = k.ndp;
  } else {
    const int mt = kind - J_ENC_M0;
    d.A = k.sv_xin; d.F_A = LDI; d.a_feat0 = m.kx_pad + m.kp_pad + 128 * mt; d.ka_cnt = max(0, min(128, Km - 128 * mt)); d.ones = 0;
    d.BT = k.dpT; d.tile_rows = k.ndp; d.n_row0 = (m.variant == NMARL_NC) ? 128 : 64; d.N = 64;
  }
  return d;
}

// The D^T tiles hold raw fp32 once.  The producer copies one tile per k-block; it doubles as the hi operand (the TF32
// datapath drops the 13 low mantissa bits -- tools/probe_tf32_operand.py); the row threads derive lo = x - trunc(x)
// into a lo buffer and signal lo_full; the issuer runs the two passes that need only the raw tile first and
// a_hi * b_lo after that barrier.
__global__ void __launch_bounds__(TC_THREADS, 1) tc_wgrad_kernel(const __grid_constant__ nmarl_model m,
                                                                 const __grid_constant__ TcWgK k) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* bst = smem;
  constexpr int NST = WG_STAGES;                                       // B stages
  constexpr uint32_t STB = WG_TILE_BYTES;                              // bytes per B stage
  uint8_t* lobuf = smem + (size_t)NST * STB;                           // WG_LO_BUFS derived lo tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(lobuf + (size_t)WG_LO_BUFS * STB);
  uint64_t* b_full = bars, *b_empty = bars + NST, *a_full = bars + 2 * NST, *a_empty = a_full + A_SLOTS;
  uint64_t* enc_full = a_empty + A_SLOTS, *acc_full = enc_full + 1;
  uint64_t* acc_free = acc_full + 1;                                   // accumulator drained by the row threads (segment flush)
  uint64_t* lo_full = acc_free + 1, *lo_empty = lo_full + WG_LO_BUFS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(lo_empty + WG_LO_BUFS);

  const int sp = blockIdx.x, jslot = blockIdx.y, i = blockIdx.z;
  const int kind = k.jobs[jslot];
  const JobDesc d = job_desc(m, k, kind, i);
  const int N_agents = m.n_agent;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int bpt = k.B / 32;                                           // 32-row k-blocks per time step
  const int kb_total = k.T * bpt;
  const int per = (kb_total + k.splits - 1) / k.splits;
  const int kb0 = sp * per, kb1 = min(kb_total, kb0 + per);
  const int nkb = (d.ka_cnt > 0) ? max(0, kb1 - kb0) : 0;
  float* wsj = k.ws + k.ws_off[jslot] + ((size_t)sp * N_agents + i) * 128 * d.N;

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) { tc::mbar_init(&b_full[s], 1); tc::mbar_init(&b_empty[s], 1); }
    for (int s = 0; s < A_SLOTS; ++s) { tc::mbar_init(&a_full[s], A_THREADS); tc::mbar_init(&a_empty[s], 1); }
    tc::mbar_init(enc_full, 1);
    tc::mbar_init(acc_full, 1);
    tc::mbar_init(acc_free, ROW_THREADS);
    for (int s = 0; s < WG_LO_BUFS; ++s) { tc::mbar_init(&lo_full[s], ROW_THREADS - A_THREADS); tc::mbar_init(&lo_empty[s], 1); }
    tc::fence_barrier_init();
  }
  if (warp == ROW_THREADS / 32 + 1) tc::tmem_alloc(tmem_slot, 512);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tile_bytes = (uint32_t)d.N * 128u;                   // rows of the tile staged per k-block
  // the D^T tile of (t, 32-env block rb)
  auto bt_tile = [&](int t, int rb) -> const uint8_t* {
    const float* tile = d.BT + t * nmarl_tc_tile_step_floats(N_agents, k.B, d.tile_rows) + ((size_t)i * bpt + rb) * d.tile_rows * 32;
    return reinterpret_cast<const uint8_t*>(tile);
  };

  if (warp < ROW_THREADS / 32) {
    RowCtx c;
    const int set = warp >> 2, quarter = warp & 3;
    const int ka = quarter * 32 + lane;                               // TMEM lane == feature within this M tile
    c.tmem = tmem; c.lane_base = (uint32_t)(quarter * 32) << 16;
    c.a_full = a_full; c.a_empty = a_empty; c.enc_full = enc_full; c.q = 0; c.e = 0; c.set = set; c.err = k.err;
    const bool one = d.ones && ka == d.ka_cnt;
    const bool is_p = ka > d.ka_cnt && ka <= d.ka_cnt + d.p_cnt;
    const bool real = ka < d.ka_cnt || is_p;
    const int feat = is_p ? d.p_feat0 + (ka - d.ka_cnt - 1) : d.a_feat0 + ka;
    // Feature-major state path: the forward kernel does not save h^ (= (1 - done) * own h_seq[t]) and, for NeurComm,
    // m~ (= the neighbours' h_seq[t]) a second time; those operand rows are read from the state sequence itself.
    int hs_agent = -1, hs_unit = 0;
    bool hs_mask = false;
    if (k.h_seq != nullptr && real && !is_p) {
      if ((kind == J_GATE0 || kind == J_GATE1) && feat >= m.s_dim) { hs_agent = i; hs_unit = feat - m.s_dim; hs_mask = true; }
      else if ((kind == J_ENC_M0 || kind == J_ENC_M1) && m.variant == NMARL_NC) {
        const int fm = feat - (m.kx_pad + m.kp_pad);
        hs_agent = m.agent[i].nbr[fm / NH]; hs_unit = fm % NH;
      }
    }
    // the A operand of k-block q: 8 consecutive envs of this thread's feature (global loads; issued one k-block AHEAD so
    // that their latency hides behind the lo pass / the barrier waits of the current k-block)
    auto load_x = [&](int q, float (&x)[WA]) {
      const int kb = kb0 + q, t = kb / bpt, rb = kb - t * bpt;
      if (hs_agent >= 0) {
        const float* src = k.h_seq + (((size_t)t * N_agents + hs_agent) * NH + hs_unit) * k.B + rb * 32 + set * WA;
#pragma unroll
        for (int p = 0; p < WA / 4; ++p) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(src + 4 * p));
          x[4 * p] = v.x; x[4 * p + 1] = v.y; x[4 * p + 2] = v.z; x[4 * p + 3] = v.w;
        }
        if (hs_mask) {
          const float* dn = k.done_pre + (size_t)t * k.B + rb * 32 + set * WA;
#pragma unroll
          for (int p = 0; p < WA / 4; ++p) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(dn + 4 * p));
            x[4 * p] *= 1.0f - v.x; x[4 * p + 1] *= 1.0f - v.y; x[4 * p + 2] *= 1.0f - v.z; x[4 * p + 3] *= 1.0f - v.w;
          }
        }
      } else if (real) {
        const float* src = d.A + (((size_t)t * N_agents + i) * d.F_A + feat) * k.B + rb * 32 + set * WA;
#pragma unroll
        for (int p = 0; p < WA / 4; ++p) {
          const float4 v = __ldcs(reinterpret_cast<const float4*>(src + 4 * p));
          x[4 * p] = v.x; x[4 * p + 1] = v.y; x[4 * p + 2] = v.z; x[4 * p + 3] = v.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < WA; ++j) x[j] = one ? 1.0f : 0.0f;
      }
    };
    // Segmented accumulation.  The tensor core adds every MMA into the fp32 accumulator with round-toward-zero: a bias
    // of ~2^-24 of the running sum per MMA that grows linearly with the chain length (measured 1.4e-4 of max|g| after
    // the 2 496 MMAs of one B = 4096, T = 60 split).  The accumulator is therefore drained every SEG_KB k-blocks
    // (240 MMAs at SEG_KB = 20) and the segment sums are added up in the CTA's own workspace slot with ordinary
    // round-to-nearest fp32 adds.
    const bool warp_active = quarter * 32 < d.ka_cnt + (d.ones ? 1 : 0) + d.p_cnt;   // tcgen05.ld is warp-collective
    float* out = wsj + ka;                                      // element (ka, n) of the partial block at out[n * 128]
    // The previous partial sums are fetched BEFORE the wait for the segment's last MMAs (the loads do not depend on
    // them) in two batches of four 8-column pieces, so that one L2 round trip, not eight, is exposed per drain.
    long long* prof = (k.prof != nullptr && sp == 1 && jslot == 0 && i == 1 && (tid == 0 || tid == A_THREADS)) ? k.prof + (tid ? 128 : 192) : nullptr;
    auto flush = [&](int seg) {
      if (prof && seg < 5) prof[3 * seg] = clock64();
      const bool mine = warp_active && (real || one);
      const bool rmw = mine && seg > 0;
      tc::mbar_wait(acc_full, seg & 1, k.err, 13);
      tc::fence_after_sync();
      if (prof && seg < 5) prof[3 * seg + 1] = clock64();
      // workspace block layout [column n][lane ka]: for a fixed column the 32 lanes of a warp are 128 contiguous bytes
#pragma unroll 2
      for (int c0 = set * 8; c0 < d.N; c0 += 8 * NSET) {
        if (warp_active) {                                         // warp-uniform: tcgen05.ld is warp-collective
          float pv[8];
          if (rmw) {
#pragma unroll
            for (int j = 0; j < 8; ++j) pv[j] = out[(size_t)(c0 + j) * 128];
          }
          float v[8];
          tc::tmem_ld8(tmem + c.lane_base + ACC_COL + c0, v);
          tc::wait_ld();
          if (mine) {
#pragma unroll
            for (int j = 0; j < 8; ++j) out[(size_t)(c0 + j) * 128] = rmw ? v[j] + pv[j] : v[j];
          }
        }
      }
      tc::fence_before_sync();
      if (prof && seg < 5) prof[3 * seg + 2] = clock64();
      tc::mbar_arrive(acc_free);
    };
    if (set < A_SETS) {
      // ---- A producers: columns [set * WA, set * WA + WA) of every k-block, loads issued one k-block ahead ------------
      float xa[WA], xb[WA];                     // the operands of the next two k-blocks (two loads in flight per thread)
      auto emit_a = [&](int q, float (&x)[WA]) {
        produce_begin(c);
#pragma unroll
        for (int p = 0; p < WA / 8; ++p) {
          float t8[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) t8[j] = x[8 * p + j];
          produce_piece(c, set * WA + 8 * p, t8);
        }
        produce_end(c);
        if (q + 2 < nkb) load_x(q + 2, x);        // refill this buffer; it is consumed two k-blocks from now
        if ((q + 1) % SEG_KB == 0 || q + 1 == nkb) flush(q / SEG_KB);
      };
      if (nkb > 0) load_x(0, xa);
      if (nkb > 1) load_x(1, xb);
      for (int q = 0; q < nkb; q += 2) {
        emit_a(q, xa);
        if (q + 1 < nkb) emit_a(q + 1, xb);
      }
    } else {
      // ---- lo derivation: lo = rn_tf32(x - trunc_tf32(x)) of the k-block's B stage -----------------------------------
      const int lt = tid - A_THREADS;
      for (int q = 0; q < nkb; ++q) {
        const int st = q % NST, lb = q % WG_LO_BUFS;
        tc::mbar_wait(&lo_empty[lb], ((q / WG_LO_BUFS) & 1) ^ 1, k.err, 42);      // the MMAs that read this lo buffer are done
        tc::mbar_wait(&b_full[st], (q / NST) & 1, k.err, 41);
        const float4* raw = reinterpret_cast<const float4*>(bst + (size_t)st * STB);
        float4* lo = reinterpret_cast<float4*>(lobuf + (size_t)lb * STB);
        for (uint32_t e = (uint32_t)lt; e < tile_bytes / 16; e += ROW_THREADS - A_THREADS) {
          const float4 v = raw[e];
          float4 l;
          l.x = tc::tf32_lo_of_raw(v.x); l.y = tc::tf32_lo_of_raw(v.y);
          l.z = tc::tf32_lo_of_raw(v.z); l.w = tc::tf32_lo_of_raw(v.w);
          lo[e] = l;
        }
        tc::fence_proxy_async();
        tc::mbar_arrive(&lo_full[lb]);
        if ((q + 1) % SEG_KB == 0 || q + 1 == nkb) flush(q / SEG_KB);
      }
    }
    if (nkb == 0 && warp_active && (real || one)) {
      for (int c0 = set * 8; c0 < d.N; c0 += 8 * NSET)
        for (int j = 0; j < 8; ++j) out[(size_t)(c0 + j) * 128] = 0.f;
    }
  } else if (warp == ROW_THREADS / 32) {
    if (tc::elect_one()) {
      for (int q = 0; q < nkb; ++q) {
        const int kb = kb0 + q, st = q % NST;
        const int t = kb / bpt, rb = kb - t * bpt;
        tc::mbar_wait(&b_empty[st], ((q / NST) & 1) ^ 1, k.err, 21);
        const uint8_t* tile = bt_tile(t, rb);
        tc::mbar_arrive_expect_tx(&b_full[st], tile_bytes);
        tc::bulk_g2s(bst + (size_t)st * STB, tile + (size_t)d.n_row0 * 128, tile_bytes, &b_full[st]);
      }
    }
  } else {
    if (tc::elect_one()) {
      const uint32_t idesc = tc::idesc_tf32(128, (uint32_t)d.N);
      long long* iprof = (k.prof != nullptr && sp == 1 && jslot == 0 && i == 1) ? k.prof : nullptr;
      for (int q = 0; q < nkb; ++q) {
        const int st = q % NST, slot = q & (A_SLOTS - 1), lb = q % WG_LO_BUFS;
        if (iprof && q < 40) iprof[3 * q] = clock64();
        const int seg = q / SEG_KB;
        const bool seg_first = (q % SEG_KB) == 0;
        if (seg_first && seg > 0) tc::mbar_wait(acc_free, (seg - 1) & 1, k.err, 34);   // previous segment drained
        tc::mbar_wait(&b_full[st], (q / NST) & 1, k.err, 31);
        tc::mbar_wait(&a_full[slot], (q / A_SLOTS) & 1, k.err, 32);
        tc::fence_after_sync();
        const uint64_t d_hi = tc::smem_desc_sw128(bst + (size_t)st * STB);
        const uint64_t d_lo = tc::smem_desc_sw128(lobuf + (size_t)lb * STB);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {                                // passes that need only the raw tile
          const uint32_t a_hi = tmem + A_COL + slot * 64 + ks * 8, a_lo = a_hi + 32;
          tc::mma_tf32_ts(tmem + ACC_COL, a_hi, d_hi + 2 * ks, idesc, (seg_first && ks == 0) ? 0u : 1u);
          tc::mma_tf32_ts(tmem + ACC_COL, a_lo, d_hi + 2 * ks, idesc, 1u);
        }
        if (iprof && q < 40) iprof[3 * q + 1] = clock64();
        tc::mbar_wait(&lo_full[lb], (q / WG_LO_BUFS) & 1, k.err, 33);
        tc::fence_after_sync();
        if (iprof && q < 40) iprof[3 * q + 2] = clock64();
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          tc::mma_tf32_ts(tmem + ACC_COL, tmem + A_COL + slot * 64 + ks * 8, d_lo + 2 * ks, idesc, 1u);
        tc::mma_commit(&a_empty[slot]);
        tc::mma_commit(&b_empty[st]);
        tc::mma_commit(&lo_empty[lb]);
        if ((q + 1) % SEG_KB == 0 || q + 1 == nkb) tc::mma_commit(acc_full);
      }
    }
  }
  __syncthreads();
  if (warp == ROW_THREADS / 32 + 1) { tc::fence_after_sync(); tc::tmem_dealloc(tmem, 512); }
}

// fixed-order reduce over the row splits + scatter into the flat gradient buffer
__global__ void __launch_bounds__(256) tc_wgrad_reduce_kernel(const __grid_constant__ nmarl_model m, const __grid_constant__ TcWgK k,
                                                             float* __restrict__ grads) {
  const int jslot = blockIdx.y, i = blockIdx.z, kind = k.jobs[jslot];
  const JobDesc d = job_desc(m, k, kind, i);
  const nmarl_agent& ag = m.agent[i];
  const int lanes = d.ka_cnt + (d.ones ? 1 : 0) + d.p_cnt;
  const int total = 128 * d.N;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int ln = e & 127, n = e >> 7;                      // partial blocks are [column n][lane]: coalesced over lanes
    if (ln >= lanes) continue;
    float s = 0.f;
    for (int sp = 0; sp < k.splits; ++sp) s += k.ws[k.ws_off[jslot] + (((size_t)sp * m.n_agent + i) * d.N + n) * 128 + ln];
    if (kind == J_GATE0 || kind == J_GATE1) grads[ag.o_wxh + (size_t)(128 * (kind - J_GATE0) + ln) * NG + n] = s;
    else if (kind == J_ENC_X) {
      if (ln < d.ka_cnt) { if (n < NH) grads[ag.o_w_ob + ln * NH + n] = s; }
      else if (ln > d.ka_cnt) { if (n >= NH && n < 2 * NH) grads[ag.o_w_fp + (ln - d.ka_cnt - 1) * NH + n - NH] = s; }   // fingerprint lanes
      else if (n < NH) grads[ag.o_b_ob + n] = s;                                       // ones lane: biases
      else if (m.variant == NMARL_NC && n < 2 * NH) grads[ag.o_b_fp + n - NH] = s;
      else grads[ag.o_b_msg + n - ((m.variant == NMARL_NC) ? 2 * NH : NH)] = s;
    } else grads[ag.o_w_msg + (size_t)(128 * (kind - J_ENC_M0) + ln) * NH + n] = s;
  }
}

// gate bias gradient: fixed-order reduce of the per-tile partial sums the backward cell kernel left in sv_dz
// ([t][agent][tile][256]); one CTA per (32 columns, agent), 8 strided partial chains per column + an ordered tail
__global__ void __launch_bounds__(256) gate_bias_reduce_kernel(const __grid_constant__ nmarl_model m, const float* __restrict__ part,
                                                              int tiles, int T, float* __restrict__ grads) {
  __shared__ float red[8][32];
  const int c = threadIdx.x & 31, p = threadIdx.x >> 5, col = blockIdx.x * 32 + c, i = blockIdx.y;
  const int n = T * tiles;
  float s = 0.f;
  for (int e = p; e < n; e += 8) {
    const int t = e / tiles, tile = e - t * tiles;
    s += part[(((size_t)t * m.n_agent + i) * tiles + tile) * NG + col];
  }
  red[p][c] = s;
  __syncthreads();
  if (p == 0) {
    float tsum = 0.f;
    for (int w = 0; w < 8; ++w) tsum += red[w][c];
    grads[m.agent[i].o_b + col] = tsum;
  }
}

int job_list(const nmarl_model* m, int* jobs) {
  int n = 0;
  jobs[n++] = J_GATE0;
  if (m->s_dim + NH > 128) jobs[n++] = J_GATE1;
  jobs[n++] = J_ENC_X;
  // (the fingerprint encoder shares the obs-encoder job: its few features sit on spare lanes of that tile)
  if (m->variant != NMARL_IA2C) {
    jobs[n++] = J_ENC_M0;
    if (m->km_pad > 128) jobs[n++] = J_ENC_M1;
  }
  return n;
}
int job_N(const nmarl_model* m, int kind) {
  if (kind == J_GATE0 || kind == J_GATE1) return 256;
  if (kind == J_ENC_X) return nmarl_tc_ndp(m);
  return 64;
}

}  // namespace

int nmarl_tc_ndp(const nmarl_model* m) { return m->variant == NMARL_NC ? 192 : (m->variant == NMARL_IA2C ? 64 : 128); }

int nmarl_tc_wgrad_splits(int n_agent) {
  int s = 37;                                   // 2 gate tiles x 37 x 8 agents = 592 CTAs = 4 waves of 148 SMs
  while (2 * s * n_agent > 148 * 8 && s > 1) s = (s + 1) / 2;
  return s;
}

int64_t nmarl_tc_wgrad_ws_floats(const nmarl_model* m) {
  int jobs[J_COUNT];
  const int nj = job_list(m, jobs);
  int64_t tot = 0;
  for (int j = 0; j < nj; ++j) tot += (int64_t)nmarl_tc_wgrad_splits(m->n_agent) * m->n_agent * 128 * job_N(m, jobs[j]);
  return tot;
}

int nmarl_tc_launch_wgrads(const nmarl_model* m, int B, int T, const float* sv_sh, const float* sv_xin, const float* dzT,
                           const float* dpT, const float* sv_dz, float* ws, float* grads, int* err, cudaStream_t st,
                           cudaStream_t st_bias, void** ev_wgrad, const float* h_seq, const float* done_pre) {
  TcWgK k{};
  k.B = B; k.T = T; k.splits = nmarl_tc_wgrad_splits(m->n_agent); k.ndp = nmarl_tc_ndp(m);
  k.sv_sh = sv_sh; k.sv_xin = sv_xin; k.dzT = dzT; k.dpT = dpT; k.ws = ws; k.err = err;
  k.h_seq = h_seq; k.done_pre = done_pre;
  k.prof = g_nmarl_prof;
  k.n_jobs = job_list(m, k.jobs);
  long long off = 0;
  for (int j = 0; j < k.n_jobs; ++j) { k.ws_off[j] = off; off += (long long)k.splits * m->n_agent * 128 * job_N(m, k.jobs[j]); }
  static bool configured = false;
  if (!configured) {
    NMARL_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM));
    configured = true;
  }
  gate_bias_reduce_kernel<<<dim3(NG / 32, m->n_agent), 256, 0, st_bias>>>(*m, sv_dz, B / 128, T, grads);   // independent of the GEMM jobs
  NMARL_LAUNCH_CHECK();
  if (ev_wgrad) NMARL_CUDA(cudaEventRecord((cudaEvent_t)ev_wgrad[0], st));
  tc_wgrad_kernel<<<dim3(k.splits, k.n_jobs, m->n_agent), TC_THREADS, WG_SMEM, st>>>(*m, k);
  NMARL_LAUNCH_CHECK();
  if (ev_wgrad) NMARL_CUDA(cudaEventRecord((cudaEvent_t)ev_wgrad[1], st));
  NMARL_DBG_SYNC(st, "tc_wgrad_kernel");
  tc_wgrad_reduce_kernel<<<dim3(64, k.n_jobs, m->n_agent), 256, 0, st>>>(*m, k, grads);
  NMARL_LAUNCH_CHECK();
  NMARL_DBG_SYNC(st, "tc_wgrad_reduce");
  return 0;
}
