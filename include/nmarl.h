/* nmarl.h -- C ABI of the B200-native networked-MARL hot path (libnmarl.so).
 *
 * Drop-in boundary (SURVEY.md 8b): the reference has no FFI; the surface it exposes is the
 * Python env/agent API.  This header is what the Python mirror of that API
 * (deeprl_network_b200/) binds with ctypes; each entry point names the reference code it
 * replaces (paths relative to the reference checkout).
 *
 * Conventions: extern "C"; every function returns 0 on success, non-zero on error
 * (message via nmarl_last_error(), thread-local); never throws; never allocates device memory and
 * keeps no global state -- the caller owns every buffer and passes raw device pointers plus an
 * explicit stream (cudaStream_t passed as void*).  The only library-owned resources are the ones
 * inside an opaque `nmarl_ctx`: one helper stream + two events used to fork side work beside the
 * BPTT chain, created by nmarl_create and freed by nmarl_destroy; entry points that fork take
 * the ctx through their argument block.  Re-entrant per ctx, not thread-safe per ctx.  All launches
 * are asynchronous on the given stream and are CUDA-graph capturable.  Device code is sm_100a only.
 *
 * Layout: every per-agent tensor is agent-major, env-minor: X[agent][env][feature]
 * (so an agent's rows are contiguous for its grouped GEMM, and the env kernel is coalesced
 * over envs).  Time-stacked buffers are [t][agent][env][feature].  fp32 unless stated.
 */
#ifndef NMARL_H
#define NMARL_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#pragma GCC visibility push(default)

#define NMARL_MAX_AGENT 32
#define NMARL_MAX_NBR   4
#define NMARL_NH        64      /* LSTM width (num_lstm = num_fc = 64 in every shipped config) */
#define NMARL_MAX_NA    8

enum { NMARL_IA2C = 0, NMARL_NC = 1, NMARL_IC3 = 2, NMARL_DIAL = 3 };
enum { NMARL_SAMPLE_NONE = 0, NMARL_SAMPLE_UNIFORM = 1, NMARL_SAMPLE_PHILOX = 2, NMARL_SAMPLE_GREEDY = 3 };
enum { NMARL_CATCHUP = 0, NMARL_SLOWDOWN = 1 };

/* ---- model description (host builds it; passed by value to kernels) -------------------- */
typedef struct {
  int32_t n_nbr;                         /* |N(i)|                                             */
  int32_t nbr[NMARL_MAX_NBR];            /* neighbours, ascending (tf.boolean_mask order,       */
                                         /*   agents/utils.py:192-194)                          */
  int32_t n_recv;                        /* agents k with i in N(k)  (backward message scatter) */
  int32_t recv_agent[NMARL_MAX_NBR];
  int32_t recv_slot[NMARL_MAX_NBR];      /* position of i inside N(k)                           */
  int32_t x_nsrc;                        /* observation gather: x~ = concat_s obs[x_src[s]][:x_w] */
  int32_t x_src[NMARL_MAX_NBR + 1];
  int32_t x_w;
  /* offsets (floats, multiples of 4) into the flat parameter / gradient / rmsprop buffers; -1 = absent */
  int32_t o_w_ob, o_b_ob;                /* obs encoder  (IA2C: lstm_i/fc)                      */
  int32_t o_w_fp, o_b_fp;                /* fingerprint encoder (NC)                            */
  int32_t o_w_msg, o_b_msg;              /* message encoder (NC, IC3, DIAL)                     */
  int32_t o_wxh;                         /* [s_dim + 64][256] = wx rows then wh rows            */
  int32_t o_b;                           /* [256]                                               */
  int32_t o_mfc_w, o_mfc_b;              /* DIAL sender-side message fc                         */
  int32_t o_pi_w, o_pi_b, o_v_w, o_v_b;  /* heads                                               */
  /* offsets into the transposed-weight scratch (backward dgrad): */
  int32_t t_wxh;                         /* [256][s_dim + 64]                                   */
  int32_t t_w_msg;                       /* [64][k_m]                                           */
  int32_t t_mfc;                         /* [64][64]                                            */
  int32_t p_begin, p_end;                /* this agent's contiguous parameter range             */
  /* offsets into the packed tensor-core operand buffer (nmarl_pack_weights); -1 = absent:              */
  int32_t tp_x, tp_p, tp_m, tp_g, tp_mfc; /* encoders (N=64 tiles), gate [wx;wh] (N=256 tiles), DIAL mfc  */
  int32_t tp_gT, tp_mT, tp_mfcT;         /* backward: [wx;wh]^T (N=s_dim+64), w_msg^T (N=k_m), w_mfc^T     */
} nmarl_agent;

typedef struct {
  int32_t variant;                       /* NMARL_IA2C / NC / IC3 / DIAL                        */
  int32_t n_agent, n_a, s_dim;           /* s_dim = 192 (NC) or 64                              */
  int32_t obs_stride;                    /* floats per obs row                                  */
  int32_t kx_pad, kp_pad, km_pad;        /* padded (x4) widths of the x~ / p~ / m~ input segments */
  int32_t n_param, n_wt;                 /* flat buffer sizes (floats)                          */
  int32_t per_agent_norm;                /* 1: clip each agent's range separately (IA2C)        */
  int32_t n_wp;                          /* floats in the packed tensor-core operand buffer     */
  nmarl_agent agent[NMARL_MAX_AGENT];
} nmarl_model;

/* ---- CACC environment constants (envs/cacc_env.py:320-343) ----------------------------- */
typedef struct {
  int32_t n_agent, platoon_len;          /* platoon_len == n_agent for CACC; <n_agent: several  */
                                         /*   independent platoons (5x5-grid dynamics stub)     */
  int32_t scenario;                      /* NMARL_CATCHUP / NMARL_SLOWDOWN                      */
  int32_t T, batch_size;                 /* episode length in steps; collision-done period      */
  int32_t global_reward;                 /* coop_gamma < 0: reward := sum over agents           */
  double dt, h_min, h_star, h_s, h_g, v_max, v_star, u_min, u_max, rew_a, rew_b, G;
} nmarl_cacc_cfg;

const char* nmarl_last_error(void);
int nmarl_version(void);
/* ---- context (SURVEY 8b): owns the helper stream/events of the CURRENT device; no other state ---------- */
typedef struct nmarl_ctx nmarl_ctx;
int nmarl_create(nmarl_ctx** out);
int nmarl_destroy(nmarl_ctx* ctx);
/* size-of checks so the ctypes mirror can assert its struct layout */
int nmarl_sizeof_model(void);
int nmarl_sizeof_agent(void);
int nmarl_sizeof_cacc_cfg(void);
int nmarl_sizeof_fwd_args(void);
int nmarl_sizeof_bwd_args(void);

/* ---- K1: environment ---------------------------------------------------------------------
 * Replaces CACCEnv.reset/_init_catchup/_init_slowdown (envs/cacc_env.py:166-189,285-318) and
 * CACCEnv.step/_get_reward/_get_state (envs/cacc_env.py:191-242,40-79).  State is float64
 * (the reference is), observations are emitted as float32.
 *   hs,vs,us  double [N][B]     t int32 [B]     collision int32 [B]     v_init double [B]
 *   u01       double [B]  one uniform per env (the reference's single np.random.rand()); may be
 *             NULL -> Philox(seed, env, episode[b])
 *   mask      float [B] or NULL: reset only envs with mask != 0
 *   obs       float [N][B][obs_stride] (first 5 columns written); fp float [N][B][n_a] := 1/n_a
 */
int nmarl_cacc_reset(const nmarl_cacc_cfg* cfg, int B, const double* u01, const float* mask,
                     uint64_t seed, int32_t* episode,
                     double* hs, double* vs, double* us, int32_t* t, int32_t* collision, double* v_init,
                     float* obs, int obs_stride, float* fp, int n_a, void* stream);
/*   action int32 [N][B];  reward double [NR][B] (NR = 1 if global_reward else N);
 *   greward double [B];  done float [B] (1.0 / 0.0)                                           */
int nmarl_cacc_step(const nmarl_cacc_cfg* cfg, int B, int train_mode, const int32_t* action,
                    double* hs, double* vs, double* us, int32_t* t, int32_t* collision, const double* v_init,
                    float* obs, int obs_stride, double* reward, double* greward, float* done, void* stream);

/* ---- K2-K6: fused message-gather + encoders + LSTM cell + heads ----------------------------
 * Replaces lstm / lstm_comm / lstm_ic3 / lstm_dial (agents/utils.py:87-115,118-217,344-417,
 * 515-599), the actor/critic heads (agents/policies.py:50-77,291-312), the 'p' / 'v' forward
 * protocol (agents/policies.py:119-134,215-230) and action sampling (utils.py:135-141).      */
typedef struct {
  int32_t B;
  const float* params;
  const float* obs;        /* [N][B][obs_stride]                                              */
  const float* fp;         /* [N][B][n_a]  previous-step policies (NC, DIAL) or NULL           */
  const float* done;       /* [B] pre-step done (1 -> own c,h zeroed; messages NOT masked)     */
  const float* c_in;       /* [N][B][64]                                                       */
  const float* h_in;       /* [N][B][64]                                                       */
  const float* msg_in;     /* DIAL: [N][B][64] relu(h_in W_mfc + b)                            */
  float* c_out;            /* p-call: new state (must not alias *_in)                          */
  float* h_out;
  float* msg_out;          /* DIAL p-call                                                      */
  float* pi;               /* p-call: [N][B][n_a]                                              */
  int32_t* action;         /* p-call: [N][B] or NULL                                           */
  int32_t sample_mode;     /* NMARL_SAMPLE_*                                                   */
  const double* uniforms;  /* [N][B] for NMARL_SAMPLE_UNIFORM                                  */
  const uint64_t* rng;     /* device [2] = {seed, counter} for NMARL_SAMPLE_PHILOX             */
  uint64_t rng_offset;     /* added to the device counter (distinct per call inside a graph)   */
  const int32_t* act_in;   /* v-call / train: [N][B] same-step actions                         */
  float* v;                /* v-call: [N][B]                                                   */
  const float* wpack;      /* packed 3xTF32 operands (nmarl_pack_weights) or NULL.  When set and  */
                           /* nmarl_tc_supported(m, B) the tcgen05 tensor-core kernel is used,    */
                           /* else FP32 FFMA                                                      */
  int32_t* tc_err;         /* device int: tensor-core pipeline watchdog (0 = ok); may be NULL      */
  /* optional (p-call, tensor-core path only): save the activations BPTT needs while rolling out, so the
   * update can skip the separate training forward (same inputs, same weights => same numbers):         */
  float* sv_xin; float* sv_sh; float* sv_gates; float* sv_enc;   /* step-t slices, see nmarl_bwd_args      */
  int32_t state_fm;        /* 1: c/h tensors are feature-major [N][64][B].  Must be 1 on the        */
                           /* tensor-core path except for DIAL, 0 otherwise (the call fails)      */
} nmarl_fwd_args;

int nmarl_policy_step_p(const nmarl_model* m, const nmarl_fwd_args* a, void* stream);
int nmarl_policy_step_v(const nmarl_model* m, const nmarl_fwd_args* a, void* stream);
/* 1 if the tensor-core kernels cover model m at B envs (whole 128-env tiles, obs / fingerprint segments of at
 * most 32 floats, packed operands laid out for every agent), else 0.  Every entry point given a wpack runs the
 * tensor-core path exactly when this holds; the caller sizes its buffers and state_fm by it.                */
int nmarl_tc_supported(const nmarl_model* m, int B);
/* Pack the GEMM weights for the tcgen05 path: per 32-wide k-block a [hi | lo] pair of 128B-swizzled
 * K-major tiles of W^T (hi = value rounded to TF32, lo = rounded remainder).  Call after every parameter
 * change.  wt (transposed weights scratch, n_wt floats) is also refreshed.                           */
int nmarl_pack_weights(const nmarl_model* m, const float* params, float* wt, float* wpack, void* stream);
/* DIAL only: msg[N][B][64] = relu(h W_mfc + b) (agents/utils.py:563-566); needed after a reset */
int nmarl_dial_msg(const nmarl_model* m, int B, const float* params, const float* h, float* msg, void* stream);
/* advance the device Philox counter by n (one tiny kernel; keeps graph replays fresh) */
int nmarl_rng_advance(uint64_t* rng, uint64_t n, void* stream);

/* ---- K7: n-step returns / advantages -------------------------------------------------------
 * Replaces add_transition's reward norm/clip (agents/models.py:26-32,198-209) and
 * _add_R_Adv / _add_s_R_Adv (agents/utils.py:763-775,800-816,837-855,888-912); float64 math,
 * float32 outputs like the reference.
 *   reward double [T][NR][B] raw;  value float [T][N][B];  done_post float [T][B];
 *   R_end float [N][B] (ignored where done_post[T-1] != 0 when zero_end_if_done);
 *   alpha < 0: global reward (NR == 1);  alpha > 0: spatial, dist int32 [N][N],
 *   alpha_pow double [maxdist+1] = alpha**d
 *   Rs, Advs float [T][N][B]                                                                 */
int nmarl_nstep_return_adv(int n_agent, int B, int T, int NR, const double* reward, const float* value,
                           const float* done_post, const float* R_end, int zero_end_if_done,
                           double gamma, double reward_norm, double reward_clip,
                           double alpha, const int32_t* dist, const double* alpha_pow, int n_pow,
                           float* Rs, float* Advs, void* stream);

/* ---- K8-K9: A2C loss, BPTT with message-gradient scatter, weight gradients ------------------
 * Replaces the 'backward' graph + prepare_loss + tf.gradients (agents/policies.py:20-39,
 * 232-264) for a batch of T steps starting from states_bw.  Buffers (all caller-owned):
 *   obs [T][N][B][obs_stride]  fp [T][N][B][n_a]  act int32 [T][N][B]  done_pre float [T][B]
 *   Rs, Advs float [T][N][B]
 *   h_seq, c_seq [T+1][N][B][64]  (index 0 = states_bw, filled by the caller)
 *   msg_seq      [T+1][N][B][64]  (DIAL; index 0 filled by nmarl_dial_msg)
 *   sv_xin [T][N][B][kx_pad+kp_pad+km_pad]  sv_sh [T][N][B][s_dim+64]  sv_gates [T][N][B][256]
 *   sv_enc [T][N][B][128] (IC3: 64 used; DIAL: 128)   sv_dlv [T][N][B][8]
 *   sv_dz [T][N][B][256]   sv_dpre [T][N][B][192]   sv_dmp [T][N][B][64] (DIAL)
 *   (tensor-core path: sv_dz = [T][N][B/128][256] per-tile gate-bias partial sums, sv_dpre unused)
 *   dh_rec, dc_rec [2][N][B][64]   dmsg [2][N][MAX_NBR][B][64]
 *   wt [n_wt] transposed weights   ws: split-K workspace of ws_floats floats
 *   loss_part float [T][N][tiles][4] per-CTA partial sums (policy, value, entropy, pad)
 *   grads [n_param] (fully overwritten)
 */
typedef struct {
  int32_t B, T;
  int32_t B_total;           /* global env count (all ranks) for the 1/(T*B_total) loss scale  */
  float v_coef, e_coef;
  const float* params;
  const float* obs; const float* fp; const int32_t* act; const float* done_pre;
  const float* Rs; const float* Advs;
  float* h_seq; float* c_seq; float* msg_seq;
  float* sv_xin; float* sv_sh; float* sv_gates; float* sv_enc; float* sv_dlv;
  float* sv_dz; float* sv_dpre; float* sv_dmp;
  float* dh_rec; float* dc_rec; float* dmsg;
  float* wt; float* ws; int64_t ws_floats;
  float* loss_part;
  float* grads;
  const float* wpack;        /* packed tensor-core operands or NULL (see nmarl_fwd_args)            */
  int32_t* tc_err;
  float* sv_dzT;             /* tensor-core path: dz^T as [T][N][B/32][256][32] swizzled raw fp32 tiles (the
                                weight-gradient kernel derives the 3xTF32 `lo` part in shared memory)               */
  float* sv_dpT;             /* tensor-core path: encoder pre-activation grads^T, [T][N][B/32][ndp][32] likewise,
                                ndp = 192 (NC) / 128 (IC3, DIAL) / 64 (IA2C).  On the tensor-core path (wpack set,
                                nmarl_tc_supported) sv_xin / sv_sh / sv_gates / sv_enc are FEATURE-MAJOR
                                [T][N][feature][B] and sv_dpre is unused.  With state_fm the done-masked own state
                                (rows s_dim.. of sv_sh) and, for NeurComm, the neighbour messages (the m~ block of
                                sv_xin) are NOT stored a second time: the weight-gradient kernel reads h_seq.        */
  int32_t state_fm;          /* 1: h_seq / c_seq / dh_rec / dc_rec / dmsg are feature-major ([..][64][B] instead of
                                [..][B][64]).  Must be 1 on the tensor-core path except for DIAL, 0 otherwise        */
  nmarl_ctx* ctx;            /* required by nmarl_a2c_bptt / nmarl_a2c_backward (forked side work)                  */
  void** ev_step;            /* optional timing hooks (bench.py): 2*T cudaEvent_t, recorded on `stream` before /
                                after the cell kernel of reverse step t at [2t], [2t+1]; NULL = none               */
  void** ev_wgrad;           /* optional: 2 cudaEvent_t around the weight-gradient GEMM kernel; NULL = none         */
  int32_t fused_heads;       /* nmarl_a2c_bptt also does the work of nmarl_a2c_train_heads (do not call it), most of it
                                on the ctx's side stream beside the first reverse steps                              */
} nmarl_bwd_args;

int nmarl_loss_tiles(const nmarl_model* m, int B);       /* tiles per agent in loss_part      */
int64_t nmarl_ws_floats(const nmarl_model* m, int B, int T);   /* required workspace          */
int nmarl_a2c_backward(const nmarl_model* m, const nmarl_bwd_args* a, void* stream);
/* the two halves, exposed for tests: training forward (saves activations, loss partials,
 * head gradients) and the reverse pass + weight gradients */
int nmarl_a2c_train_forward(const nmarl_model* m, const nmarl_bwd_args* a, void* stream);
int nmarl_a2c_bptt(const nmarl_model* m, const nmarl_bwd_args* a, void* stream);
/* when the rollout p-calls already saved the activations (nmarl_fwd_args.sv_*): only the heads, the loss
 * partials and d(loss)/d(logits, v) are computed from h_seq -- replaces nmarl_a2c_train_forward             */
int nmarl_a2c_train_heads(const nmarl_model* m, const nmarl_bwd_args* a, void* stream);

/* ---- K10: global-norm clip + TF-semantics RMSProp -------------------------------------------
 * Replaces tf.clip_by_global_norm + tf.train.RMSPropOptimizer (agents/policies.py:34-39,
 * 259-264): g *= clip/max(|g|,clip); ms = rho*ms + (1-rho) g^2 (ms0 = 1); w -= lr*g/sqrt(ms+eps).
 *   lr: device float[1];  norm_out: device float [n_groups] (n_groups = n_agent if
 *   per_agent_norm else 1);  scratch: device float [>= 1024]                                  */
int nmarl_clip_rmsprop_step(const nmarl_model* m, float* params, float* grads, float* ms,
                            const float* lr, float max_grad_norm, float rho, float eps,
                            float* norm_out, float* scratch, void* stream);

/* ---- consensus update (IA2C_CU / `ma2c_cu`) ----------------------------------------------------
 * Replaces ConsensusPolicy._consensus_update (agents/policies.py:351-359, 401-426), run after every
 * optimizer step: agent i's LSTM variables (wx, wh, b -- one contiguous block of the flat buffer) become
 * the mean of the blocks of {i} + its neighbours (ascending index), all read BEFORE any is written.
 *   scratch: device float [n_agent * ((s_dim + 64) * 256 + 256)]                                         */
int nmarl_consensus_update(const nmarl_model* m, float* params, float* scratch, void* stream);

#pragma GCC visibility pop
#ifdef __cplusplus
}
#endif
#endif /* NMARL_H */
