// bwd_common.cuh -- argument block of one reverse step, shared by cell_bwd_kernel (FFMA, train.cu) and
// tc_cell_bwd_kernel (tcgen05, tc_bwd.cu)
#pragma once
#include "common.cuh"

// the opaque context of the C ABI: helper stream + events for forked side work (created on the current device)
struct nmarl_ctx {
  cudaStream_t side;
  cudaEvent_t fork, join, heads;
  int device;
};

struct BwdK {
  int B, t, has_next;
  const float* params; const float* wt;
  const float* done_pre;        // [B] for step t
  const float* sv_gates; const float* sv_sh; const float* sv_enc; const float* sv_dlv;   // step t
  const float* c_prev; const float* c_cur;      // c_seq[t], c_seq[t+1]
  const float* dh_in; const float* dc_in; const float* dmsg_in;       // produced by step t+1
  float* dh_out; float* dc_out; float* dmsg_out;                       // consumed by step t-1
  float* sv_dz; float* sv_dpre;                                        // step t (tcgen05 path: sv_dz = [N][tiles][256] gate-bias partials)
  const float* wpack; int* tc_err;                                     // tcgen05 path (NULL -> FFMA)
  float* dzT;                                                          // step t: [N][B/32][256][32] raw fp32 tiles or NULL
  float* dpT;                                                          // step t: [N][B/32][ndp][32] raw fp32 tiles (encoder pre-act grads)
  int ndp;                                                             // rows of a dpT tile: 192 (NC) / 128 (IC3, DIAL) / 64 (IA2C)
};

// floats per time step of sv_dzT (rows = 256) / sv_dpT (rows = ndp): one rows x 32 tile per agent and 32 envs
__host__ __device__ inline size_t nmarl_tc_tile_step_floats(int n_agent, int B, int rows) {
  return (size_t)n_agent * (B / 32) * rows * 32;
}

int nmarl_tc_launch_bwd(const nmarl_model* m, const BwdK& k, cudaStream_t st);
int nmarl_tc_wgrad_splits(int n_agent);
int64_t nmarl_tc_wgrad_ws_floats(const nmarl_model* m);
int nmarl_tc_ndp(const nmarl_model* m);
// all GEMM weight gradients (gate + encoders) of the tensor-core path; activations are feature-major
int nmarl_tc_launch_wgrads(const nmarl_model* m, int B, int T, const float* sv_sh, const float* sv_xin, const float* dzT,
                           const float* dpT, const float* sv_dz, float* ws, float* grads, int* err, cudaStream_t st, cudaStream_t st_bias,
                           void** ev_wgrad = nullptr,
                           const float* h_seq = nullptr, const float* done_pre = nullptr);
