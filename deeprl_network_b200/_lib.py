"""ctypes binding of libnmarl.so (the C ABI declared in include/nmarl.h).

The product path has NO CPU fallback: if the shared library is missing or a call fails this
module raises.  PyTorch is used only for device memory, streams and torch.distributed; kernels
receive raw device pointers (``tensor.data_ptr()``) and the current stream handle.
"""
import ctypes as C
import os

import torch

MAX_AGENT, MAX_NBR, NH, MAX_NA = 32, 4, 64, 8
IA2C, NC, IC3, DIAL = 0, 1, 2, 3
SAMPLE_NONE, SAMPLE_UNIFORM, SAMPLE_PHILOX, SAMPLE_GREEDY = 0, 1, 2, 3
CATCHUP, SLOWDOWN = 0, 1

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnmarl.so')


class Agent(C.Structure):
    _fields_ = [('n_nbr', C.c_int32), ('nbr', C.c_int32 * MAX_NBR),
                ('n_recv', C.c_int32), ('recv_agent', C.c_int32 * MAX_NBR), ('recv_slot', C.c_int32 * MAX_NBR),
                ('x_nsrc', C.c_int32), ('x_src', C.c_int32 * (MAX_NBR + 1)), ('x_w', C.c_int32),
                ('o_w_ob', C.c_int32), ('o_b_ob', C.c_int32), ('o_w_fp', C.c_int32), ('o_b_fp', C.c_int32),
                ('o_w_msg', C.c_int32), ('o_b_msg', C.c_int32), ('o_wxh', C.c_int32), ('o_b', C.c_int32),
                ('o_mfc_w', C.c_int32), ('o_mfc_b', C.c_int32),
                ('o_pi_w', C.c_int32), ('o_pi_b', C.c_int32), ('o_v_w', C.c_int32), ('o_v_b', C.c_int32),
                ('t_wxh', C.c_int32), ('t_w_msg', C.c_int32), ('t_mfc', C.c_int32),
                ('p_begin', C.c_int32), ('p_end', C.c_int32),
                ('tp_x', C.c_int32), ('tp_p', C.c_int32), ('tp_m', C.c_int32), ('tp_g', C.c_int32), ('tp_mfc', C.c_int32),
                ('tp_gT', C.c_int32), ('tp_mT', C.c_int32), ('tp_mfcT', C.c_int32)]


class Model(C.Structure):
    _fields_ = [('variant', C.c_int32), ('n_agent', C.c_int32), ('n_a', C.c_int32), ('s_dim', C.c_int32),
                ('obs_stride', C.c_int32), ('kx_pad', C.c_int32), ('kp_pad', C.c_int32), ('km_pad', C.c_int32),
                ('n_param', C.c_int32), ('n_wt', C.c_int32), ('per_agent_norm', C.c_int32), ('n_wp', C.c_int32),
                ('agent', Agent * MAX_AGENT)]


class CaccCfg(C.Structure):
    _fields_ = [('n_agent', C.c_int32), ('platoon_len', C.c_int32), ('scenario', C.c_int32),
                ('T', C.c_int32), ('batch_size', C.c_int32), ('global_reward', C.c_int32)] + \
               [(k, C.c_double) for k in ('dt', 'h_min', 'h_star', 'h_s', 'h_g', 'v_max', 'v_star',
                                          'u_min', 'u_max', 'rew_a', 'rew_b', 'G')]


class FwdArgs(C.Structure):
    _fields_ = [('B', C.c_int32), ('params', C.c_void_p), ('obs', C.c_void_p), ('fp', C.c_void_p),
                ('done', C.c_void_p), ('c_in', C.c_void_p), ('h_in', C.c_void_p), ('msg_in', C.c_void_p),
                ('c_out', C.c_void_p), ('h_out', C.c_void_p), ('msg_out', C.c_void_p),
                ('pi', C.c_void_p), ('action', C.c_void_p), ('sample_mode', C.c_int32),
                ('uniforms', C.c_void_p), ('rng', C.c_void_p), ('rng_offset', C.c_uint64),
                ('act_in', C.c_void_p), ('v', C.c_void_p), ('wpack', C.c_void_p), ('tc_err', C.c_void_p),
                ('sv_xin', C.c_void_p), ('sv_sh', C.c_void_p), ('sv_gates', C.c_void_p), ('sv_enc', C.c_void_p),
                ('state_fm', C.c_int32)]


class BwdArgs(C.Structure):
    _fields_ = [('B', C.c_int32), ('T', C.c_int32), ('B_total', C.c_int32),
                ('v_coef', C.c_float), ('e_coef', C.c_float),
                ('params', C.c_void_p), ('obs', C.c_void_p), ('fp', C.c_void_p), ('act', C.c_void_p),
                ('done_pre', C.c_void_p), ('Rs', C.c_void_p), ('Advs', C.c_void_p),
                ('h_seq', C.c_void_p), ('c_seq', C.c_void_p), ('msg_seq', C.c_void_p),
                ('sv_xin', C.c_void_p), ('sv_sh', C.c_void_p), ('sv_gates', C.c_void_p), ('sv_enc', C.c_void_p),
                ('sv_dlv', C.c_void_p), ('sv_dz', C.c_void_p), ('sv_dpre', C.c_void_p), ('sv_dmp', C.c_void_p),
                ('dh_rec', C.c_void_p), ('dc_rec', C.c_void_p), ('dmsg', C.c_void_p),
                ('wt', C.c_void_p), ('ws', C.c_void_p), ('ws_floats', C.c_int64),
                ('loss_part', C.c_void_p), ('grads', C.c_void_p), ('wpack', C.c_void_p), ('tc_err', C.c_void_p),
                ('sv_dzT', C.c_void_p), ('sv_dpT', C.c_void_p), ('state_fm', C.c_int32),
                ('ctx', C.c_void_p), ('ev_step', C.c_void_p), ('ev_wgrad', C.c_void_p), ('fused_heads', C.c_int32)]


_lib = None

EXPORTS = ['nmarl_last_error', 'nmarl_version', 'nmarl_create', 'nmarl_destroy', 'nmarl_sizeof_bwd_args', 'nmarl_sizeof_fwd_args', 'nmarl_sizeof_model', 'nmarl_sizeof_agent', 'nmarl_sizeof_cacc_cfg',
           'nmarl_cacc_reset', 'nmarl_cacc_step', 'nmarl_pack_weights', 'nmarl_policy_step_p', 'nmarl_policy_step_v', 'nmarl_tc_supported', 'nmarl_dial_msg',
           'nmarl_rng_advance', 'nmarl_nstep_return_adv', 'nmarl_loss_tiles', 'nmarl_ws_floats',
           'nmarl_a2c_backward', 'nmarl_a2c_train_forward', 'nmarl_a2c_bptt', 'nmarl_a2c_train_heads',
           'nmarl_clip_rmsprop_step', 'nmarl_consensus_update']


def lib():
    """Load libnmarl.so (once).  Raises if it is not built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('libnmarl.so not found at %s -- run `python -m deeprl_network_b200.build` '
                           '(or __graft_entry__.build()); this package has no CPU fallback' % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.nmarl_last_error.restype = C.c_char_p
    L.nmarl_ws_floats.restype = C.c_int64
    P, I, D, F, U64 = C.c_void_p, C.c_int, C.c_double, C.c_float, C.c_uint64
    L.nmarl_create.argtypes = [C.POINTER(C.c_void_p)]
    L.nmarl_destroy.argtypes = [P]
    L.nmarl_cacc_reset.argtypes = [C.POINTER(CaccCfg), I, P, P, U64, P, P, P, P, P, P, P, P, I, P, I, P]
    L.nmarl_cacc_step.argtypes = [C.POINTER(CaccCfg), I, I, P, P, P, P, P, P, P, P, I, P, P, P, P]
    L.nmarl_policy_step_p.argtypes = [C.POINTER(Model), C.POINTER(FwdArgs), P]
    L.nmarl_policy_step_v.argtypes = [C.POINTER(Model), C.POINTER(FwdArgs), P]
    L.nmarl_tc_supported.argtypes = [C.POINTER(Model), I]
    L.nmarl_dial_msg.argtypes = [C.POINTER(Model), I, P, P, P, P]
    L.nmarl_pack_weights.argtypes = [C.POINTER(Model), P, P, P, P]
    L.nmarl_rng_advance.argtypes = [P, U64, P]
    L.nmarl_nstep_return_adv.argtypes = [I, I, I, I, P, P, P, P, I, D, D, D, D, P, P, I, P, P, P]
    L.nmarl_loss_tiles.argtypes = [C.POINTER(Model), I]
    L.nmarl_ws_floats.argtypes = [C.POINTER(Model), I, I]
    for fn in ('nmarl_a2c_backward', 'nmarl_a2c_train_forward', 'nmarl_a2c_bptt', 'nmarl_a2c_train_heads'):
        getattr(L, fn).argtypes = [C.POINTER(Model), C.POINTER(BwdArgs), P]
    L.nmarl_clip_rmsprop_step.argtypes = [C.POINTER(Model), P, P, P, P, F, F, F, P, P, P]
    L.nmarl_consensus_update.argtypes = [C.POINTER(Model), P, P, P]
    assert L.nmarl_sizeof_model() == C.sizeof(Model), 'nmarl_model layout mismatch'
    assert L.nmarl_sizeof_agent() == C.sizeof(Agent), 'nmarl_agent layout mismatch'
    assert L.nmarl_sizeof_cacc_cfg() == C.sizeof(CaccCfg), 'nmarl_cacc_cfg layout mismatch'
    assert L.nmarl_sizeof_bwd_args() == C.sizeof(BwdArgs), 'nmarl_bwd_args layout mismatch'
    assert L.nmarl_sizeof_fwd_args() == C.sizeof(FwdArgs), 'nmarl_fwd_args layout mismatch'
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        raise RuntimeError('%s failed (rc=%d): %s' % (what, rc, lib().nmarl_last_error().decode()))


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), 'kernels need contiguous CUDA tensors'
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('deeprl_network_b200 needs a CUDA device (sm_100a); no CPU fallback exists')
