"""Device-resident policy/learner engine: owns parameters, LSTM states, rollout and training
buffers (all torch CUDA tensors) and drives the libnmarl kernels through the C ABI.

It plays the role of the reference's TF session + policy objects (agents/policies.py) plus
the on-policy buffer (agents/utils.py:722-912), for B parallel environments:
  * ``step_p`` / ``step_v``    -- 'p' and 'v' forward calls incl. quirk Q1 (the v-call re-runs the
                                 cell from the state the p-call just stored; policies.py:215-230)
  * ``rollout``                -- n_step vectorised env steps + bootstrap (Q2), all on device
  * ``compute_returns``        -- n-step / spatially discounted returns
  * ``update``                 -- training forward, loss, BPTT, [NCCL all-reduce], clip, RMSProp,
                                 then states_bw := states_fw (policies.py:211)
"""
import ctypes as C
import os

import numpy as np
import torch

from .. import _lib as L

NH = L.NH


class PolicyEngine:
    def __init__(self, layout, n_env, n_step, hp, flat_params=None, device=None, rng_seed=0,
                 distance_mask=None, coop_gamma=-1.0, group=None, use_tc=None):
        """hp: dict(v_coef, e_coef, max_grad_norm, alpha, epsilon, gamma, reward_norm, reward_clip)."""
        L.require_cuda()
        self.layout, self.B, self.T, self.hp = layout, int(n_env), int(n_step), dict(hp)
        self.N, self.n_a = layout.N, layout.n_a
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        self.group = group
        self.world = torch.distributed.get_world_size(group) if (group is not None or (
            torch.distributed.is_available() and torch.distributed.is_initialized())) else 1
        self.model = layout.c_model()
        # kernel family: ma2c_cu runs the IA2C cell, ia2c_fp the NeurComm cell (layout.py docstring)
        self.agent_name = layout.variant
        self.variant = {'ma2c_cu': 'ia2c', 'ia2c_fp': 'ma2c_nc'}.get(layout.variant, layout.variant)
        dev, N, B, T = self.device, self.N, self.B, self.T
        f32 = dict(dtype=torch.float32, device=dev)
        if flat_params is None:
            flat_params = layout.init_flat()
        self.params = torch.as_tensor(np.asarray(flat_params, dtype=np.float32)).to(dev).contiguous()
        assert self.params.numel() == layout.n_param
        self.grads = torch.zeros(layout.n_param, **f32)
        self.ms = torch.ones(layout.n_param, **f32)             # TF RMSProp slot starts at 1
        self.wt = torch.zeros(layout.n_wt, **f32)
        # tcgen05 path: packed 3xTF32 operands; the library runs it whenever wpack is passed and nmarl_tc_supported holds
        if use_tc is None:
            use_tc = os.environ.get('NMARL_NO_TC', '0') != '1'
        self.use_tc = bool(use_tc) and bool(L.lib().nmarl_tc_supported(C.byref(self.model), self.B))
        self.wpack = torch.zeros(layout.n_wp, **f32) if self.use_tc else None
        self.tc_err = torch.zeros(1, dtype=torch.int32, device=dev)
        # tensor-core path: LSTM state (and its gradients) feature-major [N,64,B] so that lane == env accesses are
        # coalesced; DIAL keeps env-major state (its message kernels are env-major)
        self.state_fm = self.use_tc and self.variant != 'ma2c_dial'
        self._sshape = (N, NH, B) if self.state_fm else (N, B, NH)
        self.c = [torch.zeros(*self._sshape, **f32) for _ in range(2)]
        self.h = [torch.zeros(*self._sshape, **f32) for _ in range(2)]
        self.msg = [torch.zeros(N, B, NH, **f32) for _ in range(2)] if self.variant == 'ma2c_dial' else [None, None]
        self.cur = 0
        self.c_bw, self.h_bw = torch.zeros(*self._sshape, **f32), torch.zeros(*self._sshape, **f32)
        S = layout.obs_stride
        self.obs_buf = torch.zeros(T + 1, N, B, S, **f32)
        self.fp_buf = torch.full((T + 1, N, B, self.n_a), 1.0 / self.n_a, **f32)
        self.done_buf = torch.ones(T + 1, B, **f32)
        self.act_buf = torch.zeros(T, N, B, dtype=torch.int32, device=dev)
        self.val_buf = torch.zeros(T, N, B, **f32)
        self.alpha = float(coop_gamma)
        self.NR = 1 if self.alpha < 0 else N
        self.rew_buf = torch.zeros(T, self.NR, B, dtype=torch.float64, device=dev)
        self.grew_buf = torch.zeros(T, B, dtype=torch.float64, device=dev)
        self.R_end = torch.zeros(N, B, **f32)
        self.boot_pi = torch.zeros(N, B, self.n_a, **f32)
        self.boot_act = torch.zeros(N, B, dtype=torch.int32, device=dev)
        self.Rs, self.Advs = torch.zeros(T, N, B, **f32), torch.zeros(T, N, B, **f32)
        self.pi_tmp = torch.zeros(N, B, self.n_a, **f32)
        self.lr_dev = torch.zeros(1, **f32)
        self.n_groups = N if self.model.per_agent_norm else 1
        self.norm_out = torch.zeros(self.n_groups, **f32)
        self.opt_scratch = torch.zeros(1024, **f32)
        self.rng = torch.tensor([int(rng_seed) & (2 ** 63 - 1), 0], dtype=torch.int64, device=dev)
        self.uniforms = None
        if self.alpha > 0:
            dm = np.asarray(distance_mask, dtype=np.int32)
            self.dist_dev = torch.as_tensor(dm).to(dev).contiguous()
            md = int(dm.max())
            self.alpha_pow = torch.tensor([self.alpha ** d for d in range(md + 1)], dtype=torch.float64, device=dev)
        else:
            self.dist_dev, self.alpha_pow = None, None
        self._train_ready = False
        self.saved_rollout = False
        self.fuse_save = os.environ.get('NMARL_NO_FUSE_SAVE', '0') != '1'
        # v-calls run on a second stream: v(t) only feeds val_buf, so it overlaps env.step(t) and p(t+1)
        self.overlap_v = os.environ.get('NMARL_NO_OVERLAP', '0') != '1'
        self._vstream = None
        self.kernel_events = None          # bench.py: list collecting (start, end) CUDA events around each rollout p-call
        self.T_cur = T
        self.launches = 0
        self.raw_tiles = self.use_tc       # read by bench.py (profiles/traffic.json keys): operand tiles are raw fp32
        self.bwd_events = None             # bench.py: (step events [2T], wgrad events [2]) recorded inside nmarl_a2c_bptt
        self._ctx = C.c_void_p()
        L.check(L.lib().nmarl_create(C.byref(self._ctx)), 'nmarl_create')
        self.repack()

    def __del__(self):
        ctx = getattr(self, '_ctx', None)
        if ctx is not None and ctx.value:
            try:
                L.lib().nmarl_destroy(ctx)
            except Exception:
                pass
            self._ctx = None

    # ---- state ----------------------------------------------------------------------------------
    def reset_states(self, mask=None):
        """policies.py:334-336 (``_reset``): zero states_fw and states_bw; mask [B] selects envs."""
        if mask is None:
            for t in (self.c[self.cur], self.h[self.cur], self.c_bw, self.h_bw):
                t.zero_()
        else:
            keep = (1.0 - mask)[None, None, :] if self.state_fm else (1.0 - mask)[None, :, None]
            for t in (self.c[self.cur], self.h[self.cur], self.c_bw, self.h_bw):
                t.mul_(keep)
        self._refresh_msg()

    def repack(self):
        """Refresh the packed tensor-core operands after any parameter change."""
        if self.use_tc:
            L.check(L.lib().nmarl_pack_weights(C.byref(self.model), L.ptr(self.params), L.ptr(self.wt), L.ptr(self.wpack),
                                               L.stream()), 'nmarl_pack_weights')
            self.launches += 8 * self.N

    def check_tc(self):
        """Host sync: raise if the tensor-core pipeline watchdog fired."""
        code = int(self.tc_err.item())
        if code:
            raise RuntimeError('tcgen05 pipeline watchdog fired (code %d)' % code)

    def _refresh_msg(self):
        if self.variant == 'ma2c_dial':
            L.check(L.lib().nmarl_dial_msg(C.byref(self.model), self.B, L.ptr(self.params), L.ptr(self.h[self.cur]),
                                           L.ptr(self.msg[self.cur]), L.stream()), 'nmarl_dial_msg')
            self.launches += 1

    def normalize_cur(self):
        """Bring the ping-pong state index back to slot 0 (a captured CUDA graph bakes pointers, and
        an update performs an odd number of p-calls)."""
        if self.cur != 0:
            self.c[0].copy_(self.c[1]); self.h[0].copy_(self.h[1])
            if self.msg[0] is not None:
                self.msg[0].copy_(self.msg[1])
            self.cur = 0

    def get_states_fw(self):
        """[N, B, 128] = [c | h] like the reference's states_fw (env-major view whatever the device layout)."""
        c, h = self.c[self.cur], self.h[self.cur]
        if self.state_fm:
            c, h = c.permute(0, 2, 1), h.permute(0, 2, 1)
        return torch.cat([c, h], dim=-1).contiguous()

    def set_states(self, c, h, bw=True):
        """c, h: env-major [N, B, 64]."""
        if self.state_fm:
            c, h = c.permute(0, 2, 1), h.permute(0, 2, 1)
        self.c[self.cur].copy_(c); self.h[self.cur].copy_(h)
        if bw:
            self.c_bw.copy_(c); self.h_bw.copy_(h)
        self._refresh_msg()

    # ---- forward calls ----------------------------------------------------------------------------
    def _fwd_args(self, obs, fp, done):
        a = L.FwdArgs()
        a.B = self.B
        a.params, a.obs, a.fp, a.done = L.ptr(self.params), L.ptr(obs), L.ptr(fp), L.ptr(done)
        a.c_in, a.h_in, a.msg_in = L.ptr(self.c[self.cur]), L.ptr(self.h[self.cur]), L.ptr(self.msg[self.cur])
        a.wpack, a.tc_err, a.state_fm = L.ptr(self.wpack), L.ptr(self.tc_err), int(self.state_fm)
        return a

    def step_p(self, obs, fp, done, pi_out, action_out=None, sample_mode=L.SAMPLE_NONE, uniforms=None, rng_offset=0):
        """'p' call: advances and STORES the LSTM state, writes pi (and sampled/greedy actions)."""
        a = self._fwd_args(obs, fp, done)
        nxt = 1 - self.cur
        a.c_out, a.h_out, a.msg_out = L.ptr(self.c[nxt]), L.ptr(self.h[nxt]), L.ptr(self.msg[nxt])
        a.pi, a.action, a.sample_mode = L.ptr(pi_out), L.ptr(action_out), sample_mode
        a.uniforms, a.rng, a.rng_offset = L.ptr(uniforms), L.ptr(self.rng), rng_offset
        L.check(L.lib().nmarl_policy_step_p(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_policy_step_p')
        self.cur = nxt
        self.launches += 1

    def step_v(self, obs, fp, done, act_in, v_out):
        """'v' call: re-runs the cell from the CURRENT (post-p) state, state not stored (quirk Q1)."""
        a = self._fwd_args(obs, fp, done)
        a.act_in, a.v = L.ptr(act_in), L.ptr(v_out)
        L.check(L.lib().nmarl_policy_step_v(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_policy_step_v')
        self.launches += 1

    # ---- vectorised rollout (utils.py:163-197 for B envs) -------------------------------------------
    def begin_episode(self, env, obs_slot=0):
        """Copy the env's reset observation / fingerprint into slot 0 and mark done_prev = True."""
        self.obs_buf[obs_slot].copy_(env.obs_dev)
        self.fp_buf[obs_slot].copy_(env.fp_dev)
        self.done_buf[obs_slot].fill_(1.0)

    def rollout(self, env, sample='philox', uniforms=None, bootstrap=True, n_step=None):
        """n_step env steps for all B envs entirely on device.  uniforms: double [T+1, N, B] when
        sample == 'uniform' (host-supplied RNG, reference parity mode)."""
        T = self.T if n_step is None else int(n_step)
        self.T_cur = T
        mode = {'philox': L.SAMPLE_PHILOX, 'uniform': L.SAMPLE_UNIFORM, 'greedy': L.SAMPLE_GREEDY}[sample]
        # tensor-core path: the rollout p-calls save the activations BPTT needs (same inputs, same weights as
        # the reference's separate training forward => same numbers), and the LSTM state lives in h_seq/c_seq
        self.saved_rollout = bool(self.use_tc and self.fuse_save and bootstrap and sample != 'greedy' and T == self.T)
        if self.saved_rollout:
            self._alloc_train()
            self._rollout_saved(env, mode, uniforms, T)
            return
        for t in range(T):
            obs, fp, done = self.obs_buf[t], self.fp_buf[t], self.done_buf[t]
            self.step_p(obs, fp, done, self.fp_buf[t + 1], self.act_buf[t], mode,
                        None if uniforms is None else uniforms[t], rng_offset=t)
            self.step_v(obs, fp, done, self.act_buf[t], self.val_buf[t])
            env.step_device(self.act_buf[t], obs_out=self.obs_buf[t + 1], reward_out=self.rew_buf[t],
                            greward_out=self.grew_buf[t], done_out=self.done_buf[t + 1])
            self.launches += 1
        if bootstrap:
            # Q2: the bootstrap value comes from another p-call (state advanced, RNG consumed) + v-call;
            # the fingerprint is NOT updated by it (utils.py:192-196).
            self.step_p(self.obs_buf[T], self.fp_buf[T], self.done_buf[T], self.boot_pi, self.boot_act, mode,
                        None if uniforms is None else uniforms[T], rng_offset=T)
            self.step_v(self.obs_buf[T], self.fp_buf[T], self.done_buf[T], self.boot_act, self.R_end)
        if mode == L.SAMPLE_PHILOX:
            L.check(L.lib().nmarl_rng_advance(L.ptr(self.rng), T + 1, L.stream()), 'nmarl_rng_advance')
            self.launches += 1

    def _seq_call(self, t, obs, fp, done, which, **kw):
        """p- or v-call with the state taken from / written to slot t / t+1 of the saved sequences."""
        a = L.FwdArgs()
        a.B = self.B
        a.params, a.obs, a.fp, a.done = L.ptr(self.params), L.ptr(obs), L.ptr(fp), L.ptr(done)
        a.wpack, a.tc_err, a.state_fm = L.ptr(self.wpack), L.ptr(self.tc_err), int(self.state_fm)
        ms = self.msg_seq
        if which == 'p':
            a.c_in, a.h_in, a.msg_in = L.ptr(self.c_seq[t]), L.ptr(self.h_seq[t]), L.ptr(None if ms is None else ms[t])
            a.c_out, a.h_out, a.msg_out = L.ptr(self.c_seq[t + 1]), L.ptr(self.h_seq[t + 1]), L.ptr(None if ms is None else ms[t + 1])
            a.pi, a.action, a.sample_mode = L.ptr(kw['pi']), L.ptr(kw['action']), kw['mode']
            a.uniforms, a.rng, a.rng_offset = L.ptr(kw.get('uniforms')), L.ptr(self.rng), t
            if kw.get('save', False):
                a.sv_xin, a.sv_sh, a.sv_gates = L.ptr(self.sv_xin[t]), L.ptr(self.sv_sh[t]), L.ptr(self.sv_gates[t])
                a.sv_enc = L.ptr(None if self.sv_enc is None else self.sv_enc[t])
            if self.kernel_events is not None:
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
            L.check(L.lib().nmarl_policy_step_p(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_policy_step_p')
            if self.kernel_events is not None:
                ev[1].record()
                self.kernel_events.append(ev)
        else:
            a.c_in, a.h_in, a.msg_in = L.ptr(self.c_seq[t + 1]), L.ptr(self.h_seq[t + 1]), L.ptr(None if ms is None else ms[t + 1])
            a.act_in, a.v = L.ptr(kw['act']), L.ptr(kw['v'])
            L.check(L.lib().nmarl_policy_step_v(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_policy_step_v')
        self.launches += 1

    def _rollout_saved(self, env, mode, uniforms, T):
        self.h_seq[0].copy_(self.h[self.cur]); self.c_seq[0].copy_(self.c[self.cur])
        if self.msg_seq is not None:
            self.msg_seq[0].copy_(self.msg[self.cur])
        main = torch.cuda.current_stream()
        if self.overlap_v and self._vstream is None:
            self._vstream = torch.cuda.Stream(device=self.device)
        side = self._vstream if self.overlap_v else None

        def v_call(t, obs, fp, done, act, v):
            # Reads obs/fp/done[t], act and state slot t+1; writes only v.  Nothing downstream in the rollout
            # reads v, so on the second stream it fills the SMs the 256-CTA p-call / env step leave idle.
            if side is None:
                self._seq_call(t, obs, fp, done, 'v', act=act, v=v)
                return
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self._seq_call(t, obs, fp, done, 'v', act=act, v=v)

        for t in range(T):
            obs, fp, done = self.obs_buf[t], self.fp_buf[t], self.done_buf[t]
            self._seq_call(t, obs, fp, done, 'p', pi=self.fp_buf[t + 1], action=self.act_buf[t], mode=mode,
                           uniforms=None if uniforms is None else uniforms[t], save=True)
            v_call(t, obs, fp, done, self.act_buf[t], self.val_buf[t])
            env.step_device(self.act_buf[t], obs_out=self.obs_buf[t + 1], reward_out=self.rew_buf[t],
                            greward_out=self.grew_buf[t], done_out=self.done_buf[t + 1])
            self.launches += 1
        # bootstrap (Q2): one more p-call (state advanced into slot T+1, not saved for BPTT) + v-call
        self._seq_call(T, self.obs_buf[T], self.fp_buf[T], self.done_buf[T], 'p', pi=self.boot_pi, action=self.boot_act,
                       mode=mode, uniforms=None if uniforms is None else uniforms[T])
        v_call(T, self.obs_buf[T], self.fp_buf[T], self.done_buf[T], self.boot_act, self.R_end)
        if side is not None:
            main.wait_stream(side)
        self.h[self.cur].copy_(self.h_seq[T + 1]); self.c[self.cur].copy_(self.c_seq[T + 1])
        if self.msg_seq is not None:
            self.msg[self.cur].copy_(self.msg_seq[T + 1])
        if mode == L.SAMPLE_PHILOX:
            L.check(L.lib().nmarl_rng_advance(L.ptr(self.rng), T + 1, L.stream()), 'nmarl_rng_advance')
            self.launches += 1

    def roll_buffers(self):
        """Slot T becomes slot 0 of the next batch (obs, fingerprint, pre-step done)."""
        T = self.T_cur
        self.obs_buf[0].copy_(self.obs_buf[T]); self.fp_buf[0].copy_(self.fp_buf[T]); self.done_buf[0].copy_(self.done_buf[T])

    def compute_returns(self):
        """R_end is zeroed where the batch ended with done (utils.py:192-193)."""
        T = self.T_cur
        h = self.hp
        L.check(L.lib().nmarl_nstep_return_adv(self.N, self.B, T, self.NR, L.ptr(self.rew_buf), L.ptr(self.val_buf),
                                               L.ptr(self.done_buf[1:]), L.ptr(self.R_end), 1, float(h['gamma']),
                                               float(h['reward_norm']), float(h['reward_clip']), self.alpha,
                                               L.ptr(self.dist_dev), L.ptr(self.alpha_pow),
                                               0 if self.alpha_pow is None else self.alpha_pow.numel(),
                                               L.ptr(self.Rs), L.ptr(self.Advs), L.stream()), 'nmarl_nstep_return_adv')
        self.launches += 1
        if getattr(self.layout, 'hetero', False):
            # Reference quirk Q7 (agents/policies.py:241-251, non-identical branch): prob_pi [N,1,T] * ADV [N,T]
            # broadcasts to [N,N,T], so agent i's log-probability is weighted by the SUM over agents of the
            # advantages.  Reproduced for parity with the reference's heterogeneous-agent path.
            self.Advs[:T] = self.Advs[:T].sum(dim=1, keepdim=True).expand(-1, self.N, -1)

    # ---- training -------------------------------------------------------------------------------------
    def _alloc_train(self):
        if self._train_ready:
            return
        lay, N, B, T, dev = self.layout, self.N, self.B, self.T, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        z = lambda *s: torch.zeros(*s, **f32)
        self.h_seq, self.c_seq = z(T + 2, *self._sshape), z(T + 2, *self._sshape)       # +1 slot for the bootstrap p-call
        self.msg_seq = z(T + 2, N, B, NH) if self.variant == 'ma2c_dial' else None
        self.sv_xin = z(T, N, B, lay.ld_in)
        self.sv_sh = z(T, N, B, lay.s_dim + NH)
        self.sv_gates = z(T, N, B, 4 * NH)
        self.sv_enc = z(T, N, B, 128) if self.variant in ('ma2c_ic3', 'ma2c_dial') else None
        self.sv_dlv = z(T, N, B, 8)
        # tensor-core path: sv_dz holds per-tile gate-bias partial sums, sv_dpre is unused (operand tiles instead)
        self.sv_dz = z(T, N, B // 128, 4 * NH) if self.use_tc else z(T, N, B, 4 * NH)
        self.sv_dpre = z(4) if self.use_tc else z(T, N, B, 192)
        # tensor-core path: dz / encoder pre-activation gradients additionally as K-major raw fp32 operand tiles
        ndp = {'ma2c_nc': 192, 'ia2c': 64}.get(self.variant, 128)
        self.sv_dzT = z(T, N, B // 32, 256 * 32) if self.use_tc else None
        self.sv_dpT = z(T, N, B // 32, ndp * 32) if self.use_tc else None
        self.sv_dmp = z(T, N, B, NH) if self.variant == 'ma2c_dial' else None
        self.dh_rec, self.dc_rec = z(2, *self._sshape), z(2, *self._sshape)
        self.dmsg = z(2, N, L.MAX_NBR, *self._sshape[1:]) if self.variant != 'ia2c' else None
        self.ws_floats = int(L.lib().nmarl_ws_floats(C.byref(self.model), B, T))
        self.ws = z(max(self.ws_floats, 4))
        self.tiles = int(L.lib().nmarl_loss_tiles(C.byref(self.model), B))
        self.loss_part = z(T, N, self.tiles, 4)
        self._train_ready = True

    def _bwd_args(self, T):
        self._alloc_train()
        a = L.BwdArgs()
        a.B, a.T, a.B_total = self.B, T, self.B * self.world
        a.v_coef, a.e_coef = float(self.hp['v_coef']), float(self.hp['e_coef'])
        a.params, a.obs, a.act = L.ptr(self.params), L.ptr(self.obs_buf), L.ptr(self.act_buf)
        a.fp = L.ptr(self.fp_buf) if self.variant in ('ma2c_nc', 'ma2c_dial') else None
        a.done_pre, a.Rs, a.Advs = L.ptr(self.done_buf), L.ptr(self.Rs), L.ptr(self.Advs)
        a.h_seq, a.c_seq, a.msg_seq = L.ptr(self.h_seq), L.ptr(self.c_seq), L.ptr(self.msg_seq)
        a.sv_xin, a.sv_sh, a.sv_gates, a.sv_enc = L.ptr(self.sv_xin), L.ptr(self.sv_sh), L.ptr(self.sv_gates), L.ptr(self.sv_enc)
        a.sv_dlv, a.sv_dz, a.sv_dpre, a.sv_dmp = L.ptr(self.sv_dlv), L.ptr(self.sv_dz), L.ptr(self.sv_dpre), L.ptr(self.sv_dmp)
        a.dh_rec, a.dc_rec, a.dmsg = L.ptr(self.dh_rec), L.ptr(self.dc_rec), L.ptr(self.dmsg)
        a.wt, a.ws, a.ws_floats = L.ptr(self.wt), L.ptr(self.ws), self.ws_floats
        a.loss_part, a.grads = L.ptr(self.loss_part), L.ptr(self.grads)
        a.wpack, a.tc_err = L.ptr(self.wpack), L.ptr(self.tc_err)
        a.sv_dzT, a.sv_dpT = L.ptr(self.sv_dzT), L.ptr(self.sv_dpT)
        a.state_fm = int(self.state_fm)
        a.ctx = self._ctx
        if self.bwd_events is not None:
            step_ev, wg_ev = self.bwd_events
            self._ev_arrays = ((C.c_void_p * len(step_ev))(*[ev.cuda_event for ev in step_ev]),
                               (C.c_void_p * 2)(*[ev.cuda_event for ev in wg_ev]))
            a.ev_step = C.cast(self._ev_arrays[0], C.c_void_p)
            a.ev_wgrad = C.cast(self._ev_arrays[1], C.c_void_p)
        return a

    def backward(self):
        """Training forward from states_bw + loss + BPTT + weight gradients -> self.grads
        (local sum over this rank's envs, already scaled by 1/(T * B_total))."""
        T = self.T_cur
        a = self._bwd_args(T)
        if getattr(self, 'saved_rollout', False):
            # activations, h_seq / c_seq (slot 0 == states_bw) were written by the rollout p-calls
            a.fused_heads = 1        # heads / loss kernel folded into the BPTT call (side stream, beside the first steps)
            L.check(L.lib().nmarl_a2c_bptt(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_a2c_bptt')
            self.launches += 2 * T + 16
            self.saved_rollout = False
            return
        self.h_seq[0].copy_(self.h_bw); self.c_seq[0].copy_(self.c_bw)
        if self.variant == 'ma2c_dial':
            L.check(L.lib().nmarl_dial_msg(C.byref(self.model), self.B, L.ptr(self.params), L.ptr(self.h_seq[0]),
                                           L.ptr(self.msg_seq[0]), L.stream()), 'nmarl_dial_msg')
        L.check(L.lib().nmarl_a2c_backward(C.byref(self.model), C.byref(a), L.stream()), 'nmarl_a2c_backward')
        self.launches += 2 * T + 16

    def apply(self, lr):
        """[all-reduce] -> global-norm clip -> RMSProp; then states_bw := states_fw."""
        if isinstance(lr, torch.Tensor):
            if lr is not self.lr_dev:
                self.lr_dev.copy_(lr)
        else:
            self.lr_dev.fill_(float(lr))
        if self.world > 1:
            torch.distributed.all_reduce(self.grads, op=torch.distributed.ReduceOp.SUM, group=self.group)
        h = self.hp
        L.check(L.lib().nmarl_clip_rmsprop_step(C.byref(self.model), L.ptr(self.params), L.ptr(self.grads), L.ptr(self.ms),
                                                L.ptr(self.lr_dev), float(h['max_grad_norm']), float(h['alpha']),
                                                float(h['epsilon']), L.ptr(self.norm_out), L.ptr(self.opt_scratch),
                                                L.stream()), 'nmarl_clip_rmsprop_step')
        self.launches += 2
        if self.agent_name == 'ma2c_cu':     # ConsensusPolicy.backward: sess.run(_consensus_update) after the optimizer
            if getattr(self, '_cu_scratch', None) is None:
                self._cu_scratch = torch.zeros(self.N * ((self.layout.s_dim + NH) * 4 * NH + 4 * NH),
                                               dtype=torch.float32, device=self.device)
            L.check(L.lib().nmarl_consensus_update(C.byref(self.model), L.ptr(self.params), L.ptr(self._cu_scratch),
                                                   L.stream()), 'nmarl_consensus_update')
            self.launches += 2
        self.c_bw.copy_(self.c[self.cur]); self.h_bw.copy_(self.h[self.cur])
        self.repack()
        self._refresh_msg()        # DIAL: cached sender-side messages depend on the updated w_mfc

    def update(self, lr):
        self.compute_returns()
        self.backward()
        self.apply(lr)

    def losses(self):
        """Per-agent (policy, value, entropy) loss terms of the last backward, reference weighting
        (policies.py:252-254).  Host sync."""
        T = self.T_cur
        lp = self.loss_part[:T].double().sum(dim=(0, 2)).cpu().numpy()       # [N,4]
        n = float(T * self.B)
        h = self.hp
        return dict(policy_loss=lp[:, 0] / n, value_loss=lp[:, 1] / n * 0.5 * h['v_coef'],
                    entropy_loss=-lp[:, 2] / n * h['e_coef'])
