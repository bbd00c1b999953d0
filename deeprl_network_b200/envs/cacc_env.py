"""CACC platoon environment, vectorised over B parallel episodes on the GPU.

Host-side mirror of the reference ``CACCEnv`` (envs/cacc_env.py): same constructor argument
(the ``ENV_CONFIG`` section), same methods and attributes (SURVEY 8b), so ``Trainer`` /
``main.py`` drive it unchanged.  With ``n_env == 1`` every call has the reference semantics
(seed stepping, test-episode seeds, fingerprints, IA2C observation concatenation).  The state
lives in device memory as float64 [agent][env] arrays and is advanced by the ``nmarl_cacc_*``
kernels (csrc/env.cu); ``*_device`` methods expose the batched tensors without host copies.

New optional keys in ``ENV_CONFIG`` (everything else parses exactly like the reference):
  n_env        parallel episodes on this process (default 1)
  platoon_len  vehicles per platoon (default n_vehicle); < n_vehicle gives several independent
               platoons -- used only by the synthetic 5x5-grid configuration
  topology     'chain' (default) or 'grid' (row-major 4-neighbour grid, Manhattan distance)
"""
import ctypes as C
import logging

import numpy as np
import torch

from .. import _lib as L


def chain_masks(n):
    """Chain adjacency and |i-j| distances (envs/cacc_env.py:253-267)."""
    nb = np.zeros((n, n), dtype=int)
    idx = np.arange(n)
    nb[idx[1:], idx[:-1]] = 1
    nb[idx[:-1], idx[1:]] = 1
    return nb, np.abs(idx[:, None] - idx[None, :]).astype(int)


def grid_masks(side):
    """4-neighbour side x side grid in row-major order with Manhattan distances -- equals the
    large-grid adjacency/distance of envs/large_grid_env.py:58-105 (SURVEY 8d, cfg5)."""
    n = side * side
    r, c = np.divmod(np.arange(n), side)
    dist = (np.abs(r[:, None] - r[None, :]) + np.abs(c[:, None] - c[None, :])).astype(int)
    return (dist == 1).astype(int), dist


def seed_uniforms(seeds, n_platoon):
    """float64 [P, B]: column k holds the uniforms ``CACCEnv.reset(test_ind=k)`` draws for test seed ``seeds[k]``
    (``np.random.seed(seed)``, then one ``rand()`` per platoon in order).  A private RandomState gives the same
    values as the legacy global seeding and leaves the global NumPy stream untouched."""
    out = np.empty((int(n_platoon), len(seeds)), dtype=np.float64)
    for k, s in enumerate(seeds):
        out[:, k] = np.random.RandomState(int(s)).rand(int(n_platoon))
    return out


def control_row(episode, t, dt, action, global_reward):
    """One row of ``{scenario}_{agent}_control.csv`` (envs/cacc_env.py:81-137): step t of an episode."""
    return {'episode': episode, 'time_sec': t * dt, 'step': t,
            'action': ','.join(['%d' % a for a in action]), 'reward': global_reward}


def traffic_frame(episode, dt, rewards, trace, n_agent):
    """The ``_traffic.csv`` block of one episode.  rewards: [0] + the per-step global rewards; trace float64
    [steps + 1, 3, N] = (h, v, u) of every vehicle, the reset state first."""
    import pandas as pd
    tr = np.asarray(trace)
    hs, vs, us = tr[:, 0], tr[:, 1], tr[:, 2]
    df = pd.DataFrame()
    df['episode'] = np.ones(len(hs)) * episode
    df['time_sec'] = np.arange(len(hs)) * dt
    df['reward'] = np.array(rewards)
    df['lead_headway_m'] = hs[:, 0]
    df['avg_headway_m'] = np.mean(hs[:, 1:], axis=1)
    df['std_headway_m'] = np.std(hs[:, 1:], axis=1)
    df['avg_speed_mps'] = np.mean(vs, axis=1)
    df['std_speed_mps'] = np.std(vs, axis=1)
    df['avg_accel_mps2'] = np.mean(us, axis=1)
    df['std_accel_mps2'] = np.std(us, axis=1)
    for i in range(n_agent):
        df['headway_%d_m' % (i + 1)] = hs[:, i]
        df['velocity_%d_mps' % (i + 1)] = vs[:, i]
        df['accel_%d_mps2' % (i + 1)] = us[:, i]
    return df


class CACCEnv:
    def __init__(self, config, n_env=None, device=None):
        L.require_cuda()
        self.config = config
        self._load_config(config)
        if n_env is not None:
            self.n_env = int(n_env)
        self.device = torch.device(device if device is not None else 'cuda:%d' % torch.cuda.current_device())
        self.train_mode = True
        self.cur_episode = 0
        self.is_record = False
        self._init_space()
        self._alloc()
        # "required to achieve the same model initialization" (envs/cacc_env.py:21-22)
        np.random.seed(self.seed)

    # ---- configuration (envs/cacc_env.py:320-343) ---------------------------------------------
    def _load_config(self, config):
        self.dt = config.getfloat('control_interval_sec')
        self.T = int(config.getint('episode_length_sec') / self.dt)
        self.batch_size = config.getint('batch_size')
        self.h_min = config.getfloat('headway_min')
        self.h_star = config.getfloat('headway_target')
        self.h_norm = config.getfloat('norm_headway')
        self.h_s = config.getfloat('headway_st')
        self.h_g = config.getfloat('headway_go')
        self.v_max = config.getfloat('speed_max')
        self.v_star = config.getfloat('speed_target')
        self.v_norm = config.getfloat('norm_speed')
        self.u_min = config.getfloat('accel_min')
        self.u_max = config.getfloat('accel_max')
        self.name = config.get('scenario').split('_')[1]
        self.a = config.getfloat('reward_v')
        self.b = config.getfloat('reward_u')
        self.G = config.getfloat('collision_penalty')
        self.n_agent = config.getint('n_vehicle')
        self.agent = config.get('agent')
        self.coop_gamma = config.getfloat('coop_gamma')
        self.seed = config.getint('seed')
        self.init_test_seeds([int(s) for s in config.get('test_seeds').split(',')])
        self.n_env = config.getint('n_env', fallback=1)
        self.platoon_len = config.getint('platoon_len', fallback=self.n_agent)
        self.topology = config.get('topology', fallback='chain')
        if not (self.name.startswith('catchup') or self.name.startswith('slowdown')):
            raise ValueError('unknown CACC scenario %r' % self.name)

    def _init_space(self):
        if self.topology == 'grid':
            side = int(round(self.n_agent ** 0.5))
            assert side * side == self.n_agent, 'grid topology needs a square agent count'
            self.neighbor_mask, self.distance_mask = grid_masks(side)
        else:
            self.neighbor_mask, self.distance_mask = chain_masks(self.n_agent)
        self.n_a = 4
        self.n_a_ls = [4] * self.n_agent
        self.a_map = [(0, 0), (0.5, 0), (0, 0.5), (0.5, 0.5)]
        logging.info('action to h_go map:\n %r' % self.a_map)
        self.nbr = [np.where(self.neighbor_mask[i] == 1)[0] for i in range(self.n_agent)]
        self.n_s_ls = [5 * (1 if self.agent.startswith('ma2c') else 1 + len(self.nbr[i]))
                       for i in range(self.n_agent)]

    def _alloc(self):
        N, B, dev = self.n_agent, self.n_env, self.device
        P = N // self.platoon_len
        f64 = dict(dtype=torch.float64, device=dev)
        self.hs, self.vs, self.us = (torch.zeros(N, B, **f64) for _ in range(3))
        self.v_init = torch.zeros(P, B, **f64)
        self.t_dev = torch.zeros(B, dtype=torch.int32, device=dev)
        self.collision_dev = torch.zeros(B, dtype=torch.int32, device=dev)
        self.episode_dev = torch.zeros(B, dtype=torch.int32, device=dev)
        self.obs_stride = 8
        self.obs_dev = torch.zeros(N, B, self.obs_stride, dtype=torch.float32, device=dev)
        self.fp_dev = torch.full((N, B, self.n_a), 1.0 / self.n_a, dtype=torch.float32, device=dev)
        self.NR = 1 if self.coop_gamma < 0 else N
        self.reward_dev = torch.zeros(self.NR, B, **f64)
        self.greward_dev = torch.zeros(B, **f64)
        self.done_dev = torch.zeros(B, dtype=torch.float32, device=dev)
        self._action_dev = torch.zeros(N, B, dtype=torch.int32, device=dev)
        self._u01 = torch.zeros(P, B, **f64)
        self._mask0 = torch.zeros(B, dtype=torch.float32, device=dev)
        self._mask0[0] = 1.0
        c = L.CaccCfg()
        c.n_agent, c.platoon_len = N, self.platoon_len
        c.scenario = L.CATCHUP if self.name.startswith('catchup') else L.SLOWDOWN
        c.T, c.batch_size, c.global_reward = self.T, self.batch_size, int(self.coop_gamma < 0)
        c.dt, c.h_min, c.h_star, c.h_s, c.h_g = self.dt, self.h_min, self.h_star, self.h_s, self.h_g
        c.v_max, c.v_star, c.u_min, c.u_max = self.v_max, self.v_star, self.u_min, self.u_max
        c.rew_a, c.rew_b, c.G = self.a, self.b, self.G
        self.cfg = c
        self.collision = False
        self.t = 0

    # ---- device-side API (no host copies) --------------------------------------------------------
    def reset_device(self, u01=None, mask=None, obs_out=None, fp_out=None, philox_seed=None):
        """Reset envs (all, or those with mask != 0).  u01: double [P,B] tensor or None (Philox keyed
        by (seed, env, episode counter))."""
        obs = self.obs_dev if obs_out is None else obs_out
        fp = self.fp_dev if fp_out is None else fp_out
        seed = int(self.cfg_seed if philox_seed is None else philox_seed) & (2 ** 64 - 1)
        L.check(L.lib().nmarl_cacc_reset(C.byref(self.cfg), self.n_env, L.ptr(u01), L.ptr(mask), seed,
                                         L.ptr(self.episode_dev), L.ptr(self.hs), L.ptr(self.vs), L.ptr(self.us),
                                         L.ptr(self.t_dev), L.ptr(self.collision_dev), L.ptr(self.v_init),
                                         L.ptr(obs), obs.shape[-1], L.ptr(fp), self.n_a, L.stream()), 'nmarl_cacc_reset')

    def step_device(self, action, obs_out=None, reward_out=None, greward_out=None, done_out=None):
        """action int32 [N,B] device tensor.  Outputs default to the env's own buffers."""
        obs = self.obs_dev if obs_out is None else obs_out
        rew = self.reward_dev if reward_out is None else reward_out
        grew = self.greward_dev if greward_out is None else greward_out
        done = self.done_dev if done_out is None else done_out
        L.check(L.lib().nmarl_cacc_step(C.byref(self.cfg), self.n_env, int(self.train_mode), L.ptr(action),
                                        L.ptr(self.hs), L.ptr(self.vs), L.ptr(self.us), L.ptr(self.t_dev),
                                        L.ptr(self.collision_dev), L.ptr(self.v_init), L.ptr(obs), obs.shape[-1],
                                        L.ptr(rew), L.ptr(grew), L.ptr(done), L.stream()), 'nmarl_cacc_step')

    def reset_seeds(self, seeds, obs_out=None, fp_out=None):
        """Test-mode reset of all B envs in one launch: env k starts the episode ``reset(test_ind)`` would start for
        test seed ``seeds[k]`` (same uniforms, see ``seed_uniforms``).  Sets ``train_mode = False``."""
        seeds = [int(s) for s in seeds]
        if len(seeds) != self.n_env:
            raise ValueError('reset_seeds: %d seeds for %d envs' % (len(seeds), self.n_env))
        self._u01.copy_(torch.from_numpy(seed_uniforms(seeds, self._u01.shape[0])))
        self.train_mode = False
        self.reset_device(u01=self._u01, obs_out=obs_out, fp_out=fp_out)
        self.collision = False
        self.t = 0

    @property
    def cfg_seed(self):
        return getattr(self, '_cfg_seed', 0)

    # ---- reference API (host arrays, env 0 is "the" environment) -----------------------------------
    def _host_obs(self):
        base = self.obs_dev[:, 0, :5].double().cpu().numpy()
        if not self.agent.startswith('ia2c'):
            return [base[i] for i in range(self.n_agent)]
        # ia2c_fp: neighbour fingerprints are attached at the end of the state array (cacc_env.py:74-77)
        fps = (lambda i: [np.asarray(self.fp[j], dtype=np.float64) for j in self.nbr[i]]) if self.agent == 'ia2c_fp' else (lambda i: [])
        return [np.concatenate([base[i]] + [base[j] for j in self.nbr[i]] + fps(i)) for i in range(self.n_agent)]

    def reset(self, gui=False, test_ind=-1):
        """envs/cacc_env.py:166-189: seed selection, np.random.seed, ``seed += 1`` on every reset;
        one np.random.rand() drives the initial condition of env 0.  Envs b>0 (n_env > 1) draw
        their uniform from Philox keyed by (seed used, env, episode)."""
        self.cur_episode += 1
        if self.train_mode:
            seed = self.seed
        elif test_ind < 0:
            seed = self.seed - 1
        else:
            seed = self.test_seeds[test_ind]
        np.random.seed(seed)
        self.seed += 1
        # NB the reference tests the already-incremented attribute (cacc_env.py:290,311); the only
        # config seed reaching the deterministic branch (-1) is rejected by np.random.seed above.
        u = np.random.rand()
        if self.n_env > 1:
            self.reset_device(u01=None, philox_seed=seed)
            self.episode_dev[0] -= 1          # env 0 is reset again below; count its episode once
        # env 0: the reference's single np.random.rand(); further platoons (grid stub only) draw their own
        self._u01[:, 0] = torch.as_tensor([u] + [np.random.rand() for _ in range(self._u01.shape[0] - 1)],
                                          dtype=torch.float64)
        self.reset_device(u01=self._u01, mask=self._mask0)
        self.collision = False
        self.t = 0
        self.fp = np.ones((self.n_agent, self.n_a)) / self.n_a
        self.rewards = [0]
        if self.is_record:                       # the traffic log starts with the reset state (cacc_env.py:183-188)
            self._trace = [torch.stack([self.hs[:, 0], self.vs[:, 0], self.us[:, 0]]).cpu().numpy()]
        return self._host_obs()

    def step(self, action):
        """envs/cacc_env.py:191-242 for env 0 (all envs take the same action vector when n_env > 1)."""
        a = torch.as_tensor(np.asarray(action, dtype=np.int32)).to(self.device)
        self._action_dev.copy_(a[:, None].expand(-1, self.n_env))
        self.step_device(self._action_dev)
        out = torch.cat([self.reward_dev[:, 0], self.greward_dev[:1], self.done_dev[:1].double(),
                         self.collision_dev[:1].double()]).cpu().numpy()
        reward = out[0] if self.NR == 1 else out[:self.NR].copy()
        global_reward, done = out[self.NR], bool(out[self.NR + 1])
        self.collision = bool(out[self.NR + 2])
        self.t += 1
        self.rewards.append(global_reward)
        ob = self._host_obs()
        if self.is_record:
            self._log_control_data(action, global_reward)
            self._record_step()
            if done:
                self._log_traffic_data()
        return ob, reward, done, global_reward

    def get_fingerprint(self):
        return self.fp

    def update_fingerprint(self, fp):
        self.fp = fp

    def get_neighbor_action(self, action):
        action = np.asarray(action)
        return [action[self.neighbor_mask[i] == 1] for i in range(self.n_agent)]

    def terminate(self):
        return

    def collect_tripinfo(self):
        return

    def init_test_seeds(self, test_seeds):
        self.test_num = len(test_seeds)
        self.test_seeds = test_seeds

    # ---- evaluation records (envs/cacc_env.py:81-137) -------------------------------------------------
    def init_data(self, is_record, record_stats, output_path):
        self.is_record = is_record
        self.output_path = output_path
        if self.is_record:
            self.control_data = []
            self.traffic_data = []
            self._trace = []

    def _record_step(self):
        self._trace.append(torch.stack([self.hs[:, 0], self.vs[:, 0], self.us[:, 0]]).cpu().numpy())

    def _log_control_data(self, action, global_reward):
        self.control_data.append(control_row(self.cur_episode, self.t, self.dt, action, global_reward))

    def _log_traffic_data(self):
        self.traffic_data.append(traffic_frame(self.cur_episode, self.dt, self.rewards, np.array(self._trace),
                                               self.n_agent))

    def record_episode(self, episode, actions, global_rewards, trace):
        """Append one finished episode recorded elsewhere (the batched evaluator) to the same records the
        step-by-step path builds.  actions [steps, N], global_rewards float64 [steps], trace float64
        [steps + 1, 3, N] with the reset state first."""
        for s in range(len(global_rewards)):
            self.control_data.append(control_row(episode, s + 1, self.dt, actions[s], global_rewards[s]))
        self.traffic_data.append(traffic_frame(episode, self.dt, [0] + list(global_rewards), trace, self.n_agent))

    def output_data(self):
        import pandas as pd
        if not self.is_record:
            logging.error('Env: no record to output!')
            return
        pd.DataFrame(self.control_data).to_csv(self.output_path + ('%s_%s_control.csv' % (self.name, self.agent)))
        pd.concat(self.traffic_data).to_csv(self.output_path + ('%s_%s_traffic.csv' % (self.name, self.agent)))
