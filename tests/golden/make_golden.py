"""Generate golden fixtures by running the UNMODIFIED reference code.

Run in the authoring container only (needs /root/reference):
    python tests/golden/make_golden.py
Writes tests/golden/env_*.npz and tests/golden/buffer_*.npz.  The fixtures are
committed; nothing at test/bench time reads /root/reference.

Reference pieces executed here:
  * envs/cacc_env.py  CACCEnv            (imports cleanly)
  * agents/utils.py   OnPolicyBuffer, MultiAgentOnPolicyBuffer, Scheduler
    (imported with a stub `tensorflow` module: the file only needs tf.nn.relu
     as a default argument at import time -- SURVEY 8c)
"""
import configparser
import glob
import hashlib
import json
import os
import sys
import types

import numpy as np

REF = '/root/reference'
HERE = os.path.dirname(os.path.abspath(__file__))


def _import_reference():
    sys.path.insert(0, REF)
    tf = types.ModuleType('tensorflow')
    tf.nn = types.SimpleNamespace(relu=None)
    sys.modules['tensorflow'] = tf
    if not hasattr(np, 'bool'):
        np.bool = bool  # reference uses the removed alias (agents/utils.py:759,833)
    from envs.cacc_env import CACCEnv
    import agents.utils as au
    return CACCEnv, au


def _cfg(name, **over):
    cp = configparser.ConfigParser()
    cp.read(os.path.join(REF, 'config', name))
    for k, v in over.items():
        cp['ENV_CONFIG'][k] = str(v)
    return cp


def _actions(kind, T, n, seed=0):
    if kind == 'const3':
        return np.full((T, n), 3, dtype=np.int32)
    if kind == 'const0':
        return np.zeros((T, n), dtype=np.int32)
    if kind == 'const1':
        return np.full((T, n), 1, dtype=np.int32)
    if kind == 'cyc':
        t = np.arange(T)[:, None]
        i = np.arange(n)[None, :]
        return ((t + i) % 4).astype(np.int32)
    if kind == 'rand':
        return np.random.RandomState(seed).randint(0, 4, size=(T, n)).astype(np.int32)
    raise ValueError(kind)


def env_case(CACCEnv, ini, kind, test_mode=False, n_reset=1, fp_seed=None, **over):
    cp = _cfg(ini, **over)
    env = CACCEnv(cp['ENV_CONFIG'])
    eps = []
    for ep in range(n_reset):
        if test_mode:
            # mimic Trainer.run: a train reset precedes the interleaved test episode
            env.train_mode = True
            env.reset()
            env.train_mode = False
            ob = env.reset(test_ind=-1)
        else:
            ob = env.reset()
        seed_after = env.seed
        h0 = np.array(env.hs_cur, dtype=np.float64)
        v0 = np.array(env.vs_cur, dtype=np.float64)
        acts = _actions(kind, env.T, env.n_agent, seed=100 + ep)
        obs = [np.concatenate([np.asarray(o, dtype=np.float64) for o in ob])]
        rews, dones, greps, hs, vs, us, fps = [], [], [], [], [], [], []
        nstep = 0
        fp_rs = None if fp_seed is None else np.random.RandomState(fp_seed + ep)
        for t in range(env.T):
            if fp_rs is not None:
                # what Trainer.explore does before every step (utils.py:173): fingerprints = the policies just computed
                fp = fp_rs.dirichlet(np.ones(env.n_a), size=env.n_agent)
                env.update_fingerprint(fp)
                fps.append(fp)
            ob, r, d, g = env.step(acts[t])
            obs.append(np.concatenate([np.asarray(o, dtype=np.float64) for o in ob]))
            rews.append(np.broadcast_to(np.asarray(r, dtype=np.float64), (env.n_agent,)).copy())
            dones.append(d)
            greps.append(g)
            hs.append(np.array(env.hs_cur)); vs.append(np.array(env.vs_cur)); us.append(np.array(env.us_cur))
            nstep += 1
            if d:
                break
        eps.append(dict(h0=h0, v0=v0, seed_after=seed_after, acts=acts[:nstep], obs=np.array(obs),
                        rew=np.array(rews), done=np.array(dones), greward=np.array(greps),
                        hs=np.array(hs), vs=np.array(vs), us=np.array(us),
                        v0s=np.array(env.v0s), **({} if fp_rs is None else dict(fps=np.array(fps)))))
    out = {}
    for k, ep in enumerate(eps):
        for key, val in ep.items():
            out['ep%d_%s' % (k, key)] = val
    out['n_ep'] = len(eps)
    out['ini'] = ini
    out['kind'] = kind
    out['test_mode'] = test_mode
    out['over'] = repr(over)
    return out


def buffer_case(au, alpha, multi=True, T=60, n=8, seed=0):
    rs = np.random.RandomState(seed)
    dist = np.abs(np.arange(n)[:, None] - np.arange(n)[None, :])
    gamma = 0.99
    out = {}
    if multi:
        buf = au.MultiAgentOnPolicyBuffer(gamma, alpha, dist)
        rec = dict(r=[], v=[], done=[])
        for t in range(T):
            r = rs.randn() if alpha < 0 else rs.randn(n)
            ob = rs.randn(n, 5); p = rs.rand(n, 4); a = rs.randint(0, 4, n); v = rs.randn(n)
            done = (t == 29)  # a mid-batch terminal to exercise the (1-done) path
            buf.add_transition(ob, p, a, r, v, done)
            rec['r'].append(np.broadcast_to(np.asarray(r, dtype=np.float64), (n,)).copy())
            rec['v'].append(v); rec['done'].append(done)
        R_end = rs.randn(n)
        obs, ps, acts, dones, Rs, Advs = buf.sample_transition(R_end)
        out.update(obs=obs, ps=ps, acts=acts, dones_pre=dones, Rs=Rs, Advs=Advs, R_end=R_end,
                   r=np.array(rec['r']), v=np.array(rec['v']), done_post=np.array(rec['done']),
                   alpha=alpha, gamma=gamma, dist=dist)
    else:
        # IA2C: one OnPolicyBuffer per agent (models.py:153-158), shared reward object
        bufs = [au.OnPolicyBuffer(gamma, alpha, dist[i]) for i in range(n)]
        rec = dict(r=[], v=[], done=[])
        for t in range(T):
            r = rs.randn() if alpha < 0 else rs.randn(n)
            v = rs.randn(n)
            done = (t == 29)
            for i in range(n):
                bufs[i].add_transition(rs.randn(10), rs.randint(0, 4, 2), rs.randint(0, 4), r, v[i], done)
            rec['r'].append(np.broadcast_to(np.asarray(r, dtype=np.float64), (n,)).copy())
            rec['v'].append(v); rec['done'].append(done)
        R_end = rs.randn(n)
        Rs, Advs = [], []
        for i in range(n):
            _, _, _, dones, R, A = bufs[i].sample_transition(R_end[i])
            Rs.append(R); Advs.append(A)
        out.update(Rs=np.array(Rs), Advs=np.array(Advs), R_end=R_end, dones_pre=dones,
                   r=np.array(rec['r']), v=np.array(rec['v']), done_post=np.array(rec['done']),
                   alpha=alpha, gamma=gamma, dist=dist)
    return out


def eval_case(CACCEnv, ini, kind, out_prefix):
    """Evaluator-style recorded test episode (utils.py:321-336 + cacc_env.py:81-137): the reference's own CSVs."""
    cp = _cfg(ini)
    env = CACCEnv(cp['ENV_CONFIG'])
    env.init_test_seeds([2000])
    env.train_mode = False
    env.cur_episode = 0
    env.init_data(True, False, out_prefix)
    env.reset(test_ind=0)
    acts = _actions(kind, env.T, env.n_agent)
    for t in range(env.T):
        _, _, d, _ = env.step(acts[t])
        if d:
            break
    env.output_data()
    return acts[:t + 1]


def trainer_case(CACCEnv, ini, total_step):
    """The UNMODIFIED reference Trainer + Counter + CACCEnv driving a scripted agent (tests/helpers.py
    ScriptedAgent): the trace of every agent call pins the rollout control flow (utils.py:129-254, quirks Q1-Q6)."""
    import tempfile
    tf = sys.modules['tensorflow']
    tf.float32 = 'float32'
    tf.placeholder = lambda *a, **k: object()
    tf.summary = types.SimpleNamespace(scalar=lambda *a, **k: object())
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import ScriptedAgent
    import utils as ref_utils
    cp = _cfg(ini)
    env = CACCEnv(cp['ENV_CONFIG'])
    agent = ScriptedAgent(env.agent, env.n_agent, env.n_a, cp['MODEL_CONFIG'].getint('batch_size'))
    writer = types.SimpleNamespace(add_summary=lambda *a, **k: None, flush=lambda: None)
    counter = ref_utils.Counter(total_step, 10 ** 9, 10 ** 9)
    out_dir = tempfile.mkdtemp() + '/'
    tr = ref_utils.Trainer(env, agent, counter, writer, output_path=out_dir)
    tr.run()
    data = np.array([[d['step'], d['avg_reward'], d['std_reward']] for d in tr.data])
    return dict(trace=np.array(agent.trace), data=data, seed_after=env.seed, cur_step=counter.cur_step,
                ini=ini, total_step=total_step)


def agent_case(CACCEnv, ini, total_step):
    """The UNMODIFIED reference agent class (IA2C / IA2C_FP / MA2C_*: reward scaling, buffers, returns, lr schedule,
    argument marshalling -- agents/models.py) inside the reference Trainer, with only the TF policy objects replaced
    by scripted ones that record what they are called with (helpers.PolicyTrace): pins everything up to the TF
    boundary."""
    import tempfile
    from unittest.mock import MagicMock
    sys.path.insert(0, os.path.dirname(HERE))
    from helpers import PolicyTrace, script_pi, script_v
    tf = MagicMock()
    sys.modules['tensorflow'] = tf
    for mod in ('agents.models', 'utils'):
        sys.modules.pop(mod, None)
    import agents.models as am
    import utils as ref_utils
    ref_utils.tf = tf
    cp = _cfg(ini)
    env = CACCEnv(cp['ENV_CONFIG'])
    tr = PolicyTrace(env.n_agent, env.n_a)
    nbr = [np.where(env.neighbor_mask[i] == 1)[0] for i in range(env.n_agent)]

    class SinglePolicy:                       # LstmPolicy / FPPolicy stand-in (one per agent)
        def __init__(self, n_s, n_a, n_n, n_step, n_fc=64, n_lstm=64, name=None, **kw):
            self.i, self.k = int(name), 0

        def prepare_loss(self, *a, **k):
            pass

        def _reset(self):
            tr.rec(1, self.i)
            self.k = 0

        def forward(self, sess, ob, done, naction=None, out_type='p'):
            own = np.asarray(ob, dtype=np.float64)[None, :5]
            if out_type.startswith('p'):
                self.k += 1
                pi = script_pi(own, self.k, done, tr.w[self.i:self.i + 1])[0]
                tr.rec(2, self.i, float(bool(done)), np.asarray(ob, dtype=np.float32), pi)
                return pi
            v = script_v(own, self.k)[0]
            tr.rec(3, self.i, float(bool(done)), naction, v)
            return v

        def backward(self, sess, obs, nas, acts, dones, Rs, Advs, cur_lr, summary_writer=None, global_step=None):
            tr.rec(5, self.i, cur_lr, obs, nas, acts, dones, Rs, Advs)

    class MultiPolicy:                        # NC / IC3 / DIAL multi-agent policy stand-in
        def __init__(self, n_s, n_a, n_agent, n_step, neighbor_mask, **kw):
            self.k = 0

        def prepare_loss(self, *a, **k):
            pass

        def _reset(self):
            tr.rec(1)
            self.k = 0

        def forward(self, sess, ob, done, policy, action=None, out_type='p'):
            own = np.asarray(ob, dtype=np.float64)[:, :5]
            if out_type.startswith('p'):
                self.k += 1
                pi = script_pi(own, self.k, done, tr.w)
                tr.rec(2, float(bool(done)), np.asarray(ob, dtype=np.float32), np.asarray(policy, dtype=np.float32), pi)
                return pi
            v = script_v(own, self.k)
            tr.rec(3, float(bool(done)), action, v)
            return v

        def backward(self, sess, obs, ps, acts, dones, Rs, Advs, cur_lr, summary_writer=None, global_step=None):
            # reference layout [N,T,..] -> canonical [T,N,..]
            tr.rec(5, cur_lr, np.transpose(obs, (1, 0, 2)), np.transpose(ps, (1, 0, 2)), np.transpose(acts), dones,
                   np.transpose(Rs), np.transpose(Advs))

    am.LstmPolicy = am.FPPolicy = SinglePolicy
    am.NCMultiAgentPolicy = am.IC3MultiAgentPolicy = am.DIALMultiAgentPolicy = MultiPolicy
    cls = {'ia2c': am.IA2C, 'ia2c_fp': am.IA2C_FP, 'ma2c_nc': am.MA2C_NC, 'ma2c_ic3': am.MA2C_IC3,
           'ma2c_dial': am.MA2C_DIAL}[env.agent]
    model = cls(env.n_s_ls, env.n_a_ls, env.neighbor_mask, env.distance_mask, env.coop_gamma, 10 ** 6,
                cp['MODEL_CONFIG'], seed=12)
    writer = types.SimpleNamespace(add_summary=lambda *a, **k: None, flush=lambda: None)
    counter = ref_utils.Counter(total_step, 10 ** 9, 10 ** 9)
    trainer = ref_utils.Trainer(env, model, counter, writer, output_path=tempfile.mkdtemp() + '/')
    trainer.run()
    data = np.array([[d['step'], d['avg_reward'], d['std_reward']] for d in trainer.data])
    return dict(trace=np.array(tr.t), data=data, seed_after=env.seed, cur_step=counter.cur_step, ini=ini,
                total_step=total_step)


def tfnet_case(ini, total_step):
    """The UNMODIFIED reference end to end -- env, Trainer, agent class, policy classes and layer functions -- with
    TensorFlow replaced by tests/golden/tf_shim.py (the TF primitives restated on PyTorch-CPU).  Records the initial
    weights (reference variable names), every pi / v / bootstrap R the Trainer saw, and the weights after training."""
    import importlib
    import tempfile
    sys.setrecursionlimit(100000)
    sys.path.insert(0, HERE)
    tf = importlib.import_module('tf_shim')
    sys.modules['tensorflow'] = tf
    for mod in ('agents.models', 'agents.policies', 'agents.utils', 'utils', 'envs.cacc_env'):
        sys.modules.pop(mod, None)
    from envs.cacc_env import CACCEnv
    import agents.models as am
    import utils as ref_utils
    cp = _cfg(ini)
    env = CACCEnv(cp['ENV_CONFIG'])
    cls = {'ia2c': am.IA2C, 'ia2c_fp': am.IA2C_FP, 'ma2c_nc': am.MA2C_NC, 'ma2c_ic3': am.MA2C_IC3,
           'ma2c_dial': am.MA2C_DIAL, 'ma2c_cu': am.IA2C_CU}[env.agent]
    model = cls(env.n_s_ls, env.n_a_ls, env.neighbor_mask, env.distance_mask, env.coop_gamma, 10 ** 6,
                cp['MODEL_CONFIG'], seed=12)
    w0 = tf.variable_values()
    log = []

    class Rec:
        def __getattr__(self, k):
            return getattr(model, k)

        def forward(self, *a, **k):
            out = model.forward(*a, **k)
            log.append(np.array(out, dtype=np.float64).ravel())
            return out

        def backward(self, R, *a, **k):
            log.append(np.asarray(R, dtype=np.float64).ravel())
            return model.backward(R, *a, **k)
    writer = types.SimpleNamespace(add_summary=lambda *a, **k: None, flush=lambda: None)
    counter = ref_utils.Counter(total_step, 10 ** 9, 10 ** 9)
    trainer = ref_utils.Trainer(env, Rec(), counter, writer, output_path=tempfile.mkdtemp() + '/')
    trainer.run()
    w1 = tf.variable_values()
    out = dict(trace=np.concatenate(log), data=np.array([[d['step'], d['avg_reward'], d['std_reward']] for d in trainer.data]),
               seed_after=env.seed, cur_step=counter.cur_step, ini=ini, total_step=total_step, names=np.array(list(w0)))
    for n in w0:
        out['w0sha/' + n] = hashlib.sha256(np.ascontiguousarray(w0[n]).tobytes()).hexdigest()   # exact-match check only
        out['w1/' + n] = w1[n]
    return out


# ---- heterogeneous agents (SURVEY 8 f4): lstm_comm_hetero / lstm_ic3_hetero / lstm_dial_hetero ---------------------
HETERO = dict(edges=[(0, 1), (1, 2), (2, 3), (3, 4), (4, 5), (1, 4)],
              n_s_ls=[5, 7, 4, 6, 5, 3], n_a_ls=[4, 3, 5, 2, 4, 3], n_step=8, updates=3)


def hetero_case(agent):
    """The UNMODIFIED reference agent / policy / layer code for agents with UNEQUAL observation and action widths
    (agents/utils.py:220-341, 420-512, 602-702; agents/models.py:89-97, 229-235; agents/policies.py:289, 453, 502)
    on the TF shim.  CACC agents are identical, so a scripted stream stands in for the environment: random
    observations, rewards and action uniforms from a fixed RandomState; everything the policy returns is recorded."""
    import importlib
    sys.setrecursionlimit(100000)
    sys.path.insert(0, HERE)
    tf = importlib.import_module('tf_shim')
    sys.modules['tensorflow'] = tf
    for mod in ('agents.models', 'agents.policies', 'agents.utils', 'utils', 'envs.cacc_env'):
        sys.modules.pop(mod, None)
    import agents.models as am
    H = HETERO
    N = len(H['n_s_ls'])
    mask = np.zeros((N, N), dtype=int)
    for a, b in H['edges']:
        mask[a, b] = mask[b, a] = 1
    dist = np.zeros((N, N), dtype=int)
    cp = _cfg('config_ma2c_nc_catchup.ini')
    mc = cp['MODEL_CONFIG']
    mc['batch_size'] = str(H['n_step'])
    cls = {'ma2c_nc': am.MA2C_NC, 'ma2c_ic3': am.MA2C_IC3, 'ma2c_dial': am.MA2C_DIAL}[agent]
    np.random.seed(12)
    model = cls(H['n_s_ls'], H['n_a_ls'], mask, dist, -1.0, 10 ** 6, mc, seed=12)
    assert not model.identical_agent
    w0 = tf.variable_values()
    rs = np.random.RandomState(3)
    T = H['n_step']
    log, obs_l, uni_l, rew_l = [], [], [], []
    fp = [np.ones(n) / n for n in H['n_a_ls']]
    done = True
    model.reset()

    def decide(ob, done, fp):
        pi = model.forward(ob, done, fp)
        pi = [np.asarray(p, dtype=np.float64).ravel() for p in pi]
        log.append(np.concatenate(pi))
        u = rs.rand(N)
        uni_l.append(u)
        act = []
        for i in range(N):
            cdf = np.cumsum(pi[i]); cdf = cdf / cdf[-1]
            act.append(int(np.searchsorted(cdf, u[i], side='right')))
        return pi, np.array(act)
    for upd in range(H['updates']):
        for t in range(T):
            ob = [rs.randn(n) for n in H['n_s_ls']]
            obs_l.append(np.concatenate(ob))
            pi, act = decide(ob, done, fp)
            v = model.forward(ob, done, fp, act, 'v')
            log.append(np.asarray(v, dtype=np.float64).ravel())
            r = float(rs.randn() * 300.0)
            rew_l.append(r)
            model.add_transition(ob, fp, act, r, v, False)
            fp = [np.asarray(p, dtype=np.float32) for p in pi]
            done = False
        ob = [rs.randn(n) for n in H['n_s_ls']]
        obs_l.append(np.concatenate(ob))
        pi, act = decide(ob, done, fp)
        R = model.forward(ob, done, fp, act, 'v')
        log.append(np.asarray(R, dtype=np.float64).ravel())
        model.backward(R, 0)
        # the reference Trainer re-feeds the boundary observation as the first one of the next batch; the scripted
        # stream simply continues with fresh observations (the LSTM state keeps running, states_bw := states_fw)
    w1 = tf.variable_values()
    out = dict(trace=np.concatenate(log), obs=np.concatenate(obs_l), uniforms=np.array(uni_l), rewards=np.array(rew_l),
               names=np.array(list(w0)), mask=mask, n_s_ls=np.array(H['n_s_ls']), n_a_ls=np.array(H['n_a_ls']),
               n_step=T, updates=H['updates'])
    for n in w0:
        out['w0sha/' + n] = hashlib.sha256(np.ascontiguousarray(w0[n]).tobytes()).hexdigest()
        out['w0shape/' + n] = np.array(w0[n].shape)
        out['w1/' + n] = w1[n]
    return out


def configs_case():
    """Every CACC .ini of the reference as parsed key/value pairs, by file and section (what config/ must reproduce)."""
    out = {}
    for path in sorted(glob.glob(os.path.join(REF, 'config', 'config_*_catchup.ini')) +
                       glob.glob(os.path.join(REF, 'config', 'config_*_slowdown.ini'))):
        cp = configparser.ConfigParser()
        cp.read(path)
        out[os.path.basename(path)] = {s: dict(cp[s]) for s in cp.sections()}
    return out


def scheduler_case(au):
    s1 = au.Scheduler(5e-4, decay='constant')
    s2 = au.Scheduler(5e-4, 1e-4, 1e6, decay='linear')
    return dict(const=np.array([s1.get(60) for _ in range(5)]),
                linear=np.array([s2.get(60) for _ in range(20000)][::997]))


def main():
    CACCEnv, au = _import_reference()
    cases = [
        ('env_nc_catchup_const3', ('config_ma2c_nc_catchup.ini', 'const3'), {}),
        ('env_nc_catchup_cyc', ('config_ma2c_nc_catchup.ini', 'cyc'), {}),
        ('env_nc_catchup_rand2', ('config_ma2c_nc_catchup.ini', 'rand'), dict(n_reset=2)),
        ('env_nc_catchup_test', ('config_ma2c_nc_catchup.ini', 'const3'), dict(test_mode=True)),
        ('env_ic3_slowdown_const3', ('config_ma2c_cnet_slowdown.ini', 'const3'), {}),
        ('env_ic3_slowdown_cyc', ('config_ma2c_cnet_slowdown.ini', 'cyc'), {}),
        ('env_ic3_slowdown_const0', ('config_ma2c_cnet_slowdown.ini', 'const0'), {}),
        ('env_ic3_slowdown_test', ('config_ma2c_cnet_slowdown.ini', 'rand'), dict(test_mode=True)),
        ('env_ia2c_catchup_rand', ('config_ia2c_catchup.ini', 'rand'), {}),
        ('env_ia2c_slowdown_coop', ('config_ia2c_slowdown.ini', 'rand'), {}),
        ('env_dial_catchup_const1', ('config_ma2c_dial_catchup.ini', 'const1'), {}),
        # (config seed -1 -- the only value reaching the deterministic-init branch at
        #  cacc_env.py:290/311 -- is rejected by np.random.seed in __init__: dead code)
        ('env_nc_catchup_seed0', ('config_ma2c_nc_catchup.ini', 'const3'), dict(seed=0)),
    ]
    # fingerprint-carrying observations (ia2c_fp) and the remaining CACC configs; replayed by the CPU oracle test only
    cases += [
        ('envfp_ia2c_fp_catchup_rand', ('config_ia2c_fp_catchup.ini', 'rand'), dict(fp_seed=7)),
        ('envfp_ia2c_fp_slowdown_cyc', ('config_ia2c_fp_slowdown.ini', 'cyc'), dict(fp_seed=8, n_reset=2)),
        ('envfp_ma2c_cu_catchup_rand', ('config_ia2c_cu_catchup.ini', 'rand'), dict(fp_seed=9)),
    ]
    for name, (ini, kind), kw in cases:
        if os.path.exists(os.path.join(HERE, name + '.npz')) and '--force' not in sys.argv:
            continue
        out = env_case(CACCEnv, ini, kind, **kw)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'steps', len(out['ep0_done']), 'sumG', float(np.sum(out['ep0_greward'])))
    for name, ini, total in [('trainer_ma2c_nc_catchup', 'config_ma2c_nc_catchup.ini', 700),
                             ('trainer_ia2c_slowdown', 'config_ia2c_slowdown.ini', 700),
                             ('trainer_ia2c_fp_catchup', 'config_ia2c_fp_catchup.ini', 300)]:
        if os.path.exists(os.path.join(HERE, name + '.npz')) and '--force' not in sys.argv:
            continue
        out = trainer_case(CACCEnv, ini, total)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'trace', out['trace'].shape, 'data', out['data'].tolist(), 'seed', out['seed_after'], 'steps', out['cur_step'])
    for name, ini, total in [('tfnet_ma2c_nc_catchup', 'config_ma2c_nc_catchup.ini', 300),
                             ('tfnet_ia2c_slowdown', 'config_ia2c_slowdown.ini', 100),
                             ('tfnet_ia2c_fp_catchup', 'config_ia2c_fp_catchup.ini', 100),
                             ('tfnet_ma2c_ic3_slowdown', 'config_ma2c_cnet_slowdown.ini', 100),
                             ('tfnet_ma2c_dial_catchup', 'config_ma2c_dial_catchup.ini', 100),
                             ('tfnet_ma2c_cu_catchup', 'config_ia2c_cu_catchup.ini', 100)]:
        if os.path.exists(os.path.join(HERE, name + '.npz')) and '--force' not in sys.argv:
            continue
        out = tfnet_case(ini, total)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'trace', out['trace'].shape, 'data', out['data'].tolist(), 'seed', out['seed_after'], 'steps', out['cur_step'],
              'n_var', len(out['names']))
    for name, ini, total in [('agent_ma2c_nc_catchup', 'config_ma2c_nc_catchup.ini', 300),
                             ('agent_ia2c_slowdown', 'config_ia2c_slowdown.ini', 300),
                             ('agent_ia2c_fp_slowdown', 'config_ia2c_fp_slowdown.ini', 200),
                             ('agent_ma2c_ic3_slowdown', 'config_ma2c_cnet_slowdown.ini', 200),
                             ('agent_ma2c_dial_catchup', 'config_ma2c_dial_catchup.ini', 200)]:
        if os.path.exists(os.path.join(HERE, name + '.npz')) and '--force' not in sys.argv:
            continue
        out = agent_case(CACCEnv, ini, total)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'trace', out['trace'].shape, 'data', out['data'].tolist(), 'seed', out['seed_after'], 'steps', out['cur_step'])
    for agent in ('ma2c_nc', 'ma2c_ic3', 'ma2c_dial'):
        name = 'hetero_' + agent
        if os.path.exists(os.path.join(HERE, name + '.npz')) and '--force' not in sys.argv:
            continue
        out = hetero_case(agent)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'trace', out['trace'].shape, 'n_var', len(out['names']))
    path = os.path.join(HERE, 'reference_configs.json')
    if not os.path.exists(path) or '--force' in sys.argv:
        with open(path, 'w') as f:
            json.dump(configs_case(), f, indent=1, sort_keys=True)
        print('reference_configs.json')
    if '--force' not in sys.argv:
        return
    for name, alpha, multi in [('buffer_ma_global', -1, True), ('buffer_ma_spatial09', 0.9, True),
                               ('buffer_ia_global', -1, False), ('buffer_ia_spatial08', 0.8, False)]:
        out = buffer_case(au, alpha, multi)
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **out)
        print(name, 'sumRs', float(np.sum(out['Rs'])))
    # exact KAT recipe from SURVEY 8(c): no mid-batch done
    rs = np.random.RandomState(0)
    n = 8
    dist = np.abs(np.arange(n)[:, None] - np.arange(n)[None, :])
    buf = au.MultiAgentOnPolicyBuffer(0.99, -1, dist)
    for t in range(60):
        r = rs.randn(); ob = rs.randn(8, 5); p = rs.rand(8, 4); a = rs.randint(0, 4, 8); v = rs.randn(8)
        buf.add_transition(ob, p, a, r, v, False)
    R_end = rs.randn(8)
    _, _, _, _, Rs, Advs = buf.sample_transition(R_end)
    print('KAT alpha=-1: Rs[0,:3]', Rs[0, :3], 'Advs[7,-2:]', Advs[7, -2:], 'sumRs', Rs.sum())
    np.savez_compressed(os.path.join(HERE, 'scheduler.npz'), **scheduler_case(au))
    acts = eval_case(CACCEnv, 'config_ma2c_nc_catchup.ini', 'cyc', os.path.join(HERE, 'eval_'))
    np.save(os.path.join(HERE, 'eval_actions.npy'), acts)
    print('eval csvs', [f for f in os.listdir(HERE) if f.startswith('eval_')])


if __name__ == '__main__':
    main()
