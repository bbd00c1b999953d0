"""Experiment plumbing and the two training loops.

Drop-in surface (names, arguments and observable behaviour of the reference's utils.py:11-60, 70-97, 100-254,
311-336): ``Counter``, ``Trainer`` with ``explore`` / ``perform`` / ``run``, ``Tester``, ``Evaluator`` and the
directory / logging helpers.  The single-environment ``Trainer`` reproduces the reference loop call for call --
tests/test_trainer_flow.py replays traces recorded from the reference's own Trainer bit for bit -- including
its quirks (SURVEY 8a): Q1 the value call follows the policy call on the already advanced recurrent state, Q2 the
bootstrap at a non-terminal batch end is one more policy + value call, Q4 the reward that gets logged for CACC is
that of a greedy test episode run after every training episode, Q5 only training steps are counted.

``VecTrainer`` is the batched loop this package adds (n_env parallel episodes, everything device resident,
optionally one process per GPU with one NCCL gradient all-reduce per update).  ``VecEvaluator`` runs the greedy
test episodes of many seeds as one device batch, with the per-seed results of ``Evaluator``.
"""
import logging
import pathlib
import shutil
import time

import numpy as np
import torch

from . import _lib as L

_TEST_MODES = {'no_test': (False, False), 'in_train_test': (True, False),
               'after_train_test': (False, True), 'all_test': (True, True)}


# ---- directories / logging ---------------------------------------------------------------------------------------
def check_dir(cur_dir):
    return pathlib.Path(cur_dir).exists()


def copy_file(src_dir, tar_dir):
    shutil.copy(src_dir, tar_dir)


def find_file(cur_dir, suffix='.ini'):
    root = pathlib.Path(cur_dir)
    hits = sorted(f for f in root.iterdir() if f.name.endswith(suffix)) if root.is_dir() else []
    if hits:
        return '%s/%s' % (cur_dir, hits[0].name)
    logging.error('Cannot find %s file' % suffix)
    return None


def init_dir(base_dir, pathes=('log', 'data', 'model')):
    """-> {'log': '<base>/log/', ...}; creates what is missing."""
    out = {}
    for sub in pathes:
        d = pathlib.Path(base_dir) / sub
        d.mkdir(parents=True, exist_ok=True)
        out[sub] = '%s/%s/' % (base_dir, sub)
    return out


def init_log(log_dir):
    stamp = int(time.time())
    logging.basicConfig(format='%(asctime)s [%(levelname)s] %(message)s', level=logging.INFO,
                        handlers=[logging.FileHandler('%s/%d.log' % (log_dir, stamp)), logging.StreamHandler()])


def init_test_flag(test_mode):
    return _TEST_MODES.get(test_mode, (False, False))


def make_summary_writer(log_dir):
    """TensorBoard event writer (stands in for tf.summary.FileWriter); None when tensorboard is absent."""
    try:
        from torch.utils.tensorboard import SummaryWriter
        return SummaryWriter(log_dir)
    except Exception:  # pragma: no cover
        logging.warning('tensorboard not available: scalar summaries disabled')
        return None


class Counter:
    """Global step bookkeeping: counts training steps only; test / log cadence; stop condition."""

    def __init__(self, total_step, test_step, log_step):
        self.total_step, self.test_step, self.log_step = total_step, test_step, log_step
        self.cur_step = self.cur_test_step = 0
        self.stop = False

    def next(self):
        self.cur_step += 1
        return self.cur_step

    def should_test(self):
        due = self.cur_step - self.cur_test_step >= self.test_step
        if due:
            self.cur_test_step = self.cur_step
        return due

    def should_log(self):
        return self.cur_step % self.log_step == 0

    def should_stop(self):
        return self.stop or self.cur_step >= self.total_step


def eval_due(n_update, per_update, eval_interval, total_step):
    """Cadence of the batched trainer's greedy evaluations (TRAIN_CONFIG.eval_interval, in environment steps):
    True after the update that reaches or crosses a multiple of eval_interval, and after the final update
    (the one that reaches total_step).  Never when eval_interval is absent or 0."""
    if not eval_interval or eval_interval <= 0:
        return False
    done = int(n_update) * int(per_update)
    if done >= total_step:
        return True
    return done // int(eval_interval) > (done - int(per_update)) // int(eval_interval)


# ---- the single-environment loop -----------------------------------------------------------------------------------
class _AgentPort:
    """The two call conventions of the agent classes behind one face.  MA2C-style agents take the whole
    fingerprint matrix with every call and the joint action for the value; IA2C-style agents take nothing extra
    for the policy and, per agent, its neighbours' actions for the value.  ``aux`` is whatever the last call used
    and is what ``add_transition`` stores next to the observation."""

    def __init__(self, env, model):
        self.env, self.model = env, model
        self.joint = env.agent.startswith('ma2c')
        self.aux = None

    def policy(self, ob, done):
        if not self.joint:
            return self.model.forward(ob, done)
        self.aux = self.env.get_fingerprint()
        return self.model.forward(ob, done, self.aux)

    def value(self, ob, done, action):
        if self.joint:
            return self.model.forward(ob, done, self.aux, np.array(action), 'v')
        self.aux = self.env.get_neighbor_action(action)
        return self.model.forward(ob, done, self.aux, 'v')

    def store(self, ob, action, reward, value, done):
        self.model.add_transition(ob, self.aux, action, reward, value, done)


class Trainer:
    """One environment, one episode at a time (the reference's protocol).  ``uniform_fn`` optionally supplies the
    uniform behind each sampled action (tests feed the CUDA path and the oracle the same stream); by default
    actions come from ``np.random.choice`` like in the reference."""

    def __init__(self, env, model, global_counter, summary_writer, output_path=None, uniform_fn=None):
        self.env, self.model, self.global_counter = env, model, global_counter
        self.summary_writer, self.output_path, self.uniform_fn = summary_writer, output_path, uniform_fn
        self.agent = env.agent
        self.sess = getattr(model, 'sess', None)
        self.n_step = model.n_step
        if env.T % self.n_step:
            raise AssertionError('episode length %d is not a multiple of the batch size %d' % (env.T, self.n_step))
        self.cur_step = 0
        self.data = []
        self.episode_rewards = []
        self.env.train_mode = True
        self._port = _AgentPort(env, model)

    # -- action selection --
    def _draw(self, pi):
        if self.uniform_fn is None:
            return np.random.choice(np.arange(len(pi)), p=pi)
        cdf = np.cumsum(np.asarray(pi, dtype=np.float64))
        return int(np.searchsorted(cdf / cdf[-1], self.uniform_fn(), side='right'))

    def _decide(self, ob, done, greedy=False):
        policy = self._port.policy(ob, done)
        pick = np.argmax if greedy else self._draw
        return policy, np.array([pick(pi) for pi in policy])

    # -- logging --
    def _add_summary(self, reward, global_step, is_train=True):
        if self.summary_writer is not None:
            self.summary_writer.add_scalar('train_reward' if is_train else 'test_reward', reward, global_step)

    def _log_episode(self, global_step, mean_reward, std_reward):
        self.data.append(dict(agent=self.agent, step=global_step, test_id=-1, avg_reward=mean_reward,
                              std_reward=std_reward))
        self._add_summary(mean_reward, global_step)
        if self.summary_writer is not None:
            self.summary_writer.flush()

    # -- one batch of at most n_step transitions + its bootstrap target --
    def explore(self, prev_ob, prev_done):
        ob, done, port = prev_ob, prev_done, self._port
        for _ in range(self.n_step):
            policy, action = self._decide(ob, done)
            value = port.value(ob, done, action)                  # Q1: evaluated after the policy call
            self.env.update_fingerprint(policy)
            nxt, reward, done, global_reward = self.env.step(action)
            self.episode_rewards.append(global_reward)
            step = self.global_counter.next()
            self.cur_step += 1
            port.store(ob, action, reward, value, done)
            if self.global_counter.should_log():
                logging.info('Training: global step %d, episode step %d, ob: %s, a: %s, pi: %s, r: %.2f, '
                             'train r: %.2f, done: %r' % (step, self.cur_step, ob, action, policy, global_reward,
                                                          np.mean(reward), done))
            if done:                                              # CACC episodes may end inside a batch
                return ob, done, np.zeros(self.model.n_agent)
            ob = nxt
        _, action = self._decide(ob, done)                        # Q2: the bootstrap is a full policy + value call
        return ob, done, port.value(ob, done, action)

    # -- one evaluation episode --
    def perform(self, test_ind, gui=False):
        ob, done = self.env.reset(gui=gui, test_ind=test_ind), True      # done=True clears the recurrent state
        self.model.reset()
        greedy = not self.env.name.startswith('atsc')                    # CACC is evaluated with the arg-max policy
        rewards = []
        while True:
            policy, action = self._decide(ob, done, greedy=greedy)
            self.env.update_fingerprint(policy)
            ob, _, done, global_reward = self.env.step(action)
            rewards.append(global_reward)
            if done:
                rewards = np.array(rewards)
                return np.mean(rewards), np.std(rewards)

    def _train_episode(self):
        ob, done = self.env.reset(), True
        self.model.reset()
        self.cur_step, self.episode_rewards = 0, []
        while True:
            ob, done, R = self.explore(ob, done)
            step = self.global_counter.cur_step
            self.model.backward(R, self.env.T - self.cur_step, self.summary_writer, step)
            if done:
                self.env.terminate()
                return step

    def run(self, max_episodes=None):
        episodes = 0
        while not self.global_counter.should_stop() and (max_episodes is None or episodes < max_episodes):
            step = self._train_episode()
            rewards = np.array(self.episode_rewards)
            mean_reward, std_reward = np.mean(rewards), np.std(rewards)
            if not self.env.name.startswith('atsc'):              # Q4: a greedy episode provides the logged reward
                self.env.train_mode = False
                mean_reward, std_reward = self.perform(-1)
                self.env.train_mode = True
            self._log_episode(step, mean_reward, std_reward)
            episodes += 1
        if self.output_path is not None:
            import pandas as pd
            pd.DataFrame(self.data).to_csv(self.output_path + 'train_reward.csv')


class Tester(Trainer):
    """Present in the reference's import list but never run by its main.py (SURVEY row 11); kept so that the
    import keeps working."""

    def __init__(self, env, model, global_counter, summary_writer, output_path):
        super().__init__(env, model, global_counter, summary_writer, output_path=output_path)
        self.env.train_mode = False
        self.test_num = env.test_num


class Evaluator(Tester):
    """Runs every test seed of the environment once with the loaded model and writes the episode records."""

    def __init__(self, env, model, output_path, gui=False):
        self.env, self.model, self.output_path, self.gui = env, model, output_path, gui
        self.agent = env.agent
        self.env.train_mode = False
        self.test_num = env.test_num
        self.uniform_fn = None
        self._port = _AgentPort(env, model)

    def run(self):
        self.env.cur_episode = 0
        self.env.init_data(not self.gui, False, self.output_path)
        for test_ind in range(self.test_num):
            reward, _ = self.perform(test_ind, gui=self.gui)
            self.env.terminate()
            logging.info('test %i, avg reward %.2f' % (test_ind, reward))
            self.env.collect_tripinfo()
        self.env.output_data()


class VecTrainer:
    """Batched training loop: n_env parallel episodes advance in lock-step on the device.

    Per update: ``rollout`` (n_step x [p-call, v-call, env step] + bootstrap) -> returns ->
    training forward/BPTT/wgrad -> [all-reduce] -> clip + RMSProp, then per-env auto-reset of the
    environments whose episode ended (model.reset() + env.reset() of the reference, per env).
    With ``graph=True`` one update is captured once into a CUDA graph and replayed.
    """

    def __init__(self, env, model, graph=True, sample='philox'):
        self.env, self.model, self.engine = env, model, model.engine
        assert env.n_env == model.n_env
        self.sample = sample
        self.use_graph = graph
        self.graph = None
        self.n_update = 0
        self.env.train_mode = True
        # Episodes end (env `done`) only at multiples of the env's batch_size and at T: the per-env auto-reset below
        # looks at the done flag of the LAST step of an update only, so updates must tile the episode exactly
        # (the reference's Trainer has the same requirement implicitly, utils.py:129-197).
        if env.T % model.n_step or env.batch_size % model.n_step:
            raise AssertionError('VecTrainer: episode length %d / env batch_size %d are not multiples of the update '
                                 'length %d' % (env.T, env.batch_size, model.n_step))
        self.data = []                     # one record per update (train_reward.csv of the batched loop)
        self.eval_data = []                # one record per test seed and evaluation (eval_reward.csv)
        self.evaluator = None

    def start(self):
        self._seed = self.env.seed
        self.env.reset_device(u01=None, philox_seed=self._seed)
        self.engine.reset_states()
        self.engine.begin_episode(self.env)

    def _one_update(self, uniforms=None):
        e, env = self.engine, self.env
        e.rollout(env, sample=self.sample, uniforms=uniforms)
        e.update(self._lr)
        # episode boundaries: envs whose last step returned done restart (per-env model.reset/env.reset)
        done = e.done_buf[e.T_cur]
        e.roll_buffers()
        e.reset_states(mask=done)
        env.reset_device(u01=None, mask=done, obs_out=e.obs_buf[0], fp_out=e.fp_buf[0], philox_seed=self._seed)
        e.normalize_cur()

    def update(self, uniforms=None):
        e = self.engine
        # the schedule counts ENVIRONMENT steps (main.py's total_step): one update consumes n_step steps of every
        # env on every rank, so a linear lr_decay reaches lr_min at total_step whatever n_env / world size is
        lr = self.model.lr_scheduler.get(self.model.n_step * self.env.n_env * e.world)
        e.lr_dev.fill_(float(lr))
        self._lr = e.lr_dev
        if not self.use_graph:
            self._one_update(uniforms)
        else:
            if self.graph is None:
                self._static_uniforms = uniforms
                # warm-up outside capture (sets kernel attributes, allocates training buffers)
                self._one_update(uniforms)
                torch.cuda.synchronize()
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._one_update(self._static_uniforms)
                self.n_update += 1
                return
            self.graph.replay()
        self.n_update += 1

    def mean_reward(self):
        """Mean per-step global reward of the last batch (host sync)."""
        return float(self.engine.grew_buf[:self.engine.T_cur].mean().item())

    def log_rewards(self, global_step, summary_writer=None):
        """One `train_reward.csv` record (same columns as Trainer._log_episode): mean / std of the per-step global
        reward over the last batch of every env.  Unlike the one-env Trainer (quirk Q4) no greedy test episode is
        interleaved: these are the TRAINING rewards.  Host sync."""
        g = self.engine.grew_buf[:self.engine.T_cur]
        mean, std = float(g.mean().item()), float(g.std(unbiased=False).item())
        self.data.append(dict(agent=self.env.agent, step=int(global_step), test_id=-1, avg_reward=mean, std_reward=std))
        if summary_writer is not None:
            summary_writer.add_scalar('train_reward', mean, int(global_step))
        return mean

    def evaluate(self, global_step, summary_writer=None):
        """One greedy episode on each of ENV_CONFIG.test_seeds with the current weights (``VecEvaluator``: own env,
        LSTM states and buffers; the training state, RNG and buffers are not touched).  Appends one
        `eval_reward.csv` record per seed (``test_id`` = index into test_seeds) and writes the TB scalar
        `test_reward`, the mean over seeds, which it returns.  Host sync."""
        if self.evaluator is None:
            self.evaluator = VecEvaluator(self.env.config, self.model, self.env.test_seeds)
        res = self.evaluator.run()
        for k, (mean, std) in enumerate(res):
            self.eval_data.append(dict(agent=self.env.agent, step=int(global_step), test_id=k, avg_reward=mean,
                                       std_reward=std))
        mean = float(np.mean([m for m, _ in res]))
        if summary_writer is not None:
            summary_writer.add_scalar('test_reward', mean, int(global_step))
        return mean

    def write_csv(self, output_path):
        import pandas as pd
        pd.DataFrame(self.data).to_csv(output_path + 'train_reward.csv')
        if self.eval_data:
            pd.DataFrame(self.eval_data).to_csv(output_path + 'eval_reward.csv')


def _gather_layout(layout):
    """The layout of the same parameters with observations gathered on the device (IA2C's 'concat' API mode
    packs the same flat parameters; the batched episode has no host-side concatenation)."""
    if layout.obs_mode == 'gather':
        return layout
    from .layout import ModelLayout
    g = ModelLayout(layout.variant, layout.n_s_ls, layout.n_a, layout.mask, obs_mode='gather')
    assert g.entries == layout.entries and g.n_param == layout.n_param, 'gather layout moves the parameters'
    return g


class VecEvaluator:
    """Greedy test episodes of B = len(seeds) seeds advancing together on the device, forward only.

    Seed k gives what ``Trainer.perform`` / ``Evaluator`` give for it, bit for bit: the reset draws the same
    uniforms (``CACCEnv.reset_seeds``), the policy runs the FFMA cell kernel whose rows do not depend on B (the
    tensor-core path is never used here, so a seed's trajectory does not depend on how many seeds share its batch),
    the greedy choice is np.argmax's first maximum, and mean / std are taken on the host over the episode's steps.

    The engine reads the model's ``params`` tensor itself (shared, not copied), so an evaluation during training
    sees the current weights; LSTM states, DIAL messages, the obs / fingerprint / done / action buffers, the Philox
    counter and the env are its own.  The episode runs in chunks of ENV_CONFIG.batch_size steps (an episode can end
    only at such a boundary or at T) with no host synchronisation inside a chunk; after a chunk one small read
    decides whether every env is done."""

    def __init__(self, env_config, model, seeds):
        from .agents.engine import PolicyEngine
        from .envs.cacc_env import CACCEnv
        self.seeds = [int(s) for s in seeds]
        if not self.seeds:
            raise ValueError('VecEvaluator needs at least one seed')
        src = model.engine
        rng_state = np.random.get_state()      # CACCEnv seeds the global stream (reference behaviour): keep it as it was
        try:
            self.env = CACCEnv(env_config, n_env=len(self.seeds), device=src.device)
        finally:
            np.random.set_state(rng_state)
        self.env.init_test_seeds(self.seeds)
        self.T, self.chunk = self.env.T, self.env.batch_size
        lay = _gather_layout(model.layout)
        self.engine = PolicyEngine(lay, len(self.seeds), self.T, src.hp, flat_params=np.zeros(lay.n_param, np.float32),
                                   device=src.device, distance_mask=self.env.distance_mask,
                                   coop_gamma=self.env.coop_gamma, use_tc=False)
        self.engine.params = src.params
        self.trace = None

    def begin(self, record=False):
        """Reset every env to its seed's test episode, the recurrent state to zero, pre-step done = 1 and the
        fingerprints to 1/n_a (reset + model.reset() of ``Trainer.perform``)."""
        e, env = self.engine, self.env
        env.reset_seeds(self.seeds, obs_out=e.obs_buf[0], fp_out=e.fp_buf[0])
        e.reset_states()
        e.done_buf[0].fill_(1.0)
        self.trace = None
        if record:
            N, B = env.n_agent, env.n_env
            self.trace = torch.zeros(self.T + 1, 3, N, B, dtype=torch.float64, device=e.device)
            torch.stack((env.hs, env.vs, env.us), out=self.trace[0])

    def run_chunk(self, t0):
        """Steps t0 .. t0 + batch_size - 1 (at most up to T), launches only; returns the step reached."""
        e, env = self.engine, self.env
        t1 = min(t0 + self.chunk, self.T)
        for t in range(t0, t1):
            # greedy p-call; pi goes straight into the next step's fingerprint slot (env.update_fingerprint)
            e.step_p(e.obs_buf[t], e.fp_buf[t], e.done_buf[t], e.fp_buf[t + 1], e.act_buf[t], L.SAMPLE_GREEDY)
            env.step_device(e.act_buf[t], obs_out=e.obs_buf[t + 1], reward_out=e.rew_buf[t],
                            greward_out=e.grew_buf[t], done_out=e.done_buf[t + 1])
            if self.trace is not None:
                torch.stack((env.hs, env.vs, env.us), out=self.trace[t + 1])
        return t1

    def all_done(self, t):
        """Host sync: has every env's episode ended within steps 1..t?"""
        return bool(self.engine.done_buf[1:t + 1].amax(dim=0).min().item())

    def run(self, record=False):
        """One greedy episode per seed -> list of per-seed (mean, std) of the per-step global reward, over the
        steps up to and including the episode's first done.  With record=True the episodes are also appended,
        in seed order as episodes 1..B, to the env's records (``env.init_data`` first; ``env.output_data()``
        writes them)."""
        self.begin(record)
        t = 0
        while t < self.T:
            t = self.run_chunk(t)
            if t < self.T and self.all_done(t):
                break
        e = self.engine
        done = e.done_buf[1:t + 1].cpu().numpy()                       # [t, B]
        grew = np.ascontiguousarray(e.grew_buf[:t].cpu().numpy().T)     # [B, t]
        steps = done.argmax(axis=0) + 1                                 # first done (an env is done at T at the latest)
        assert done[steps - 1, np.arange(len(self.seeds))].all(), 'an episode did not end'
        self.steps = [int(n) for n in steps]                            # episode length per seed
        # contiguous per-seed rows: NumPy's reductions then sum in the same order as on the sequential path's arrays
        res = [(np.mean(grew[k, :n]), np.std(grew[k, :n])) for k, n in enumerate(steps)]
        if record:
            acts = np.ascontiguousarray(np.transpose(e.act_buf[:t].cpu().numpy(), (2, 0, 1)))         # [B, t, N]
            trace = np.ascontiguousarray(np.transpose(self.trace[:t + 1].cpu().numpy(), (3, 0, 1, 2)))  # [B, t+1, 3, N]
            for k, n in enumerate(steps):
                self.env.record_episode(k + 1, acts[k, :n], grew[k, :n], trace[k, :n + 1])
        return res

    def evaluate(self, output_path, gui=False):
        """``Evaluator.run`` for the whole batch: the same log lines and the same control / traffic files."""
        self.env.init_data(not gui, False, output_path)
        res = self.run(record=not gui)
        for k, (reward, _) in enumerate(res):
            logging.info('test %i, avg reward %.2f' % (k, reward))
        self.env.output_data()
        return res
