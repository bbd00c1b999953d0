"""GPU: batched greedy evaluation (VecEvaluator, `main.py evaluate --batched`, TRAIN_CONFIG.eval_interval).
(1) the batched evaluator writes byte-identical files and gives the per-seed (mean, std) of the sequential
Evaluator; (2) a seed's result does not depend on the batch it runs in; (3) a chunk runs without host
synchronisation; (4) evaluating during training leaves training bit-identical; (5) end to end through main.py."""
import configparser
import filecmp
import os

import numpy as np
import pytest
import torch

import main
from helpers import CFG, load_cfg, random_params

pytestmark = pytest.mark.gpu

SEEDS = list(range(2000, 2120, 10))                 # a dozen of the default evaluation seeds
CASES = [(a, CFG[a], {}) for a in ('ia2c', 'ia2c_fp', 'ma2c_cu', 'ma2c_nc', 'ma2c_ic3', 'ma2c_dial')] + \
        [('ma2c_nc', 'config_ma2c_nc_grid5x5_stub.ini', {})] + \
        [('ma2c_ic3', CFG['ma2c_ic3'], {'bias_to_zero': True})]   # slow-down, mostly action 0: collisions
_LENGTHS = {}                                       # case -> (episode lengths, T), for the coverage check at the end


def _setup(cfg_name, seeds, params_seed=0, bias_to_zero=False):
    from deeprl_network_b200.envs.cacc_env import CACCEnv
    cp = load_cfg(cfg_name, n_env=1)
    env = CACCEnv(cp['ENV_CONFIG'])
    env.init_test_seeds(seeds)
    model = main.init_agent(env, cp['MODEL_CONFIG'], 0, 0)
    params = random_params(model.layout.creation_order(), seed=params_seed)
    if bias_to_zero:
        for name in params:
            if '/pi' in name and name.endswith('/b'):
                params[name] = np.array([3.0, 0.0, 0.0, 0.0], dtype=np.float32)
    model.set_weights(params)
    return cp, env, model


def _sequential(env, model, out):
    """Evaluator.run, keeping the per-seed (mean, std) that it only logs."""
    from deeprl_network_b200.utils import Evaluator
    ev = Evaluator(env, model, out)
    env.cur_episode = 0
    env.init_data(True, False, out)
    res = [ev.perform(k) for k in range(env.test_num)]
    env.output_data()
    return res


@pytest.mark.parametrize('agent,cfg_name,kw', CASES, ids=['%s-%s%s' % (a, c[:-4], '-bias0' if k else '') for a, c, k in CASES])
def test_batched_files_and_rewards_equal_sequential(tmp_path, agent, cfg_name, kw):
    from deeprl_network_b200.utils import VecEvaluator
    cp, env, model = _setup(cfg_name, SEEDS, **kw)
    assert env.agent == agent
    seq_dir, bat_dir = str(tmp_path / 'seq') + '/', str(tmp_path / 'bat') + '/'
    os.makedirs(seq_dir); os.makedirs(bat_dir)
    ref = _sequential(env, model, seq_dir)
    ev = VecEvaluator(cp['ENV_CONFIG'], model, SEEDS)
    assert not ev.engine.use_tc and ev.engine.params.data_ptr() == model.engine.params.data_ptr()
    res = ev.evaluate(bat_dir)
    for k in range(len(SEEDS)):
        assert res[k][0] == ref[k][0] and res[k][1] == ref[k][1], (k, res[k], ref[k])
    for kind in ('control', 'traffic'):
        name = '%s_%s_%s.csv' % (env.name, env.agent, kind)
        assert filecmp.cmp(seq_dir + name, bat_dir + name, shallow=False), name
    _LENGTHS[(agent, cfg_name, bool(kw))] = (np.array(ev.steps), ev.T)


def test_seed_result_does_not_depend_on_batch():
    from deeprl_network_b200.utils import VecEvaluator
    seeds = list(range(2000, 2000 + 256 * 10, 10))
    target = seeds[200]
    cp, env, model = _setup(CFG['ma2c_nc'], [target])
    runs = []
    for batch in ([target], seeds[195:200] + [target] + seeds[201:207], seeds):
        ev = VecEvaluator(cp['ENV_CONFIG'], model, batch)
        assert not ev.engine.use_tc                          # B = 256 would select the tensor-core path otherwise
        k = batch.index(target)
        res = ev.run()
        n = ev.steps[k]
        e = ev.engine
        runs.append((res[k], n, e.act_buf[:n, :, k].cpu().numpy(), e.grew_buf[:n, k].cpu().numpy(),
                     e.fp_buf[1:n + 1, :, k].cpu().numpy()))
    for other in runs[1:]:
        assert other[0] == runs[0][0] and other[1] == runs[0][1]
        for a, b in zip(other[2:], runs[0][2:]):
            np.testing.assert_array_equal(a, b)


def test_chunk_runs_without_host_sync():
    from deeprl_network_b200.utils import VecEvaluator
    cp, env, model = _setup(CFG['ma2c_dial'], SEEDS)
    ev = VecEvaluator(cp['ENV_CONFIG'], model, SEEDS)
    ev.begin(record=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        t = ev.run_chunk(0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert t == ev.chunk
    torch.cuda.synchronize()


def _trainer(agent, B, graph):
    from deeprl_network_b200.envs.cacc_env import CACCEnv
    from deeprl_network_b200.utils import VecTrainer
    cp = load_cfg(CFG[agent], n_env=B, test_seeds='2000,2010,2020')
    env = CACCEnv(cp['ENV_CONFIG'])
    model = main.init_agent(env, cp['MODEL_CONFIG'], 10 ** 6, 12)
    return env, model, VecTrainer(env, model, graph=graph)


@pytest.mark.parametrize('graph', [False, True], ids=['eager', 'graph'])
@pytest.mark.parametrize('agent', ['ma2c_nc', 'ma2c_dial'])
def test_evaluation_does_not_perturb_training(agent, graph):
    outs = []
    for with_eval in (False, True):
        env, model, vt = _trainer(agent, 16, graph)
        vt.start()
        np_state = np.random.get_state()
        for k in range(3):
            vt.update()
            if with_eval:
                vt.evaluate(k + 1)
        torch.cuda.synchronize()
        assert np.array_equal(np.random.get_state()[1], np_state[1])
        e = model.engine
        outs.append((e.params.clone(), e.grew_buf.clone(), env.t_dev.clone(), e.rng.clone()))
        if with_eval:
            assert len(vt.eval_data) == 3 * 3 and [r['test_id'] for r in vt.eval_data[:3]] == [0, 1, 2]
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


def test_train_with_eval_interval_then_evaluate_batched(tmp_path):
    import pandas as pd
    cp = configparser.ConfigParser()
    cp.read(os.path.join(os.path.dirname(main.__file__), 'config', CFG['ma2c_nc']))
    per_update = 60 * 128
    cp['ENV_CONFIG']['n_env'] = '128'
    cp['TRAIN_CONFIG']['total_step'] = str(4 * per_update)
    cp['TRAIN_CONFIG']['log_interval'] = '1e4'
    cp['TRAIN_CONFIG']['eval_interval'] = '15000'
    ini = str(tmp_path / 'exp.ini')
    with open(ini, 'w') as f:
        cp.write(f)
    base = str(tmp_path / 'run')
    main.train(main.parse_args(['--base-dir', base, 'train', '--config-dir', ini]))
    tr = pd.read_csv(base + '/data/train_reward.csv', float_precision='round_trip')
    assert list(tr.columns)[1:] == ['agent', 'step', 'test_id', 'avg_reward', 'std_reward']
    assert list(tr['step']) == [per_update * k for k in (1, 2, 3, 4)] and (tr['test_id'] == -1).all()
    ev = pd.read_csv(base + '/data/eval_reward.csv', float_precision='round_trip')
    assert list(ev.columns)[1:] == ['agent', 'step', 'test_id', 'avg_reward', 'std_reward']
    assert list(ev['step']) == [2 * per_update, 4 * per_update] and list(ev['test_id']) == [0, 0]
    test_seeds = cp['ENV_CONFIG']['test_seeds']
    res = main.evaluate(main.parse_args(['--base-dir', base, 'evaluate', '--evaluation-seeds', test_seeds, '--batched']))
    assert len(res) == len(test_seeds.split(','))
    final = ev[ev['step'] == 4 * per_update]
    for k, (mean, _) in enumerate(res):
        assert float(final['avg_reward'].iloc[k]) == float(mean)
    assert sorted(os.listdir(base + '/eva_data')) == ['catchup_ma2c_nc_control.csv', 'catchup_ma2c_nc_traffic.csv']


def test_cases_cover_early_ends_and_full_episodes():
    """Across the module the seed sets include episodes that end early (collision) and episodes that reach T."""
    assert len(_LENGTHS) == len(CASES)
    assert any((n < T).any() for n, T in _LENGTHS.values())
    assert any((n == T).any() for n, T in _LENGTHS.values())
