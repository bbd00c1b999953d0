"""CPU: host-side pieces of the batched greedy evaluation -- the per-seed reset uniforms (checked against the
reference env's own reset and against the global NumPy stream), the `evaluate --batched` flag and the cadence of
the batched trainer's evaluations (TRAIN_CONFIG.eval_interval)."""
import numpy as np
import pytest

import main
from deeprl_network_b200.envs.cacc_env import seed_uniforms
from deeprl_network_b200.utils import eval_due
from helpers import CFG, load_cfg
from oracle.cacc import OracleCACC

SEEDS = [2000, 2010, 2250, 10000, 7, 123456]


@pytest.mark.parametrize('cfg', [CFG['ma2c_nc'], CFG['ma2c_ic3'], 'config_ia2c_slowdown.ini', 'config_ma2c_dial_catchup.ini'])
def test_seed_uniforms_equal_reference_reset(cfg):
    cp = load_cfg(cfg)
    u = seed_uniforms(SEEDS, 1)
    assert u.shape == (1, len(SEEDS)) and u.dtype == np.float64
    env = OracleCACC(cp['ENV_CONFIG'])
    env.init_test_seeds(SEEDS)
    env.train_mode = False
    for k in range(len(SEEDS)):
        env.reset(test_ind=k)
        ref = OracleCACC(cp['ENV_CONFIG'])
        ref.train_mode = False
        ref.init_test_seeds(SEEDS)
        ref.reset(test_ind=k, u01=u[0, k])
        np.testing.assert_array_equal(env.hs_cur, ref.hs_cur)
        np.testing.assert_array_equal(env.vs_cur, ref.vs_cur)
        np.testing.assert_array_equal(env.v0s, ref.v0s)
        if env.name.startswith('catchup'):
            assert env.hs_cur[0] == env.h_star * (1.5 + u[0, k])
        else:
            assert env.vs_cur[0] == env.v_star * (1.5 + u[0, k])


@pytest.mark.parametrize('n_platoon', [1, 5])
def test_seed_uniforms_equal_global_stream_and_leave_it_alone(n_platoon):
    np.random.seed(99)
    before = np.random.get_state()
    u = seed_uniforms(SEEDS, n_platoon)
    after = np.random.get_state()
    assert before[0] == after[0] and np.array_equal(before[1], after[1]) and before[2:] == after[2:]
    for k, s in enumerate(SEEDS):
        np.random.seed(s)
        # CACCEnv.reset: one np.random.rand() for the first platoon, then one per further platoon
        draws = [np.random.rand()] + [np.random.rand() for _ in range(n_platoon - 1)]
        np.testing.assert_array_equal(u[:, k], draws)


def test_grid_stub_draws_five_uniforms_per_seed():
    cp = load_cfg('config_ma2c_nc_grid5x5_stub.ini')
    e = cp['ENV_CONFIG']
    P = e.getint('n_vehicle') // e.getint('platoon_len')
    assert P == 5
    assert seed_uniforms([10000], P).shape == (5, 1)


def test_batched_flag_is_parsed():
    a = main.parse_args(['evaluate', '--evaluation-seeds', '2000,2010', '--batched'])
    assert a.option == 'evaluate' and a.batched and a.evaluation_seeds == '2000,2010'
    assert not main.parse_args(['evaluate']).batched


def _fires(per_update, eval_interval, total_step):
    n, out = 0, []
    done = 0
    while done < total_step:                 # main._train_batched's loop
        n += 1
        done += per_update
        if eval_due(n, per_update, eval_interval, total_step):
            out.append(n)
    return out


def test_eval_cadence():
    # 100 env steps per update, evaluate every 250: crossings at updates 3 (300), 5 (500), 8 (800), 10 (1000) + final 11
    assert _fires(100, 250, 1050) == [3, 5, 8, 10, 11]
    # exact multiples count when reached; the final update is not repeated
    assert _fires(100, 200, 1000) == [2, 4, 6, 8, 10]
    # interval smaller than one update: every update
    assert _fires(7680, 1000, 7680 * 4) == [1, 2, 3, 4]
    # interval beyond total_step: only the final update
    assert _fires(100, 10 ** 9, 450) == [5]
    # absent or 0: never, not even after the final update
    for off in (0, None):
        assert _fires(100, off, 1000) == []
