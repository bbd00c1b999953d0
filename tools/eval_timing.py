"""Wall-clock cost of greedy evaluation on the GPU, one JSON line:

  * `main.py evaluate` of the default 50 seeds, sequential (Evaluator, one seed at a time through the host) vs
    `--batched` (VecEvaluator, all seeds as one device batch), for the NeurComm and DIAL catch-up configs.  Each
    time is bounded by torch.cuda.synchronize(), includes writing the control / traffic CSVs (into a temporary
    directory) and excludes loading the checkpoint; both variants are warmed up first and then alternated.
  * one in-training evaluation (VecTrainer.evaluate on ENV_CONFIG.test_seeds) next to one 4096-env update
    (CUDA-graph replay, as main.py trains).

Weights are the reference initialisation (untrained), so episode lengths are those of an untrained policy; they
are reported.  Needs a CUDA device; there is no CPU mode.
Usage: python tools/eval_timing.py [--repeats 3] [--n-seeds 50] [--n-env 4096]"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from helpers import load_cfg  # noqa: E402


def _gpu_info():
    info = {'device': torch.cuda.get_device_name()}
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        dev = torch.cuda.current_device()
        info['power_limit'], info['max_sm_clock'] = [s.strip() for s in out[dev].split(',')]
    except Exception as exc:                       # report, do not guess
        info['power_limit'] = info['max_sm_clock'] = 'unavailable (%s)' % type(exc).__name__
    return info


def _timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def _eval_compare(cfg_name, seeds, repeats, tmp):
    import main as M
    from deeprl_network_b200.envs.cacc_env import CACCEnv
    from deeprl_network_b200.utils import Evaluator, VecEvaluator
    cp = load_cfg(cfg_name, n_env=1)
    env = CACCEnv(cp['ENV_CONFIG'])
    env.init_test_seeds(seeds)
    model = M.init_agent(env, cp['MODEL_CONFIG'], 0, 0)
    vec = VecEvaluator(cp['ENV_CONFIG'], model, seeds)
    dirs = {k: os.path.join(tmp, cfg_name[:-4], k) + '/' for k in ('seq', 'bat')}
    for d in dirs.values():
        os.makedirs(d)
    run = {'seq': lambda: Evaluator(env, model, dirs['seq']).run(), 'bat': lambda: vec.evaluate(dirs['bat'])}
    for k in ('seq', 'bat'):                       # warm-up: module loads, allocations, pandas
        run[k]()
    times = {'seq': [], 'bat': []}
    for _ in range(repeats):
        for k in ('seq', 'bat'):
            times[k].append(_timed(run[k])[0])
    name = '%s_%s_%%s.csv' % (env.name, env.agent)
    same = all(filecmp.cmp(dirs['seq'] + name % kind, dirs['bat'] + name % kind, shallow=False)
               for kind in ('control', 'traffic'))
    seq, bat = float(np.median(times['seq'])), float(np.median(times['bat']))
    return {'config': cfg_name, 'seeds': len(seeds), 'T': env.T,
            'episode_steps_total': int(sum(vec.steps)), 'episodes_ended_early': int(sum(n < env.T for n in vec.steps)),
            'sequential_s': [round(t, 4) for t in times['seq']], 'batched_s': [round(t, 4) for t in times['bat']],
            'sequential_median_s': round(seq, 4), 'batched_median_s': round(bat, 4),
            'speedup_median': round(seq / bat, 2), 'files_identical': bool(same)}


def _in_training(n_env, repeats):
    import main as M
    from deeprl_network_b200.envs.cacc_env import CACCEnv
    from deeprl_network_b200.utils import VecTrainer
    cfg_name = 'config_ma2c_nc_catchup.ini'
    cp = load_cfg(cfg_name, n_env=n_env)
    env = CACCEnv(cp['ENV_CONFIG'])
    model = M.init_agent(env, cp['MODEL_CONFIG'], 10 ** 9, 12)
    vt = VecTrainer(env, model, graph=True)
    vt.start()
    for k in range(3):                             # capture + warm replays; one evaluation to build the evaluator
        vt.update()
    vt.evaluate(0)
    upd, evl = [], []
    for _ in range(max(repeats, 5)):
        upd.append(_timed(vt.update)[0])
        evl.append(_timed(lambda: vt.evaluate(0))[0])
    u, e = float(np.median(upd)), float(np.median(evl))
    return {'config': cfg_name, 'n_env': n_env, 'test_seeds': env.test_seeds, 'episode_steps': vt.evaluator.steps,
            'update_median_ms': round(1e3 * u, 3), 'evaluation_median_ms': round(1e3 * e, 3),
            'evaluation_over_update': round(e / u, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--n-seeds', type=int, default=50)
    ap.add_argument('--n-env', type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('eval_timing.py measures on a CUDA device; none found')
    import main as M
    seeds = [int(s) for s in M.DEFAULT_EVAL_SEEDS.split(',')][:args.n_seeds]
    out = _gpu_info()
    with tempfile.TemporaryDirectory() as tmp:
        out['evaluate'] = [_eval_compare(c, seeds, args.repeats, tmp)
                           for c in ('config_ma2c_nc_catchup.ini', 'config_ma2c_dial_catchup.ini')]
    out['in_training'] = _in_training(args.n_env, args.repeats)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
