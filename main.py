"""Command line of the B200-native CACC / networked-A2C hot path.

The reference's command line is kept verbatim (main.py:21-40 there) so existing scripts keep working:

    python main.py --base-dir D train    --config-dir F.ini
    python main.py --base-dir D evaluate [--evaluation-seeds s1,s2,...] [--demo] [--batched]

and so is the .ini surface (MODEL_CONFIG / TRAIN_CONFIG / ENV_CONFIG).  Optional new keys:
  ENV_CONFIG.n_env            parallel episodes per process.  n_env = 1 runs the reference's one-episode-at-a-time
                              Trainer; n_env > 1 the device-resident VecTrainer.
  TRAIN_CONFIG.eval_interval  environment steps between greedy test episodes of the batched trainer (n_env > 1
                              only): after the update that reaches or crosses each multiple, and after the final
                              update, every ENV_CONFIG.test_seeds seed runs one greedy episode with the current
                              weights; one row per seed goes to data/eval_reward.csv and the mean over seeds to the
                              TB scalar `test_reward`.  Absent or 0: no evaluation.
`evaluate --batched` runs all evaluation seeds as one device batch (VecEvaluator); it logs and writes what the
sequential evaluator does.  Agents: ia2c, ia2c_fp, ma2c_cu, ma2c_nc, ma2c_ic3, ma2c_dial on the CACC scenarios;
ATSC/SUMO environments are out of scope (SURVEY row 10).
"""
import argparse
import configparser
import logging
import os

from deeprl_network_b200.agents import models as agent_models
from deeprl_network_b200.envs.cacc_env import CACCEnv
from deeprl_network_b200 import utils as U

AGENTS = {'ia2c': agent_models.IA2C, 'ia2c_fp': agent_models.IA2C_FP, 'ma2c_cu': agent_models.IA2C_CU,
          'ma2c_nc': agent_models.MA2C_NC, 'ma2c_ic3': agent_models.MA2C_IC3, 'ma2c_dial': agent_models.MA2C_DIAL}
DEFAULT_EVAL_SEEDS = ','.join(str(s) for s in range(2000, 2500, 10))


def parse_args(argv=None):
    top = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    top.add_argument('--base-dir', type=str, default='./runs/ma2c_nc_catchup', help='experiment base dir')
    modes = top.add_subparsers(dest='option', help='train or evaluate')
    tr = modes.add_parser('train', help='train the agent named in the config under the base dir')
    tr.add_argument('--config-dir', type=str, default='./config/config_ma2c_nc_catchup.ini', help='experiment config path')
    ev = modes.add_parser('evaluate', help='evaluate the agent stored under the base dir')
    ev.add_argument('--evaluation-seeds', type=str, default=DEFAULT_EVAL_SEEDS, help='random seeds for evaluation, split by ,')
    ev.add_argument('--demo', action='store_true', help='accepted for compatibility (SUMO gui in the reference); no files are written')
    ev.add_argument('--batched', action='store_true',
                    help='run all evaluation seeds as one batch on the GPU (same results and files as the default)')
    args = top.parse_args(argv)
    if args.option is None:
        top.print_help()
        raise SystemExit(1)
    return args


def read_config(path):
    cfg = configparser.ConfigParser()
    if not cfg.read(path):
        raise FileNotFoundError(path)
    return cfg


def init_env(config, port=0):
    """ENV_CONFIG section -> environment (only the CACC family exists here)."""
    if config.get('scenario').startswith('atsc'):
        raise NotImplementedError('ATSC/SUMO environments are outside the accelerated hot path')
    return CACCEnv(config)


def init_agent(env, config, total_step, seed, **kw):
    """MODEL_CONFIG section -> agent object of the class ENV_CONFIG.agent names (None if unknown)."""
    if env.agent not in AGENTS:
        logging.error('agent %r is not on the accelerated hot path' % env.agent)
        return None
    if env.agent == 'ia2c' and env.n_env > 1:     # device-resident rollouts gather neighbour observations in the kernel
        kw.setdefault('obs_mode', 'gather')
    return AGENTS[env.agent](env.n_s_ls, env.n_a_ls, env.neighbor_mask, env.distance_mask, env.coop_gamma,
                             total_step, config, seed=seed, n_env=env.n_env, **kw)


def _train_batched(env, model, total_step, log_interval, writer=None, output_path=None, eval_interval=0):
    """n_env > 1: whole updates on the device until total_step environment steps (summed over envs) are done.
    Every `log_interval` environment steps one record goes to data/train_reward.csv (and the TB scalar
    `train_reward`): mean / std of the per-step global TRAINING reward of the last batch.  With eval_interval > 0
    greedy test episodes run on the cadence of utils.eval_due -> data/eval_reward.csv, TB scalar `test_reward`."""
    loop = U.VecTrainer(env, model)
    loop.start()
    done_steps, per_update = 0, model.n_step * env.n_env
    every = max(1, int(log_interval) // per_update)
    while done_steps < total_step:
        loop.update()
        done_steps += per_update
        if loop.n_update % every == 0 or done_steps >= total_step:
            r = loop.log_rewards(done_steps, writer)
            logging.info('update %d, env steps %d, mean step reward %.2f' % (loop.n_update, done_steps, r))
        if U.eval_due(loop.n_update, per_update, eval_interval, total_step):
            r = loop.evaluate(done_steps, writer)
            logging.info('update %d, env steps %d, test reward %.2f' % (loop.n_update, done_steps, r))
    if output_path is not None:
        loop.write_csv(output_path)
    return done_steps


def train(args):
    dirs = U.init_dir(args.base_dir)
    U.init_log(dirs['log'])
    U.copy_file(args.config_dir, dirs['data'])             # evaluate finds the config next to the results
    cfg = read_config(args.config_dir)
    steps = {k: int(cfg.getfloat('TRAIN_CONFIG', k)) for k in ('total_step', 'test_interval', 'log_interval')}
    env = init_env(cfg['ENV_CONFIG'])
    logging.info('Training: a dim %r, agent dim: %d' % (env.n_a_ls, env.n_agent))
    model = init_agent(env, cfg['MODEL_CONFIG'], steps['total_step'], cfg.getint('ENV_CONFIG', 'seed'))
    if model is None:
        raise SystemExit(2)
    if env.n_env > 1:
        eval_interval = int(cfg.getfloat('TRAIN_CONFIG', 'eval_interval', fallback=0))
        final_step = _train_batched(env, model, steps['total_step'], steps['log_interval'],
                                    U.make_summary_writer(dirs['log']), dirs['data'], eval_interval=eval_interval)
    else:
        counter = U.Counter(steps['total_step'], steps['test_interval'], steps['log_interval'])
        U.Trainer(env, model, counter, U.make_summary_writer(dirs['log']), output_path=dirs['data']).run()
        final_step = counter.cur_step
    logging.info('Training: save final model at step %d ...' % final_step)
    model.save(dirs['model'], final_step)


def evaluate_fn(agent_dir, output_dir, seeds, port, demo, batched=False):
    """Load <agent_dir>/data/*.ini and the newest checkpoint under <agent_dir>/model/, run one recorded episode per seed.
    batched: all seeds as one device batch (VecEvaluator); returns the per-seed (mean, std) rewards."""
    if not U.check_dir(agent_dir):
        logging.error('Evaluation: %s does not exist!' % os.path.basename(agent_dir))
        return
    ini = U.find_file(agent_dir + '/data/')
    if not ini:
        return
    cfg = read_config(ini)
    cfg['ENV_CONFIG']['n_env'] = '1'
    env = init_env(cfg['ENV_CONFIG'], port=port)
    env.init_test_seeds(seeds)
    model = init_agent(env, cfg['MODEL_CONFIG'], 0, 0)
    if model is not None and model.load(agent_dir + '/model/'):
        if batched:
            return U.VecEvaluator(cfg['ENV_CONFIG'], model, seeds).evaluate(output_dir, gui=demo)
        U.Evaluator(env, model, output_dir, gui=demo).run()


def evaluate(args):
    output_dir = None
    if not args.demo:
        dirs = U.init_dir(args.base_dir, pathes=['eva_data', 'eva_log'])
        U.init_log(dirs['eva_log'])
        output_dir = dirs['eva_data']
    logging.info('Evaluation: random seeds: %s' % args.evaluation_seeds)
    seeds = [int(s) for s in args.evaluation_seeds.split(',') if s]
    return evaluate_fn(args.base_dir, output_dir, seeds, 1, args.demo, batched=getattr(args, 'batched', False))


if __name__ == '__main__':
    cli = parse_args()
    {'train': train, 'evaluate': evaluate}[cli.option](cli)
