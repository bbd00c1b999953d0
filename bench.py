"""bench.py -- agent-env-steps/sec of the CACC + A2C + NeurComm hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full update of the hot path over one batch: n_step (60) env steps of B parallel
CACC Catch-up episodes x 8 agents [p-call, sampling, v-call, env step], bootstrap, n-step returns,
training forward + BPTT + weight gradients, (NCCL all-reduce), clip + RMSProp.  Workload =
BASELINE.json configs[1]: config_ma2c_nc_catchup.ini, 4096 parallel envs per GPU (weak scaling).

Prints ONE JSON line (rank 0).  `value` is device-timed with inputs resident in HBM; `e2e` runs
the same update with HOST buffers: the action uniforms (the reference draws them with the host
NumPy RNG) are copied from pinned memory every step and the per-step rewards + loss terms are
read back, copies inside the timed region.  `roofline` follows SURVEY 8(d): algorithmic bytes per
agent-env-step x agent-env-steps per launch / the in-situ CUDA-event duration of the fused
step+message+cell forward kernel (rollout p-call) / the measured HBM peak; beside it `frac_with_saves`
(adds the BPTT activations that kernel also writes), `dram_frac` (ncu DRAM bytes / time / peak) and
`tensor_frac` (issued TF32 FLOP/s over half the measured bf16 peak), and the same triple for the
backward cell kernel and the weight-gradient GEMM.  `cpu_baseline` times the restated reference (TF
unavailable) on the host cores.  `configs` holds the other BASELINE.json configurations at their TOTAL env
counts split over the N ranks (cfg2 strong-scaling point, cfg3 CommNet, cfg4 DIAL, cfg5 5x5 grid), and
`dropin_b1` the reference-facing list/NumPy API at one env (main.py train's loop).

`--dump-outputs DIR` writes what the last of the K timed updates computed (rank 0) as DIR/<name>.npy, so that two
builds run with the same arguments can be compared output for output: the inputs (configs, seeds, Philox streams)
are identical from run to run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
METRIC = 'agent-env-steps/sec CACC Catch-up NeurComm A2C'
UNIT = 'agent-env-steps/s'
CONFIG = 'config_ma2c_nc_catchup.ini'
N_ENV = 4096


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20, help='timed updates of the headline workload (and of its e2e arm)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed update as DIR/<name>.npy')
    ap.add_argument('--n-env', type=int, default=N_ENV, help='parallel envs per GPU')
    ap.add_argument('--config', default=CONFIG)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip the `configs` block and the B=1 drop-in timing')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs needs --impl ours')
    return args


def load_cfg(name, **env_over):
    import configparser
    cp = configparser.ConfigParser()
    assert cp.read(os.path.join(ROOT, 'config', name)), name
    for k, v in env_over.items():
        cp['ENV_CONFIG'][k] = str(v)
    return cp


# ---- CPU arm: the restated reference trainer (oracle/) on the host cores -----------------------
def cpu_reference_best(cfg_name, updates):
    """The reference is single-process with TF's default thread pools; M=1 GEMVs gain nothing from
    threads, so time it with 1 thread and with all host threads and keep the faster."""
    import torch
    n_all = torch.get_num_threads()
    best = None
    for nt in sorted({1, n_all}):
        torch.set_num_threads(nt)
        v, cores, sample, dt = cpu_reference(cfg_name, updates=max(2, updates // 2), warm_updates=1)
        r = (v, nt, sample + ', torch threads=%d of %d host cores' % (nt, os.cpu_count()), dt / max(2, updates // 2))
        if best is None or v > best[0]:
            best = r
    torch.set_num_threads(n_all)
    return best


def cpu_reference(cfg_name, updates, warm_updates=1):
    """Times `updates` update cycles (n_step env steps each, B=1, per-agent Python loops, one
    forward per call -- the reference's structure) of the restated reference.  Returns
    (agent-env-steps/s, cores, sample description, seconds)."""
    import numpy as np
    import torch
    from oracle.cacc import OracleCACC
    from oracle.trainer import Counter, OracleAgent, OracleTrainer
    cp = load_cfg(cfg_name)
    env = OracleCACC(cp['ENV_CONFIG'])
    variant = cp['ENV_CONFIG']['agent']
    ag = OracleAgent(variant, env.n_s_ls, env.n_a_ls, env.neighbor_mask, env.distance_mask, env.coop_gamma, 10 ** 6,
                     cp['MODEL_CONFIG'], seed=12)
    tr = OracleTrainer(env, ag, Counter(10 ** 9, 10 ** 9, 10 ** 9))
    cores = torch.get_num_threads()
    done_updates, steps, t0 = 0, 0, None
    while done_updates < updates + warm_updates:
        ob = env.reset(); done = True; ag.reset(); tr.cur_step = 0; tr.episode_rewards = []
        while True:
            if done_updates == warm_updates and t0 is None:
                t0 = time.perf_counter(); steps = 0
            c0 = tr.global_counter.cur_step
            ob, done, R = tr.explore(ob, done)
            ag.backward(R)
            steps += tr.global_counter.cur_step - c0
            done_updates += 1
            if done or done_updates >= updates + warm_updates:
                break
    dt = time.perf_counter() - t0
    n = env.n_agent
    return steps * n / dt, cores, '%d update cycles of %d env steps, B=1, %s' % (updates, ag.n_step, cfg_name), dt


class ClockSampler:
    """Streams `nvidia-smi -lms 100` while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.5)
        except Exception:
            self.proc = None

    def summary(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        time.sleep(0.2)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            out = ''
        samples = [[x.strip() for x in l.split(',')] for l in out.strip().splitlines() if l.count(',') >= 5]
        if not samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(float(s[0]) for s in samples)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for k, n in enumerate(names) if any(s[2 + k].lower().startswith('active') for s in samples)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(samples[0][1]), 'reasons': reasons, 'samples': len(sm)}


# BASELINE.json configs measured beside the headline: (key, ini, TOTAL envs over all ranks)
EXTRA = [('cfg2_strong', 'config_ma2c_nc_catchup.ini', 4096),
         ('cfg3_ic3_slowdown', 'config_ma2c_cnet_slowdown.ini', 4096),
         ('cfg4_dial_catchup', 'config_ma2c_dial_catchup.ini', 8192),
         ('cfg5_grid5x5_nc', 'config_ma2c_nc_grid5x5_stub.ini', 2048)]


def survey_bytes(agent, n_s, n_a, mask, global_reward=True, n_h=64):
    """SURVEY 8(d): algorithmic HBM bytes per agent-env-step of the fused step+message+cell forward
    = B_K1 + B_K2 + B_state + B_out (1 640 NeurComm/CACC, 1 612 CommNet, 1 628 DIAL, 2 063 NeurComm on the grid)."""
    N = len(mask)
    nm = float(sum(int(sum(r)) for r in mask)) / N
    k1 = 8 + 4 + 12 + 4 * n_s + 4 * (1.0 / N if global_reward else 1.0)
    if agent in ('ma2c_nc', 'ia2c_fp'):
        k2 = 4 * n_s + nm * 4 * (n_s + n_a + n_h)
    elif agent == 'ma2c_ic3':
        k2 = 4 * n_s + nm * 4 * (n_s + n_h)
    elif agent == 'ma2c_dial':
        k2 = 4 * n_s + 4 * n_a + nm * 4 * (n_s + n_h)
    else:                                   # ia2c / ma2c_cu: own + neighbours' observations only
        k2 = 4 * n_s + nm * 4 * n_s
    return k1 + k2 + 16 * n_h + 4 * (2 * n_a + 2)


def issued_flops(lay, B, T):
    """TF32 FLOPs the tensor-core kernels ISSUE per launch (3 MMAs per fp32 product, K padded to 8, M = 128-row
    tiles, encoder N = 64, gate N = 256) -- from the same k-block schedules the kernels build."""
    N, SD = lay.N, lay.s_dim
    var = {'ma2c_cu': 'ia2c', 'ia2c_fp': 'ma2c_nc'}.get(lay.variant, lay.variant)
    k8 = lambda k: (k + 7) // 8 * 8
    fwd = bwd = 0
    for i in range(N):
        nn = len(lay.nbr[i])
        kx = k8(lay._kx(i))
        enc = kx
        if var == 'ma2c_nc':
            enc += k8(nn * lay.n_a) + 64 * nn
        elif var == 'ma2c_ic3':
            enc += 64
        elif var == 'ma2c_dial':
            enc += 64 * nn + 64                      # + sender-side mfc of the p-call
        fwd += 3 * 2 * B * (enc * 64 + (SD + 64) * 256)
        km = 0 if var == 'ia2c' else (64 if var == 'ma2c_ic3' else 64 * nn)
        bwd += 3 * 2 * B * (256 * (SD + 64) + 64 * km)
    ndp = {'ma2c_nc': 192, 'ia2c': 64}.get(var, 128)
    jobs = [256] * (2 if SD + 64 > 128 else 1) + [ndp] + ([] if var == 'ia2c' else [64] * (2 if lay.km_pad > 128 else 1))
    wgrad = 3 * 2 * 128 * sum(jobs) * T * B * N
    return fwd, bwd, wgrad


def build(config, B, rank, **env_over):
    from deeprl_network_b200.agents.models import MA2C_NC, MA2C_IC3, MA2C_DIAL, IA2C, IA2C_FP, IA2C_CU
    from deeprl_network_b200.envs.cacc_env import CACCEnv
    import numpy as np
    cp = load_cfg(config, n_env=B, seed=12 + 1000 * rank, **env_over)
    env = CACCEnv(cp['ENV_CONFIG'])
    cls = {'ma2c_nc': MA2C_NC, 'ma2c_ic3': MA2C_IC3, 'ma2c_dial': MA2C_DIAL, 'ia2c': IA2C, 'ia2c_fp': IA2C_FP,
           'ma2c_cu': IA2C_CU}[env.agent]
    np.random.seed(12)                                   # identical initial weights on every rank
    kw = dict(obs_mode='gather') if env.agent == 'ia2c' else {}
    model = cls(env.n_s_ls, env.n_a_ls, env.neighbor_mask, env.distance_mask, env.coop_gamma, 10 ** 9,
                cp['MODEL_CONFIG'], seed=12 + rank, n_env=B, **kw)
    return cp, env, model


DUMP_BYTES = 63 * 10 ** 6       # array data of --dump-outputs; with the .npy headers the directory stays under 64 MB


def dump_outputs(e, out_dir):
    """Writes what the last update handed its caller as <out_dir>/<name>.npy (float32 or float64): the updated weights,
    the gradient and its norm, the per-agent loss terms, and per env the rollout (global rewards, dones, actions, pi,
    values, observations after each step, bootstrap values) with its n-step returns and advantages.  When all envs
    do not fit in DUMP_BYTES, a fixed seeded subset of them is written; env_index.npy lists which."""
    import numpy as np
    import torch
    T, B = e.T_cur, e.B
    whole = {'params': e.params, 'grads': e.grads, 'grad_norm': e.norm_out}
    # (tensor, env axis); slot t + 1 of obs / fp / done holds what step t produced
    per_env = {'rewards': (e.grew_buf[:T], 1), 'dones': (e.done_buf[1:T + 1], 1), 'actions': (e.act_buf[:T].float(), 2),
               'pi': (e.fp_buf[1:T + 1], 2), 'values': (e.val_buf[:T], 2), 'obs': (e.obs_buf[1:T + 1], 2),
               'bootstrap_values': (e.R_end, 1), 'returns': (e.Rs[:T], 2), 'advantages': (e.Advs[:T], 2)}
    fixed = sum(t.numel() * t.element_size() for t in whole.values())
    env_bytes = sum(t.numel() // B * t.element_size() for t, _ in per_env.values()) + 8
    k = min(B, (DUMP_BYTES - fixed) // env_bytes)
    idx = np.sort(np.random.RandomState(0).choice(B, k, replace=False))
    out = {n: t.cpu().numpy() for n, t in whole.items()}
    out.update(e.losses())
    sel = torch.as_tensor(idx, device=e.device)
    out.update({n: t.index_select(d, sel).cpu().numpy() for n, (t, d) in per_env.items()})
    out['env_index'] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for n, a in out.items():
        assert a.dtype in (np.float32, np.float64), (n, a.dtype)
        np.save(os.path.join(out_dir, n + '.npy'), a)


class Runner:
    """Device-timed and end-to-end throughput of whole updates for one configuration."""

    def __init__(self, world, local):
        self.world, self.local = world, local

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, K):
        import torch
        import torch.distributed as dist
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(K):
            fn()
        ev1.record()
        self.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda')
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def measure(self, env, model, steps, warmup, e2e=True, clocks=False, dump=None):
        import torch
        from deeprl_network_b200.utils import VecTrainer
        e = model.engine
        T, N, B = e.T, e.N, e.B
        per_update = T * B * N
        out = {'envs_per_gpu': B, 'global_envs': B * self.world, 'agents': N, 'n_step': T,
               'tensor_core_path': bool(e.use_tc)}
        if not e.use_tc:
            out['note'] = 'FP32 FFMA fallback kernels (needs envs_per_gpu % 128 == 0 and narrow encoders for tcgen05)'
            sys.stderr.write('[bench] WARNING: %s x %d envs runs on the FFMA fallback kernels, not tcgen05\n' % (env.agent, B))
        vt = VecTrainer(env, model, graph=True, sample='philox')
        vt.start()
        l0 = e.launches
        vt.update()                                          # eager warm-up + capture
        out['launches_per_update'] = (e.launches - l0) // 2  # eager pass + capture pass issue the same calls
        for _ in range(max(0, warmup - 1)):
            vt.update()
        sampler = None
        if clocks:
            sampler = ClockSampler(self.local)
            sampler.start()
        ms = self.timed(vt.update, steps)
        if sampler is not None:
            out['clocks'] = sampler.summary()
        if dump is not None:
            dump_outputs(e, dump)          # before the e2e arm below trains the same model further
        out['value'] = steps * per_update * self.world / (ms * 1e-3)
        out['ms_per_step'] = ms / steps
        if e2e:
            uni_host = torch.rand(T + 1, N, B, dtype=torch.float64).pin_memory()
            uni_dev = torch.zeros(T + 1, N, B, dtype=torch.float64, device='cuda')
            rew_host = torch.zeros(T, B, dtype=torch.float64).pin_memory()
            loss_host = torch.zeros(N, 4, dtype=torch.float32).pin_memory()
            vt2 = VecTrainer(env, model, graph=True, sample='uniform')
            vt2._seed = vt._seed

            # H2D pipelining: step k+1's uniforms travel from pinned host memory on a copy stream while update k runs;
            # at the start of step k+1 they are moved (device to device) into the buffer the captured graph reads.
            # Every timed step still performs one full H2D copy of a step's inputs and the D2H read of its results.
            copy_stream = torch.cuda.Stream()
            uni_next = torch.zeros_like(uni_dev)
            arrived = torch.cuda.Event()

            def prefetch():
                with torch.cuda.stream(copy_stream):
                    uni_next.copy_(uni_host, non_blocking=True)                # H2D: the NEXT step's action uniforms
                    arrived.record(copy_stream)
            prefetch()

            def e2e_step():
                main = torch.cuda.current_stream()
                main.wait_event(arrived)                                       # this step's uniforms are on the device
                uni_dev.copy_(uni_next, non_blocking=True)
                copy_stream.wait_stream(main)                                  # uni_next is free again after that copy
                prefetch()
                vt2.update(uniforms=uni_dev)
                rew_host.copy_(e.grew_buf, non_blocking=True)                  # D2H: per-step global rewards
                loss_host.copy_(e.loss_part.sum(dim=(0, 2)), non_blocking=True)  # D2H: loss terms
                main.synchronize()                                             # the caller reads the results
            for _ in range(max(2, warmup)):
                e2e_step()
            ms2 = self.timed(e2e_step, steps)
            out['e2e'] = {'value': steps * per_update * self.world / (ms2 * 1e-3), 'unit': UNIT,
                          'h2d_bytes_per_step': uni_host.numel() * 8,
                          'd2h_bytes_per_step': rew_host.numel() * 8 + loss_host.numel() * 4,
                          'ms_per_step': ms2 / steps,
                          'api': 'VecTrainer.update(uniforms=<host RNG stream>) -> rewards, loss terms',
                          'h2d_overlap': 'the next step\'s uniforms are copied on a second stream during the current update'}
        self.vt = vt
        return out


def kernel_rooflines(env, model, vt, peaks, runner):
    """In-situ CUDA-event durations of the three tensor-core kernels of one eagerly launched update, and the
    SURVEY-8(d) roofline numbers built from them."""
    import numpy as np
    import torch
    from deeprl_network_b200 import _lib as L
    e = model.engine
    T, N, B = e.T, e.N, e.B
    lay = model.layout
    peak = float(peaks.get('hbm_gbs', 6650.0))
    tf32_peak = float(peaks.get('bf16_tflops', 1590.0)) / 2
    src = 'MEASURED_PEAKS.json (burst)' if peaks else 'fallback 6.65 TB/s / 1.59 PF bf16'
    b_step = survey_bytes(env.agent, 5, e.n_a, env.neighbor_mask, env.coop_gamma < 0)
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
    except Exception:
        pass
    per = traffic.get('per_kernel_bytes_per_launch', {})

    def ncu_bytes(name):
        return per.get(name)

    if not (e.use_tc and getattr(e, 'fuse_save', False)):
        # FFMA fallback: back-to-back launches of the p-call on one input
        pi = torch.zeros(N, B, e.n_a, device='cuda'); act = torch.zeros(N, B, dtype=torch.int32, device='cuda')
        f = lambda: e.step_p(e.obs_buf[0], e.fp_buf[0], e.done_buf[0], pi, act, L.SAMPLE_PHILOX, rng_offset=0)
        for _ in range(5):
            f()
        ms_k = runner.timed(f, 50) / 50
        ach = b_step * N * B / (ms_k * 1e-3) / 1e9
        return {'kernel': 'cell_fwd_kernel<P> (FP32 FFMA fallback)', 'bound': 'hbm', 'achieved': ach, 'peak': peak,
                'unit': 'GB/s', 'frac': ach / peak, 'traffic': None, 'us_per_launch': ms_k * 1e3,
                'algorithmic_bytes_per_agent_step': b_step, 'peak_source': src, 'timing': 'back-to-back launches'}
    # one more update, launched eagerly: events around each of its T saving p-calls (v-calls kept on the main stream
    # for this pass so nothing shares the SMs with the kernel being timed), each reverse step and the wgrad GEMM
    ov = e.overlap_v
    e.overlap_v, e.kernel_events = False, []
    e.rollout(env, sample=vt.sample)
    e.overlap_v = ov
    mk = lambda: torch.cuda.Event(enable_timing=True)
    step_ev, wg_ev = [mk() for _ in range(2 * T)], [mk(), mk()]
    for ev in step_ev + wg_ev:
        ev.record()                                       # instantiates the cudaEvent_t handles
    e.bwd_events = (step_ev, wg_ev)
    e.compute_returns(); e.backward()
    torch.cuda.synchronize()
    e.bwd_events = None
    fwd_us = 1e3 * float(np.mean([a.elapsed_time(b) for a, b in e.kernel_events[:T]]))
    e.kernel_events = None
    bwd_us = 1e3 * float(np.mean([step_ev[2 * t].elapsed_time(step_ev[2 * t + 1]) for t in range(T)]))
    wg_us = 1e3 * wg_ev[0].elapsed_time(wg_ev[1])
    e.apply(5e-4); e.roll_buffers(); e.normalize_cur()    # leave the engine in a consistent state
    f_fwd, f_bwd, f_wg = issued_flops(lay, B, T)
    save_b = 3072                                          # SURVEY 8(d) "Backward": s, gates, c, h, pre-activations (~768 floats)
    var = '%d' % {'ia2c': 0, 'ma2c_nc': 1, 'ma2c_ic3': 2, 'ma2c_dial': 3}.get(e.variant, 1)
    # template arguments: forward <VAR, MODE_PS = 3, state_fm>, backward <VAR, state_fm, raw_tiles>, wgrad <raw_tiles>
    t_fwd = ncu_bytes('tc_cell_fwd_kernel<%s, 3, %d>' % (var, int(e.state_fm)))
    t_bwd = ncu_bytes('tc_cell_bwd_kernel<%s, %d, %d>' % (var, int(e.state_fm), int(e.raw_tiles)))
    t_wg = ncu_bytes('tc_wgrad_kernel<%d>' % int(e.raw_tiles))

    def triple(alg_bytes, us, ncu_b, flops):
        ach = alg_bytes / (us * 1e-6) / 1e9
        return {'us_per_launch': us, 'algorithmic_bytes_per_launch': alg_bytes, 'achieved': ach, 'frac': ach / peak,
                'traffic': ncu_b, 'dram_frac': None if ncu_b is None else ncu_b / (us * 1e-6) / 1e9 / peak,
                'issued_tf32_tflops': flops / (us * 1e-6) / 1e12, 'tensor_frac': flops / (us * 1e-6) / 1e12 / tf32_peak}
    fwd = triple(b_step * N * B, fwd_us, t_fwd, f_fwd)
    r = {'kernel': 'tc_cell_fwd_kernel<PS> (tcgen05 3xTF32: fused gather + encoders + LSTM cell + heads + sampling + '
                   'activation save; rollout p-call)', 'bound': 'hbm', 'unit': 'GB/s', 'peak': peak, 'peak_source': src,
         'tf32_peak_tflops': tf32_peak,
         'timing': 'CUDA events on the launching stream around each launch of one eagerly launched update (in situ)',
         'algorithmic_bytes_per_agent_step': b_step,
         'frac_with_saves': (b_step + save_b) * N * B / (fwd_us * 1e-6) / 1e9 / peak,
         'note': 'frac = SURVEY 8(d) bytes (%.0f B per agent-env-step x %d) / in-situ time / measured HBM peak; the kernel is '
                 'declared compute-bound by 8(d) (3xTF32 GEMMs), so tensor_frac is the relevant utilisation; traffic = '
                 'ncu dram bytes per launch of the last committed profile (profiles/traffic.json)' % (b_step, N * B)}
    r.update(fwd)
    r['bwd'] = dict(kernel='tc_cell_bwd_kernel (one reverse BPTT step)', **triple(6200.0 * N * B, bwd_us, t_bwd, f_bwd))
    r['wgrad'] = dict(kernel='tc_wgrad_kernel (all GEMM weight gradients of one update)',
                      **triple(3400.0 * N * B * T, wg_us, t_wg, f_wg))
    return r


def dropin_b1(config, updates=3):
    """The reference-facing API itself: host observation lists in, NumPy out, one environment (`main.py train`)."""
    import main as M
    import torch
    from deeprl_network_b200.utils import Counter, Trainer
    cp = load_cfg(config, n_env=1)
    env = M.init_env(cp['ENV_CONFIG'])
    model = M.init_agent(env, cp['MODEL_CONFIG'], 10 ** 6, 12)
    model.engine.world = 1                 # one process drives this API (rank 0 only): no gradient all-reduce
    tr = Trainer(env, model, Counter(10 ** 9, 10 ** 9, 10 ** 9), None)
    ob, done = env.reset(), True
    model.reset()
    t0, steps = None, 0
    for k in range(updates + 1):
        if k == 1:
            torch.cuda.synchronize(); t0 = time.perf_counter(); steps = 0
        c0 = tr.global_counter.cur_step
        ob, done, R = tr.explore(ob, done)
        model.backward(R, 0, None, tr.global_counter.cur_step)
        steps += tr.global_counter.cur_step - c0
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {'value': steps * env.n_agent / dt, 'unit': UNIT, 'envs': 1, 'updates': updates, 'seconds': dt,
            'api': 'Trainer.explore + model.backward (forward / add_transition / backward with host lists, B = 1; '
                   'launch-bound: ~3 kernel launches + 3 host syncs per env step)'}


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))

    if args.impl == 'reference':
        if rank != 0:
            return
        import torch
        val, cores, sample, dt = cpu_reference_best(args.config, updates=max(2, 2 * args.steps))
        cp = load_cfg(args.config)
        T, N = int(cp['MODEL_CONFIG']['batch_size']), int(cp['ENV_CONFIG']['n_vehicle'])
        print(json.dumps({
            'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * dt, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': args.config + ', restated reference (TF unavailable), 1 env x %d agents, CPU' % N},
            'cpu_baseline': {'value': val, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    # stdout carries exactly one JSON line: NCCL (version banner, NCCL_DEBUG output) and any library chatter write to
    # file descriptor 1 as well, so fd 1 is pointed at stderr for the run and the line goes to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import gc
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    B = args.n_env
    runner = Runner(world, local)
    cp, env, model = build(args.config, B, rank)
    e = model.engine
    T, N = e.T, e.N
    head = runner.measure(env, model, args.steps, args.warmup, e2e=not args.no_e2e, clocks=True,
                          dump=args.dump_outputs if rank == 0 else None)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    roofline = kernel_rooflines(env, model, runner.vt, peaks, runner)
    # whole-update aggregate on SURVEY 8(d) bytes: rollout 2 x forward state traffic (~2.7 KB) + backward 6.2 KB
    agg_bytes = (survey_bytes(env.agent, 5, e.n_a, env.neighbor_mask, env.coop_gamma < 0) + 1024 + 40 + 6200 + 12.5)
    roofline['whole_update'] = {'algorithmic_bytes_per_agent_step': agg_bytes,
                                'achieved': agg_bytes * head['value'] / world / 1e9,
                                'frac': agg_bytes * head['value'] / world / 1e9 / roofline['peak']}
    launches = head['launches_per_update']
    del runner.vt, model, env, e
    gc.collect(); torch.cuda.empty_cache()

    configs = None
    if not args.no_extra:
        configs = {}
        for key, ini, total in EXTRA:
            if total % world or (key == 'cfg2_strong' and world == 1):
                continue
            try:
                cpx, envx, modx = build(ini, total // world, rank)
                r = runner.measure(envx, modx, max(3, args.steps // 2), max(3, args.warmup), e2e=not args.no_e2e)
                r['workload'] = '%s, %d envs in total over %d GPU(s), %d agents, n_step %d' % (ini, total, world, r['agents'], r['n_step'])
                configs[key] = r
            except Exception as ex:                       # a failing side configuration must not lose the headline
                configs[key] = {'error': repr(ex)[:300]}
            finally:
                runner.vt = None
                envx = modx = None
                gc.collect(); torch.cuda.empty_cache()

    cpu = drop = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample, dt = cpu_reference_best(args.config, updates=16)
        cpu = {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
               'label': 'restated reference (TF unavailable)', 'seconds': dt}
    if rank == 0 and not args.no_extra:
        try:
            drop = dropin_b1(args.config)
            if cpu is not None:
                drop['cpu_port_same_api'] = cpu['value']
        except Exception as ex:
            drop = {'error': repr(ex)[:300]}

    if rank == 0:
        emit = lambda line: os.write(json_fd, (line + '\n').encode())
        emit(json.dumps({
            'metric': METRIC, 'value': head['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': head['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': '%s, %d parallel envs per GPU x %d agents, n_step %d (BASELINE configs[1])' %
                                   (args.config, B, N, T), 'global_envs': B * world, 'parallelism': 'dp%d' % world,
                       'tensor_core_path': head['tensor_core_path'],
                       'l2_policy': 'per-step working set (activations %.1f GB) exceeds L2' %
                                    (T * N * B * 800 * 4 / 1e9)},
            'clocks': head.get('clocks'), 'e2e': head.get('e2e'), 'gpu_launches': launches * args.steps,
            'roofline': roofline, 'cpu_baseline': cpu, 'configs': configs, 'dropin_b1': drop}))
    if world > 1:
        # captured CUDA graphs hold NCCL kernels: tearing the communicator down under them can block, so leave
        # together after a final barrier instead of destroy_process_group()
        sys.stdout.flush()
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == '__main__':
    main()
