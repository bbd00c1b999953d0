"""CPU: host logic -- flat parameter layout, model descriptor, and that libnmarl.so loads and
exports every symbol include/nmarl.h declares (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from helpers import CFG, GOLDEN, ROOT, load_cfg
from deeprl_network_b200 import _lib as L
from deeprl_network_b200.envs.cacc_env import chain_masks, grid_masks
from deeprl_network_b200.layout import ModelLayout
from oracle import nets

N_PARAM = {'ma2c_nc': 598496, 'ma2c_ic3': 307680, 'ma2c_dial': 365536, 'ia2c': 274400,   # SURVEY 2.2 C1
           'ia2c_fp': 409568, 'ma2c_cu': 269920}     # 2 edge + 6 inner agents, counted by hand from policies.py:157-185, 366-399
N_S_LS = {'ia2c': [10, 15, 15, 15, 15, 15, 15, 10], 'ia2c_fp': [14, 23, 23, 23, 23, 23, 23, 14]}


def _layout(variant, **kw):
    mask, _ = chain_masks(8)
    n_s_ls = N_S_LS.get(variant, [5] * 8)
    return ModelLayout(variant, n_s_ls, 4, mask, **kw), mask, n_s_ls


@pytest.mark.parametrize('variant', list(N_PARAM))
def test_param_counts_and_names_match_reference_graph(variant):
    lay, mask, n_s_ls = _layout(variant, obs_mode='concat' if variant == 'ia2c' else 'gather')
    assert lay.n_real_param() == N_PARAM[variant]
    ref = nets.param_shapes(variant, n_s_ls, 4, mask)
    assert [n for n, _ in lay.creation_order()] == [n for n, _ in ref]
    assert dict(lay.creation_order()) == dict(ref)
    for name, off, shape in lay.entries:
        assert off % 4 == 0, name            # 16-byte alignment for cp.async / float4
    for a in lay.agents_off:
        assert a['p_begin'] < a['p_end'] <= lay.n_param


@pytest.mark.parametrize('variant', list(N_PARAM))
def test_pack_unpack_roundtrip_and_init_order(variant):
    lay, mask, n_s_ls = _layout(variant, obs_mode='concat' if variant == 'ia2c' else 'gather')
    np.random.seed(12)
    flat = lay.init_flat()
    np.random.seed(12)
    ref = nets.init_params(variant, n_s_ls, 4, mask)          # oracle consumes np.random in the same order
    mine = lay.unpack(flat)
    for k in ref:
        np.testing.assert_array_equal(mine[k], ref[k])
    np.testing.assert_array_equal(lay.pack(mine), flat)
    w = mine[[k for k in mine if k.endswith('wx_hid') or k.endswith('/wx')][0]]
    np.testing.assert_allclose(w.T @ w if w.shape[0] >= w.shape[1] else w @ w.T, 2 * np.eye(min(w.shape)), atol=1e-4)


def test_model_descriptor_chain_and_grid():
    lay, mask, _ = _layout('ma2c_nc')
    m = lay.c_model()
    assert (m.n_agent, m.n_a, m.s_dim, m.kx_pad, m.kp_pad, m.km_pad) == (8, 4, 192, 16, 8, 128)
    assert list(m.agent[0].nbr)[:1] == [1] and m.agent[0].n_nbr == 1
    assert list(m.agent[3].nbr)[:2] == [2, 4] and list(m.agent[3].x_src)[:3] == [3, 2, 4]
    a3 = m.agent[3]            # 3 is slot 1 of agent 2's list [1,3] and slot 0 of agent 4's list [3,5]
    assert sorted(zip(list(a3.recv_agent)[:2], list(a3.recv_slot)[:2])) == [(2, 1), (4, 0)]
    gm, gd = grid_masks(5)
    assert gm.sum(1).tolist().count(2) == 4 and gm.sum(1).tolist().count(3) == 12 and gm.sum(1).tolist().count(4) == 9
    assert gd.max() == 8 and (gm == gm.T).all()
    lay2 = ModelLayout('ma2c_nc', [5] * 25, 4, gm)
    assert lay2.n_real_param() == sum(int(np.prod(s)) for _, s in nets.param_shapes('ma2c_nc', [5] * 25, 4, gm))
    assert lay2.c_model().km_pad == 256


def test_ia2c_gather_and_concat_layouts_share_weights():
    a, _, _ = _layout('ia2c', obs_mode='concat')
    b, _, _ = _layout('ia2c', obs_mode='gather')
    assert [(n, o, s) for n, o, s in a.entries] == [(n, o, s) for n, o, s in b.entries]
    assert a.c_model().agent[1].x_nsrc == 1 and a.c_model().agent[1].x_w == 15 and a.obs_stride == 16
    assert b.c_model().agent[1].x_nsrc == 3 and b.c_model().agent[1].x_w == 5 and b.obs_stride == 8


def test_fp_and_consensus_agents_reuse_kernel_families():
    """SURVEY 8(f2): ia2c_fp is laid out as a NeurComm cell with unnamed zero padding where the message encoder
    and wx rows 128..191 sit; ma2c_cu is the IA2C cell fed with the agent's own observation."""
    lay, _, _ = _layout('ia2c_fp')
    m = lay.c_model()
    assert (m.variant, m.s_dim, m.per_agent_norm, m.kx_pad, m.kp_pad, m.km_pad) == (L.NC, 192, 1, 16, 8, 128)
    flat = lay.pack({n: np.ones(s, dtype=np.float32) for n, _, s in lay.entries})
    a = lay.agents_off[3]
    assert not flat[a['o_w_msg']:a['o_w_msg'] + 128 * 64].any() and not flat[a['o_b_msg']:a['o_b_msg'] + 64].any()
    assert flat[a['o_wxh']:a['o_wxh'] + 128 * 256].all() and not flat[a['o_wxh'] + 128 * 256:a['o_wxh'] + 192 * 256].any()
    assert flat[a['o_wxh'] + 192 * 256:a['o_wxh'] + 256 * 256].all()          # wh directly behind the padded wx
    assert int(flat.sum()) == lay.n_real_param() < lay.n_param
    lay, _, _ = _layout('ma2c_cu')
    m = lay.c_model()
    assert (m.variant, m.s_dim, m.per_agent_norm, m.kx_pad) == (L.IA2C, 64, 0, 8)
    assert m.agent[3].x_nsrc == 1 and m.agent[3].x_w == 5 and m.agent[3].n_nbr == 2
    assert m.agent[3].o_b == m.agent[3].o_wxh + 128 * 256                        # block nmarl_consensus_update averages


def test_unsupported_configurations_fail_loudly():
    mask, _ = chain_masks(8)
    with pytest.raises(ValueError):
        ModelLayout('greedy', [5] * 8, 4, mask)
    with pytest.raises(ValueError):
        ModelLayout('ma2c_nc', [5] * 8, 4, mask, n_h=128)


def test_library_loads_and_exports_header_symbols():
    assert os.path.exists(L.LIB_PATH), 'build libnmarl.so first (python -m deeprl_network_b200.build)'
    lib = L.lib()
    hdr = open(os.path.join(ROOT, 'include', 'nmarl.h')).read()
    declared = set(re.findall(r'\b(nmarl_[a-z0-9_]+)\s*\(', hdr))
    assert declared == set(L.EXPORTS), declared ^ set(L.EXPORTS)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.nmarl_version() >= 100
    assert lib.nmarl_sizeof_model() == ctypes.sizeof(L.Model)
    lay, _, _ = _layout('ma2c_nc')
    m = lay.c_model()
    assert lib.nmarl_ws_floats(ctypes.byref(m), 4096, 60) > 0
    assert lib.nmarl_loss_tiles(ctypes.byref(m), 4096) == 64


def test_tc_supported_needs_whole_128_env_tiles():
    """nmarl_tc_supported is the one rule for the tensor-core path; PolicyEngine.use_tc and the buffers it sizes follow it."""
    lib = L.lib()
    lay, _, _ = _layout('ma2c_nc')
    m = lay.c_model()
    assert lib.nmarl_tc_supported(ctypes.byref(m), 4096) == 1
    assert lib.nmarl_tc_supported(ctypes.byref(m), 100) == 0


def test_no_product_import_of_oracle():
    """The product package must never import the oracle (it is test infrastructure)."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'deeprl_network_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f
    assert 'oracle' not in open(os.path.join(ROOT, 'main.py')).read()


def test_shipped_configs_equal_the_reference_configs():
    """Drop-in contract: every CACC .ini of the reference runs unchanged (key- and value-identical copies under
    config/).  tests/golden/reference_configs.json holds the reference's catch-up and slow-down configs as parsed
    sections (tests/golden/make_golden.py)."""
    import configparser
    import json
    with open(os.path.join(GOLDEN, 'reference_configs.json')) as f:
        ref = json.load(f)
    assert len(ref) == 12
    for n, sections in sorted(ref.items()):
        mine = configparser.ConfigParser()
        assert mine.read(os.path.join(ROOT, 'config', n)), 'missing ' + n
        assert {s: dict(mine[s]) for s in mine.sections()} == sections, n


def test_hetero_layout_embedding_round_trip():
    """HeteroLayout (SURVEY 8 f4): reference (tight) tensors <-> padded flat buffer.  Every tight element maps to its own
    slot, everything else is zero except the policy-head bias of padded actions (-1e30), unpack(pack(x)) == x, names and
    shapes follow the reference's *_hetero creation order (tests/golden/hetero_*.npz)."""
    from deeprl_network_b200.layout import PI_PAD_BIAS, HeteroLayout
    from helpers import golden, random_params
    for agent in ('ma2c_nc', 'ma2c_ic3', 'ma2c_dial'):
        g = golden('hetero_' + agent)
        n_s, n_a = [int(x) for x in g['n_s_ls']], [int(x) for x in g['n_a_ls']]
        lay = HeteroLayout(agent, n_s, n_a, g['mask'])
        order = lay.creation_order()
        assert [n for n, _ in order] == [str(n) for n in g['names']]
        assert all(tuple(s) == tuple(g['w0shape/' + n]) for n, s in order)
        params = random_params(order, seed=3)
        flat = lay.pack(params)
        back = lay.unpack(flat)
        assert all(np.array_equal(back[n], params[n]) for n, _ in order)
        used = np.concatenate([lay._idx[n] for n, _ in order])
        assert len(used) == len(set(used.tolist())) == lay.n_real_param()
        rest = np.ones(lay.n_param, bool); rest[used] = False
        pad_bias = np.zeros(lay.n_param, bool); pad_bias[lay.pi_pad] = True
        assert np.all(flat[rest & ~pad_bias] == 0) and np.all(flat[pad_bias] == np.float32(PI_PAD_BIAS))
        assert len(lay.pi_pad) == sum(max(n_a) - a for a in n_a)
        m = lay.c_model()
        assert m.n_a == max(n_a) and m.agent[1].x_w == max(n_s) and m.agent[1].n_nbr == int(g['mask'][1].sum())
        assert lay.kx_pad <= 32 and lay.kp_pad <= 32          # fits the tensor-core path's one-k-block encoders
    with pytest.raises(NotImplementedError):
        iso = np.zeros((3, 3), int); iso[0, 1] = iso[1, 0] = 1
        HeteroLayout('ma2c_ic3', [5, 4, 3], [4, 3, 2], iso)   # CommNet agent without neighbours: mean over an empty set
