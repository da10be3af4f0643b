"""CPU tests of the oracle (oracle/gcbf_oracle.py):
  1. against the committed golden fixtures (generated from the reference by oracle/make_golden.py);
  2. bit for bit against stored runs of the reference's own train step and replay buffer (tests/golden/reference_runs.json);
  3. semantic known-answer on the shipped pretrained checkpoints (when the reference checkout is present).
"""
import hashlib
import json
import os

import pytest
import torch

import gcbf_oracle as O
import ref_loader
from conftest import GOLDEN_DIR, digest_close, golden_cases, load_golden
from helpers import case_inputs, oracle_batch, sd_clone, seeded_algo

PRETRAINED_CBF = os.path.join(ref_loader.REFERENCE_ROOT, 'pretrained', 'SimpleCar', 'models', 'step_500000', 'cbf.pkl')


@pytest.fixture(autouse=True)
def _fixture_threads():
    """The seeded initialisation runs MKL's QR (orthogonal_), whose rounding depends on the number of intra-op threads: the port
    reproduces the stored reference weights bit for bit only at the thread count the fixtures were made with."""
    import make_golden
    n = torch.get_num_threads()
    torch.set_num_threads(make_golden.THREADS)
    yield
    torch.set_num_threads(n)


def _run_port(fix_like_meta, sb, n_steps):
    env_name, n = sb.env, sb.num_agents
    _, algo = seeded_algo(env_name, n, torch.device('cpu'), fix_like_meta['init_seed'],
                          {'num_obs': sb.num_obs, 'area_size': sb.area_size})
    cbf, act = sd_clone(algo.cbf), sd_clone(algo.actor)
    ob = oracle_batch(sb)
    e_attr = O.edge_attr(env_name, sb.states, ob['edge_index'])
    import copy
    with torch.no_grad():
        h = O.cbf_forward(copy.deepcopy(cbf), ob['x'], e_attr, ob['edge_index'], ob['agent_mask'])
        u = O.actor_forward(act, ob['x'], e_attr, ob['edge_index'], ob['agent_mask'], ob['u_ref'])
    oc, oa, steps = {}, {}, []
    for _ in range(n_steps):
        steps.append(O.update_step(env_name, cbf, act, oc, oa, sb.states, sb.goals, ob['edge_index'], ob['u_ref'],
                                   sb.num_graphs, n, sb.num_obs, K=ob['K']))
    return dict(ob=ob, edge_attr=e_attr, h=h, u=u, steps=steps, cbf=cbf, actor=act, init=(sd_clone(algo.cbf), sd_clone(algo.actor)))


@pytest.mark.parametrize('case', golden_cases())
def test_port_matches_golden(case):
    fix = load_golden(case)
    meta = fix['meta']
    sb = case_inputs(meta)
    if case.endswith('freeze'):
        sb.states[0, :2] = sb.goals[0, :2]
        sb.states[3, :2] = sb.goals[3, :2] + 0.01
    assert torch.equal(sb.states, fix['states']) and torch.equal(sb.goals, fix['goals'])
    r = _run_port(meta, sb, meta['steps'])
    assert not digest_close(r['init'][0], fix['cbf_init'], 0, 0), 'seeded CBF init differs from the reference'
    assert not digest_close(r['init'][1], fix['actor_init'], 0, 0)
    assert torch.equal(r['ob']['edge_index'], fix['edge_index'])                      # bit-exact
    assert torch.equal(r['ob']['u_ref'], fix['u_ref'])
    assert torch.equal(r['edge_attr'], fix['edge_attr'])
    assert torch.allclose(r['h'], fix['h_probe'], rtol=0, atol=1e-7)
    assert torch.allclose(r['u'], fix['u_probe'], rtol=0, atol=1e-6)
    assert torch.equal(r['steps'][0]['unsafe_mask'], fix['unsafe_mask'])
    assert torch.equal(r['steps'][0]['safe_mask'], fix['safe_mask'])
    for st, gold in zip(r['steps'], fix['steps']):
        for tag, key in (('loss/unsafe', 'loss_unsafe'), ('loss/safe', 'loss_safe'), ('loss/derivative', 'loss_h_dot'),
                         ('loss/action', 'loss_action'), ('acc/unsafe', 'acc_unsafe'), ('acc/safe', 'acc_safe'),
                         ('acc/derivative', 'acc_h_dot')):
            assert abs(float(st[key]) - gold['scalars'][tag]) <= 1e-6, (tag, float(st[key]), gold['scalars'][tag])
    assert not digest_close(r['cbf'], fix['cbf_final'], 1e-6, 1e-6)
    assert not digest_close(r['actor'], fix['actor_final'], 1e-6, 1e-6)


@pytest.mark.parametrize('case', ['dubins_n16_o4_b3', 'simplecar_c1', 'drone_n8_b2'])
def test_port_apply_matches_golden(case):
    """GCBF.apply (test-time controller, noise off) of the port against the reference's own apply()."""
    fix = load_golden(case)
    meta = fix['meta']
    sb = case_inputs(meta)
    _, algo = seeded_algo(sb.env, sb.num_agents, torch.device('cpu'), meta['init_seed'],
                          {'num_obs': sb.num_obs, 'area_size': sb.area_size})
    cbf, act = sd_clone(algo.cbf), sd_clone(algo.actor)
    ob = oracle_batch(sb)
    n, N = sb.num_agents, sb.nodes_per_graph
    ei0 = ob['edge_index'][:, ob['edge_index'][1] < N]
    a, it = O.apply_controller(sb.env, cbf, act, sb.states[:N], sb.goals, ei0, ob['u_ref'][:n], n, sb.num_obs,
                               O.HYPERPARAMS[sb.env]['alpha'], K=ob['K'])
    assert it >= 1
    assert torch.allclose(a, fix['apply_action'], rtol=1e-4, atol=1e-4), (a - fix['apply_action']).abs().max()


def _reference_runs():
    with open(os.path.join(GOLDEN_DIR, 'reference_runs.json')) as f:
        return json.load(f)


def _sha256(t):
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


@pytest.mark.parametrize('cfg', [('SimpleCar', 12, 0, 2, 2.0), ('DubinsCar', 10, 3, 2, 2.0), ('SimpleDrone', 6, 6, 2, 1.0)])
def test_port_matches_live_reference(cfg):
    """One train step of the port bit for bit against the reference's own (oracle/ref_harness.py, stored by
    `oracle/make_golden.py live`): edge_index, h, u and every tensor of both post-step state dicts (by SHA-256)."""
    env_name, n, obs, graphs, area = cfg
    ref = next(c for c in _reference_runs()['train_step'] if (c['env'], c['n'], c['obs'], c['graphs'], c['area']) == cfg)
    from gcbf_b200 import synth
    sb = synth.make_states(env_name, n, obs, graphs, area, ref['seed'])
    r = _run_port(dict(init_seed=0), sb, 1)
    assert torch.equal(r['ob']['edge_index'], torch.tensor(ref['edge_index'], dtype=r['ob']['edge_index'].dtype))
    assert torch.equal(r['h'], torch.tensor(ref['h_probe'], dtype=torch.float32))
    assert torch.equal(r['u'], torch.tensor(ref['u_probe'], dtype=torch.float32))
    for got, want in ((r['cbf'], ref['cbf_final_sha256']), (r['actor'], ref['actor_final_sha256'])):
        assert list(got) == list(want)
        for k in want:
            assert _sha256(got[k]) == want[k], k


@pytest.mark.skipif(not os.path.exists(PRETRAINED_CBF), reason="needs the reference checkout's trained SimpleCar checkpoint (49 MB)")
def test_pretrained_semantic_known_answer():
    """The shipped SimpleCar CBF must separate colliding from well-separated agents when evaluated through the
    port's restatement of PyG's message ordering / attention (SURVEY section 4): a wrong gather order or softmax
    grouping destroys this."""
    cbf = torch.load(PRETRAINED_CBF, map_location='cpu')
    from gcbf_b200 import synth
    hs, safe, coll = [], [], []
    for seed in range(20):
        sb = synth.make_states('SimpleCar', 16, 0, 1, 2.0, 100 + seed)
        sb.states[:, 2:] = 0
        ob = oracle_batch(sb)
        ea = O.edge_attr('SimpleCar', sb.states, ob['edge_index'])
        with torch.no_grad():
            hs.append(O.cbf_forward(cbf, ob['x'], ea, ob['edge_index'], None).reshape(-1))
        d = torch.cdist(sb.states[:, :2], sb.states[:, :2]) + torch.eye(16) * 10
        safe.append(d.min(dim=1)[0] > 0.3)
        coll.append(d.min(dim=1)[0] < 0.1)
    h, safe, coll = torch.cat(hs), torch.cat(safe), torch.cat(coll)
    assert coll.sum() > 5 and safe.sum() > 50
    assert (h[coll] < 0).float().mean() > 0.9
    assert (h[safe] >= 0).float().mean() > 0.9


def test_fp16x3_model_accuracy():
    """The arithmetic of the tensor-core layers (three fp16 products of [hi | lo] companions, 256-wide chunk promotion) is
    as accurate as an fp32 GEMM relative to the tensor scale -- for well-scaled data, for activations / gradients spanning
    several decades, and independently of the absolute magnitude; rows far below the tensor's max keep their ABSOLUTE accuracy
    (error <= 2^-39 of the max per element) but lose relative accuracy, which is the documented trade of the per-tensor scale."""
    import fp16x3_model as F16
    g = torch.Generator().manual_seed(0)
    M, N, K = 256, 192, 2048
    b = torch.randn(N, K, generator=g) / 45
    cases = {
        'normal': torch.randn(M, K, generator=g),
        'relu x 1e-6': torch.randn(M, K, generator=g).relu() * 1e-6,
        'heavy tail': torch.randn(M, K, generator=g) * torch.exp(3 * torch.randn(M, K, generator=g)),
        'x 1e12': torch.randn(M, K, generator=g) * 1e12,
    }
    for name, a in cases.items():
        ref = a.double() @ b.double().T
        scale = ref.abs().max()
        err16 = ((F16.gemm(a, b).double() - ref).abs().max() / scale).item()
        err32 = (((a @ b.T).double() - ref).abs().max() / scale).item()
        assert err16 < 1e-6, (name, err16)
        assert err16 < 4 * err32 + 2e-7, (name, err16, err32)
    # rows scaled down to 1e-8 of the largest: absolute error stays at the 2^-39-of-max level, relative error of those rows grows
    a = torch.randn(M, K, generator=g) * 10 ** (-8 * torch.linspace(0, 1, M).unsqueeze(1))
    ref = a.double() @ b.double().T
    err = (F16.gemm(a, b).double() - ref).abs()
    assert (err.max() / ref.abs().max()).item() < 1e-6
    small = torch.linspace(0, 1, M) > 0.75                        # rows below 1e-6 of the largest: their lo plane is subnormal
    per_elem_bound = K * (a.abs().max() * 2.0 ** -39) * b.abs().max()
    assert err[small].max().item() <= per_elem_bound.item()       # absolute accuracy of the small rows ...
    assert (err[small] / ref[small].abs().clamp_min(1e-300)).max().item() > 1e-6   # ... which is no longer fp32-relative
    # the companion reconstructs x to 22 bits (or 2^-39 of the max, whichever is larger)
    hi, lo, s = F16.split(a)
    rec = (hi.double() + lo.double()) / s
    assert ((rec - a.double()).abs() <= a.abs().double() * 2.0 ** -21 + a.abs().max().item() * 2.0 ** -39).all()


def test_buffer_sampling_matches_live_reference():
    """The replay buffers' index semantics (append, safe / unsafe bookkeeping, merge, segment sampling and its consumption
    of the host RNG streams) against the reference's OWN gcbf/algo/buffer.py (stored by `oracle/make_golden.py live`)."""
    import random
    import types
    import numpy as np
    want = _reference_runs()['buffer_sampling']
    from gcbf_b200.algo.buffer import Buffer
    from gcbf_b200.algo.device_buffer import DeviceReplay

    def graph(i):
        return types.SimpleNamespace(states=torch.full((2, 4), float(i)), u_ref=torch.full((2, 2), float(i)))

    buf, other, ring, ring_other = Buffer(), Buffer(), DeviceReplay('cpu', 16), DeviceReplay('cpu', 16)
    for i in range(90):
        buf.append(i, i % 4 != 0)
        ring.append(graph(i), i % 4 != 0)
    for i in range(200, 230):
        other.append(i, i % 3 == 0)
        ring_other.append(graph(i), i % 3 == 0)
    got, got_ring = [], []
    for seed, (n, m, bal) in enumerate([(12, 3, False), (16, 3, True), (7, 1, False), (20, 5, True)]):
        np.random.seed(seed), random.seed(seed)
        got.append(buf.sample(n, m, bal))
        np.random.seed(seed), random.seed(seed)
        got_ring.append([int(x) for x in ring.states_of(ring.sample(n, m, bal))[:, 0, 0]])
    buf.merge(other), ring.merge(ring_other)
    np.random.seed(9), random.seed(9)
    got.append(buf.sample(24, 3, True))
    np.random.seed(9), random.seed(9)
    got_ring.append([int(x) for x in ring.states_of(ring.sample(24, 3, True))[:, 0, 0]])
    got.append([buf.size, buf.safe_data[-3:], buf.unsafe_data[-3:]])
    assert got == want
    assert got_ring == want[:-1]
    assert [ring.size, ring.safe_data[-3:], ring.unsafe_data[-3:]] == want[-1]


@pytest.mark.parametrize('env_name,n,obs,B,area', [('DubinsCar', 12, 3, 5, 2.0), ('SimpleCar', 10, 0, 4, 1.5), ('SimpleDrone', 6, 6, 3, 1.0)])
def test_chunked_forward_step_matches_update_step(env_name, n, obs, B, area):
    """oracle.forward_step_chunked (used by the full-size GPU parity tests) against oracle.update_step on a batch small enough
    for both: same h / actions / h_next / h_next_new / masks / re-linked edges / losses, same spectral-norm state afterwards."""
    import copy
    from gcbf_b200 import synth
    sb = synth.make_states(env_name, n, obs, B, area, 91)
    ob = oracle_batch(sb)
    _, algo = seeded_algo(env_name, n, torch.device('cpu'), 3, {'num_obs': sb.num_obs, 'area_size': area})
    cbf_a, act_a = sd_clone(algo.cbf), sd_clone(algo.actor)
    cbf_b, act_b = copy.deepcopy(cbf_a), copy.deepcopy(act_a)
    want = O.update_step(env_name, cbf_a, act_a, {}, {}, sb.states, sb.goals, ob['edge_index'], ob['u_ref'], B, n, sb.num_obs,
                         K=ob['K'], apply_optim=False)
    got = O.forward_step_chunked(env_name, cbf_b, act_b, sb.states, sb.goals, ob['edge_index'], ob['u_ref'], B, n, sb.num_obs,
                                 K=ob['K'], chunk_graphs=2)
    assert torch.equal(got['edge_index_new'], want['edge_index_new'])
    assert torch.equal(got['unsafe_mask'], want['unsafe_mask']) and torch.equal(got['safe_mask'], want['safe_mask'])
    for k in ('h', 'actions', 'h_next', 'h_next_new', 'states_next'):
        assert (got[k].reshape(-1) - want[k].reshape(-1)).abs().max().item() <= 2e-7, k       # batched vs chunked GEMM blocking
    for k in ('loss_unsafe', 'loss_safe', 'loss_h_dot', 'loss_action', 'loss'):
        assert abs(float(got[k]) - float(want[k])) <= 1e-7, k
    for k in cbf_a:
        if k.endswith(('weight_u', 'weight_v')):
            assert torch.equal(cbf_a[k], cbf_b[k]), k
