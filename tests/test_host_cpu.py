"""CPU tests of the host side: C-ABI library loads and exports every symbol include/gcbf_b200.h declares (no
compute calls without a GPU), graph containers, replay buffer, checkpoint key contract, and that the product
path refuses to run without CUDA (no silent CPU fallback)."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT
from gcbf_b200 import _C, native   # noqa: F401  (native registers the chain-level entry points)
from gcbf_b200.data import Batch, Data


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'gcbf_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(gcbf_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    assert _C.library_available(), 'libgcbf_b200.so missing: run python gcbf-pytorch_b200/csrc/build.py'
    lib = ctypes.CDLL(_C.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in include/gcbf_b200.h but not exported'
    assert sorted(_C.EXPORTED_SYMBOLS) == declared, set(_C.EXPORTED_SYMBOLS) ^ set(declared)
    assert _C.lib().gcbf_abi_version() == 4


def test_env_cfg_struct_layout():
    assert ctypes.sizeof(_C.EnvCfg) == 4 * 4 + 4 * 8


def test_no_cpu_fallback():
    from gcbf_b200.nn import MLP
    m = MLP(8, 4, (16,))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m(torch.zeros(3, 8))


def test_data_semantics():
    d = Data(x=torch.zeros(3, 4), states=torch.ones(3, 4), edge_attr=None)
    assert d.edge_attr is None and d.edge_index is None and 'edge_attr' not in d
    assert not hasattr(d, 'agent_mask') and hasattr(d, 'states')
    d.update(Data(u_ref=torch.zeros(3, 2)))
    assert 'u_ref' in d and d.num_nodes == 3
    d.u_ref = None
    assert not hasattr(d, 'u_ref')


def test_batch_roundtrip():
    gs = []
    for k in range(3):
        n = 4
        ei = torch.tensor([[1, 2, 0], [0, 0, 3]])
        gs.append(Data(x=torch.full((n, 4), float(k)), states=torch.rand(n, 4), edge_index=ei,
                       edge_attr=torch.rand(3, 4), agent_mask=torch.tensor([True, True, False, False])))
    b = Batch.from_data_list(gs)
    assert b.num_graphs == 3 and b.num_nodes == 12
    assert b.edge_index.shape == (2, 9) and torch.equal(b.edge_index[:, 3:6], gs[1].edge_index + 4)
    assert torch.equal(b.batch, torch.arange(3).repeat_interleave(4)) and b.ptr.tolist() == [0, 4, 8, 12]
    back = b.to_data_list()
    for g, r in zip(gs, back):
        for k in g.keys():
            assert torch.equal(g[k], r[k]), k
    assert isinstance(b, Batch) and isinstance(b, Data)


def test_buffer_sampling():
    import numpy as np
    import random
    from gcbf_b200.algo.buffer import Buffer
    np.random.seed(0)
    random.seed(0)
    buf = Buffer()
    for i in range(50):
        buf.append(i, is_safe=(i % 5 != 0))
    s = buf.sample(10, 3)
    assert len(s) == len(set(s)) and s == sorted(s) and len(s) <= 30
    s2 = buf.sample(10, 3, True)
    assert len(s2) == len(set(s2))
    other = Buffer()
    other.append(100, True)
    buf.merge(other)
    assert buf.size == 51 and buf.safe_data[-1] == 50
    buf.clear()
    assert buf.size == 0


def test_state_dict_key_contract():
    from gcbf_b200.algo.gcbf import CBFGNN
    from gcbf_b200.controller import GNNController
    cbf = CBFGNN(16, 4, 5, 256)
    keys = list(cbf.state_dict().keys())
    assert 'feat_transformer.module_0.phi.net.0.weight_orig' in keys
    assert 'feat_transformer.module_0.phi.net.4.weight_v' in keys
    assert 'feat_transformer.module_0.aggr_module.gate_nn.net.4.weight' in keys
    assert 'feat_2_CBF.net.6.bias' in keys and len(keys) == 38
    assert cbf.state_dict()['feat_transformer.module_0.phi.net.0.weight_orig'].shape == (2048, 13)
    act = GNNController(16, 4, 5, 256, 2)
    ak = list(act.state_dict().keys())
    assert len(ak) == 26 and 'feat_2_action.net.0.weight' in ak
    assert act.state_dict()['feat_2_action.net.0.weight'].shape == (512, 1026)


@pytest.mark.parametrize('env_name', ['SimpleCar', 'DubinsCar', 'SimpleDrone'])
def test_shipped_checkpoints_load_strictly(env_name, tmp_path):
    """Checkpoints laid out as the six shipped files (pretrained/<env>/models/step_500000/{cbf,actor}.pkl, SURVEY 8a row a13:
    key order, shapes and state-dict metadata from tests/golden/pretrained_checkpoints.json, seeded values in place of the
    trained weights) load with strict=True into the product modules through GCBF.load, also AFTER the parameters were
    re-homed into the flat bucket, and GCBF.save writes files of the shipped files' size (no bucket-sized storages) that
    the oracle port reads back unchanged."""
    import json
    from collections import OrderedDict
    from conftest import GOLDEN_DIR
    from gcbf_b200.synth import seeded_algo
    with open(os.path.join(GOLDEN_DIR, 'pretrained_checkpoints.json')) as f:
        layout = json.load(f)[env_name]
    ckpt = str(tmp_path / 'step_500000')
    os.makedirs(ckpt)
    g = torch.Generator().manual_seed(0)
    for net in ('cbf', 'actor'):
        sd = OrderedDict((k, torch.randn(shape, generator=g)) for k, shape in layout[net]['keys'])
        sd._metadata = OrderedDict(layout[net]['metadata'])
        torch.save(sd, os.path.join(ckpt, f'{net}.pkl'))
    env, algo = seeded_algo(env_name, 16, torch.device('cpu'))
    algo._ensure_bucket()                               # parameters become views into the flat bucket
    algo.load(ckpt)
    want_c = torch.load(os.path.join(ckpt, 'cbf.pkl'), map_location='cpu')
    want_a = torch.load(os.path.join(ckpt, 'actor.pkl'), map_location='cpu')
    for mod, want in ((algo.cbf, want_c), (algo.actor, want_a)):
        sd = mod.state_dict()
        assert list(sd.keys()) == list(want.keys())
        for k in want:
            assert torch.equal(sd[k], want[k]), k
    assert algo.cbf.feat_transformer.module_0.phi.net[2].weight_orig.data_ptr() >= algo._bucket.flat.data_ptr()   # still a bucket view
    algo.save(str(tmp_path))
    for f, want in (('cbf.pkl', want_c), ('actor.pkl', want_a)):
        size = os.path.getsize(tmp_path / f)
        assert abs(size - layout[f[:-4]]['file_bytes']) < 65536, (f, size)      # not 2x: each file holds ONE net
        back = torch.load(tmp_path / f, map_location='cpu')
        assert all(torch.equal(back[k], want[k]) for k in want)


def test_flat_bucket_views_survive_load_state_dict():
    from gcbf_b200.algo import make_algo
    from gcbf_b200.env import make_env
    dev = torch.device('cpu')
    env = make_env('SimpleCar', 4, dev)
    algo = make_algo('gcbf', env, 4, 4, 4, 2, dev)
    b = algo._ensure_bucket()
    n_params = sum(p.numel() for p in algo.cbf.parameters()) + sum(p.numel() for p in algo.actor.parameters())
    assert n_params <= b.flat.numel() < n_params + 64 * len(b.params)       # every parameter starts on a 256-byte boundary
    assert all(o % 64 == 0 for o in b.offsets)
    sd = {k: v.clone() + 1 for k, v in algo.cbf.state_dict().items()}
    algo.cbf.load_state_dict(sd)
    p0 = next(algo.cbf.parameters())
    assert p0.data_ptr() == b.flat.data_ptr() and torch.equal(b.flat[:p0.numel()].view_as(p0), p0)
    assert p0.grad.data_ptr() == b.grad.data_ptr()


def test_dropin_alias():
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r);"
            "from gcbf.nn import MLP, CBFGNNLayer; from gcbf.algo import make_algo; from gcbf.env import make_env;"
            "from gcbf.controller import GNNController; from gcbf.trainer import Trainer; import gcbf.algo.gcbf as g;"
            "print(g.GCBF.__module__)") % (os.path.join(ROOT, 'gcbf-pytorch_b200'), os.path.join(ROOT, 'gcbf-pytorch_b200', 'dropin'))
    out = subprocess.check_output([sys.executable, '-c', code], text=True)
    assert out.strip() == 'gcbf_b200.algo.gcbf'


def test_step_arena_views_are_disjoint_aligned_and_rewound():
    """The step arena (bump allocator behind every activation of train_step): views must not overlap, must honour
    dtype and shape, stay 256-byte aligned relative to the chunk, spill into a new chunk when one is full, and
    begin() must rewind."""
    import torch
    from gcbf_b200 import arena
    A = arena.StepArena()
    dev = torch.device('cpu')
    A.begin(dev)
    ts = [A.alloc((3, 5), torch.float32), A.alloc((7,), torch.int32), A.alloc((2, 4, 8), torch.float16),
          A.alloc((0, 4), torch.float32), A.alloc((1,), torch.int64)]
    base = A.chunks[0].data_ptr()
    spans = []
    for t in ts:
        if t.numel() == 0:
            continue
        assert t.is_contiguous() and (t.data_ptr() - base) % 256 == 0
        spans.append((t.data_ptr(), t.data_ptr() + t.numel() * t.element_size()))
    spans.sort()
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))
    for i, t in enumerate(ts):
        t.fill_(i + 1)
    for i, t in enumerate(ts):
        assert (t == i + 1).all()
    first = ts[0].data_ptr()
    big = A.alloc((arena._CHUNK_BYTES // 4 + 10,), torch.float32)     # does not fit the rest of chunk 0 -> new chunk
    assert len(A.chunks) == 2 and big.numel() == arena._CHUNK_BYTES // 4 + 10
    A.end()
    assert A.high_water > arena._CHUNK_BYTES
    A.begin(dev)
    assert A.alloc((3, 5), torch.float32).data_ptr() == first
    A.end()


def test_tensor_core_dispatch_rule():
    """Which layers of the reference's MLPs go to the tcgen05 kernel (host-side rule, no GPU needed)."""
    from gcbf_b200 import ops
    assert ops.use_h(24196, 2048, 2048) and ops.use_h(8192, 1024, 2048) and ops.use_h(8192, 2048, 260)
    assert ops.use_h(24196, 128, 256)                       # gate 256 -> 128
    assert not ops.use_h(24196, 2048, 12)                   # first phi layer: skinny-K stream kernel
    assert not ops.use_h(24196, 1, 128) and not ops.use_h(8192, 32, 128)   # tiny-N tails
    assert not ops.use_h(72, 2048, 2048)                    # too few rows for a 128-row tile to pay off
    old = ops.GEMM_IMPL
    try:
        ops.GEMM_IMPL = 1
        assert not ops.use_h(24196, 2048, 2048)
    finally:
        ops.GEMM_IMPL = old
    # the host rule is the library's rule
    from gcbf_b200 import _C, native   # noqa: F401  (native registers the chain-level entry points)
    lib = _C.lib()
    for M in (1, 255, 256, 4531, 24196):
        for N in (1, 32, 95, 96, 128, 2048):
            for K in (12, 95, 96, 260, 2048):
                assert ops.use_h(M, N, K) == bool(lib.gcbf_linear_h_supported(M, N, K)), (M, N, K)


def test_device_replay_matches_list_buffer(monkeypatch):
    """The device-resident replay ring (algo/device_buffer.py) against the list buffer that mirrors the reference's
    gcbf/algo/buffer.py: identical safe / unsafe bookkeeping, drop-oldest, merge and -- under the same host RNG seeds -- the
    same sampled graphs, through capacity growth and ring wrap-around (CPU tensors: the ring is plain torch indexing)."""
    import random
    import types
    import numpy as np
    import torch
    from gcbf_b200.algo.buffer import Buffer
    from gcbf_b200.algo.device_buffer import DeviceReplay
    monkeypatch.setattr(Buffer, 'MAX_SIZE', 37)

    def graph(i):
        return types.SimpleNamespace(states=torch.full((5, 4), float(i)), u_ref=torch.full((3, 2), -float(i)), tag=i)

    def check(lst, ring):
        assert lst.size == ring.size and lst.safe_data == ring.safe_data and lst.unsafe_data == ring.unsafe_data
        want = torch.stack([g.states for g in lst.data]) if lst.size else torch.empty(0, 5, 4)
        assert torch.equal(ring.states_of(range(ring.size)), want)
        for seed, (n, m, bal) in enumerate([(6, 3, False), (8, 3, True), (4, 1, False), (10, 5, True)]):
            if lst.size < max(n, m):
                continue
            np.random.seed(seed), random.seed(seed)
            a = [g.tag for g in lst.sample(n, m, bal)]
            np.random.seed(seed), random.seed(seed)
            idx = ring.sample(n, m, bal)
            assert [int(x) for x in ring.states_of(idx)[:, 0, 0]] == a and [int(-x) for x in ring.u_ref_of(idx)[:, 0, 0]] == a

    lst, ring = Buffer(), DeviceReplay('cpu', capacity=8)
    for i in range(60):                                   # grows 8 -> 16 -> 32 -> 37, then wraps (drop-oldest)
        lst.append(graph(i), is_safe=(i % 3 != 0))
        ring.append(graph(i), is_safe=(i % 3 != 0))
        if i % 7 == 0:
            check(lst, ring)
    check(lst, ring)
    lst2, ring2 = Buffer(), DeviceReplay('cpu', capacity=4)
    for i in range(100, 125):
        lst2.append(graph(i), is_safe=(i % 2 == 0))
        ring2.append(graph(i), is_safe=(i % 2 == 0))
    lst.merge(lst2), ring.merge(ring2)                    # 37 + 25 > MAX_SIZE: the oldest 25 drop out
    check(lst, ring)
    lst.clear(), ring.clear()
    check(lst, ring)
    lst.merge(lst2), ring.merge(ring2)
    check(lst, ring)


def test_trainer_loop_with_stub_env_and_algo(tmp_path):
    """gcbf_b200.trainer.Trainer is host glue around env / algo calls: drive it with CPU stubs and check the reference's
    contract (gcbf/trainer/trainer.py:42-141) -- exploration probability decays linearly from 1, u_ref is attached before the
    algorithm sees a graph, resets on `done`, update / checkpoint cadence, and eval() reports mean episode reward, the
    fraction of agents that never collided and the reach fraction of the last step."""
    import numpy as np
    import torch
    from gcbf_b200.data import Data
    from gcbf_b200.trainer import Trainer

    class Env:
        num_agents = 4

        def __init__(self, horizon):
            self.horizon, self.t, self.resets = horizon, 0, 0

        def reset(self):
            self.t, self.resets = 0, self.resets + 1
            return Data(states=torch.zeros(4, 2))

        def u_ref(self, graph):
            return graph.states + 1.0

        def step(self, action):
            self.t += 1
            info = {'safe': 1.0, 'reach': torch.tensor([True, False, True, True]),
                    'collision': torch.tensor([1]) if self.t == 2 else torch.tensor([], dtype=torch.long)}
            return Data(states=torch.full((4, 2), float(self.t))), np.full(4, 0.5), self.t >= self.horizon, info

    class Algo:
        def __init__(self):
            self.probs, self.updates, self.saved, self.seen_u_ref = [], [], [], True
            self._env = None

        def step(self, graph, prob):
            self.probs.append(prob)
            self.seen_u_ref &= hasattr(graph, 'u_ref')
            return torch.zeros(4, 2)

        def post_step(self, graph, action, reward, done, nxt):
            self.seen_u_ref &= hasattr(nxt, 'u_ref')

        def is_update(self, step):
            return step % 4 == 0

        def update(self, step, writer):
            self.updates.append(step)
            return {'acc/safe': 1.0}

        def apply(self, graph):
            self.seen_u_ref &= hasattr(graph, 'u_ref')
            return torch.zeros(4, 2)

        def save(self, path):
            self.saved.append(os.path.basename(path))

    env, env_test, algo = Env(horizon=3), Env(horizon=5), Algo()
    tr = Trainer(env, env_test, algo, str(tmp_path / 'run'))
    tr.train(steps=8, eval_interval=4, eval_epi=2)
    assert np.allclose(algo.probs, [1 - k / 8 for k in range(8)]) and algo.seen_u_ref
    assert algo.updates == [4, 8] and algo.saved == ['step_4', 'step_8']
    assert env.resets == 1 + 2                       # initial reset + one per finished 3-step episode (steps 3 and 6)
    assert algo._env is env
    reward, info = tr.eval(9, 3)
    assert abs(reward - 5 * 0.5) < 1e-9 and info == {'safe': 0.75, 'reach': 0.75}
    assert os.path.isdir(tmp_path / 'run' / 'models')


def test_c_abi_rejects_bad_arguments_before_touching_the_gpu():
    """Error behaviour of the C ABI (include/gcbf_b200.h): bad arguments return GCBF_E_INVALID (-1) with a message in
    gcbf_last_error() -- checked here for the tensor-core entry points, whose argument validation runs before any CUDA call, so
    no GPU is needed.  (Pointers below are never dereferenced on the host.)"""
    lib = _C.lib()
    ok_ptr, odd_ptr = 0x7f0000000000, 0x7f0000000004          # 16-byte aligned / misaligned fake device addresses

    def err():
        return lib.gcbf_last_error().decode()

    # companion buffers must be 16-byte aligned with a pitch that is a multiple of 8 halves
    assert lib.gcbf_split_f16(ok_ptr, 64, 4, 64, ok_ptr, odd_ptr, 64, None, 0, None) == -1 and 'aligned' in err()
    assert lib.gcbf_split_f16(ok_ptr, 64, 4, 64, ok_ptr, ok_ptr, 60, None, 0, None) == -1 and ('pitch' in err() or 'bad arguments' in err())
    assert lib.gcbf_split_f16(ok_ptr, 32, 4, 64, ok_ptr, ok_ptr, 64, None, 0, None) == -1          # ld < cols
    assert lib.gcbf_amax_f32(ok_ptr, 8, 4, 8, None, 0, None) == -1                                  # no amax slot
    # GEMM entry points: missing amax words, output pitch smaller than the row, misaligned companions
    args = dict(Xh=ok_ptr, ldx=64, xa=ok_ptr, Wh=ok_ptr, ldw=64, wa=ok_ptr)
    assert lib.gcbf_linear_fwd_h(args['Xh'], 64, None, args['Wh'], 64, ok_ptr, None, None, ok_ptr, 256, 512, 256, 64, 0, None, None) == -1
    assert lib.gcbf_linear_fwd_h(args['Xh'], 64, ok_ptr, args['Wh'], 64, ok_ptr, None, None, ok_ptr, 100, 512, 256, 64, 0, None, None) == -1
    assert lib.gcbf_linear_fwd_h(odd_ptr, 64, ok_ptr, args['Wh'], 64, ok_ptr, None, None, ok_ptr, 256, 512, 256, 64, 0, None, None) == -1
    assert 'gcbf_linear_fwd_' in err()          # (the per-tensor entry points forward to the general gcbf_linear_fwd_t)
    assert lib.gcbf_linear_bwd_data_h(ok_ptr, 256, ok_ptr, ok_ptr, 64, ok_ptr, None, ok_ptr, 32, ok_ptr, 64, 512, 256, 64, 0, None, None) == -1   # ld_relu < K
    assert lib.gcbf_linear_bwd_weight_h(ok_ptr, 256, ok_ptr, ok_ptr, 62, ok_ptr, None, ok_ptr, 64, 512, 256, 64, 0, None) == -1    # pitch not a multiple of 8
    assert lib.gcbf_amax_split_batched(None, 3, None) == -1
    assert lib.gcbf_sn_power_iter_batched(None, 1, ok_ptr, 0, None) == -1
    # the fp32 entry points keep their "tensor-core path has its own entry point" answer for impl = 2
    assert lib.gcbf_linear_fwd(ok_ptr, 64, ok_ptr, 64, None, None, ok_ptr, 64, 0, 64, 64, 0, 2, None, None) in (0, -3)


def test_apply_entry_point_without_a_gpu():
    """gcbf_apply (the test-time controller as one library call): the workspace query replays the call without launching, and
    the argument checks run before any CUDA call -- one graph only, noise required when rand != 0, aligned workspace."""
    from gcbf_b200 import synth
    from gcbf_b200.synth import seeded_algo
    sb = synth.make_states('DubinsCar', 16, 4, 1, 2.0, 1)
    env, algo = seeded_algo(sb.env, sb.num_agents, torch.device('cpu'), 0, {'num_obs': sb.num_obs, 'area_size': sb.area_size})
    env.set_goal(sb.goals)
    d = algo._step_desc()[0]

    def batch(B, E=300):
        cfg_s = env._cfg(B)
        ctypes.memmove(ctypes.byref(d.env), ctypes.byref(cfg_s), ctypes.sizeof(_C.EnvCfg))
        b = native.StepBatch()
        fake = 1 << 20
        b.states, b.ld_state, b.x, b.edge_attr, b.edge_index, b.rowptr, b.u_ref = fake, env.state_dim, fake, fake, fake, fake, fake
        b.row_index = fake
        b.num_edges, b.num_nodes, b.num_agents_total = E, B * sb.nodes_per_graph, B * sb.num_agents
        return b

    b1 = batch(1)
    need = native.fn('gcbf_apply_workspace_bytes')(ctypes.byref(d), ctypes.byref(b1))
    assert need > 0, _C.lib().gcbf_last_error()
    bigger = native.fn('gcbf_apply_workspace_bytes')(ctypes.byref(d), ctypes.byref(batch(1, 3000)))
    assert bigger > need
    b1 = batch(1)
    call = native.fn('gcbf_apply')
    rounds = ctypes.c_int(0)
    ok = 0x7f0000000000
    assert call(ctypes.byref(d), ctypes.byref(b1), 0.1, 30.0, None, 30, ok, 2, ctypes.byref(rounds), ok, need, None) == -1     # rand without noise
    assert 'noise' in _C.lib().gcbf_last_error().decode()
    assert call(ctypes.byref(d), ctypes.byref(b1), 0.1, 0.0, None, 30, ok, 1, ctypes.byref(rounds), ok, need, None) == -1      # pitch < action_dim
    assert call(ctypes.byref(d), ctypes.byref(b1), 0.1, 0.0, None, 30, ok, 2, ctypes.byref(rounds), ok + 8, need, None) == -1  # misaligned workspace
    assert call(ctypes.byref(d), ctypes.byref(b1), 0.1, 0.0, None, 30, ok, 2, ctypes.byref(rounds), ok, 1024, None) == native.E_WORKSPACE
    b2 = batch(2)
    assert call(ctypes.byref(d), ctypes.byref(b2), 0.1, 0.0, None, 30, ok, 2, ctypes.byref(rounds), ok, need * 4, None) == -1  # two graphs
    assert 'one graph' in _C.lib().gcbf_last_error().decode()


def test_abi_struct_mirrors_and_workspace_queries_without_a_gpu():
    """The ctypes mirrors of the chain-level ABI structures have the library's sizes, and the workspace queries (which replay a
    call's allocation sequence without launching) work on descriptors built from CPU tensors: sizes grow with the edge count and a
    whole C3 step (~206 k edges, 65,536 agents) fits one B200 (180 GB) with room to spare."""
    from gcbf_b200 import synth
    from gcbf_b200.synth import seeded_algo
    mirrors = [_C.EnvCfg, native.LinearDesc, native.NetDesc, native.StepDesc, native.StepBatch, native.StepOut, native.NetCtx,
               native.MlpCtx, native.StepCtx, native.TimeRec, _C.SnLayer, _C.SplitDesc, native.H16Desc]
    for i, m in enumerate(mirrors):
        assert ctypes.sizeof(m) == _C.lib().gcbf_abi_struct_size(i), m.__name__
    assert _C.lib().gcbf_abi_struct_size(99) == 0
    sizes = {}
    for cfg, E in (('C2', 24196), ('C3', 206139)):
        c = dict(synth.CONFIGS[cfg])
        sb = synth.make_states(c['env'], c['num_agents'], c['num_obs'], 1, c['area_size'], 1)
        env, algo = seeded_algo(sb.env, sb.num_agents, torch.device('cpu'), 0, {'num_obs': sb.num_obs, 'area_size': sb.area_size})
        env.set_goal(sb.goals)
        d = algo._step_desc()[0]
        B = c['num_graphs']
        cfg_s = env._cfg(B)
        ctypes.memmove(ctypes.byref(d.env), ctypes.byref(cfg_s), ctypes.sizeof(_C.EnvCfg))
        b = native.StepBatch()
        fake = 1 << 20
        b.states, b.ld_state, b.x, b.edge_attr, b.edge_index, b.rowptr, b.u_ref = fake, env.state_dim, fake, fake, fake, fake, fake
        b.row_index = fake if sb.num_obs else None
        b.num_edges, b.num_nodes, b.num_agents_total = E, B * sb.nodes_per_graph, B * sb.num_agents
        need = native.fn('gcbf_step_workspace_bytes')(ctypes.byref(d), ctypes.byref(b))
        relink = native.fn('gcbf_step_relink_workspace_bytes')(ctypes.byref(d), ctypes.byref(b), E)
        assert need > 0 and relink > 0, _C.lib().gcbf_last_error()
        sizes[cfg] = (need, relink)
        b.num_agents_total += 1                                   # inconsistent batch: rejected, not a crash
        assert native.fn('gcbf_step_workspace_bytes')(ctypes.byref(d), ctypes.byref(b)) == 0
    assert sizes['C2'][0] < sizes['C3'][0] < 80e9 and sizes['C3'][1] < 20e9
