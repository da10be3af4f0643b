"""TEST INFRASTRUCTURE ONLY (build container only).  Generates tests/golden/*.pt from the UNMODIFIED reference
running on oracle/shim (oracle/ref_harness.py).  Inputs are reproducible from (config, seeds) via
gcbf_b200/synth.py and a seeded module construction, so the fixtures hold only outputs + weight digests.

    python oracle/make_golden.py            # regenerate every GCBF case
    python oracle/make_golden.py macbf      # regenerate the MACBF cases (tests/golden/macbf_*.pt)
    python oracle/make_golden.py live       # regenerate tests/golden/reference_runs.json
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness  # noqa: E402

CASES = {
    'simplecar_n16_b3_dense': dict(env='SimpleCar', n=16, obs=0, graphs=3, area=1.5, seed=11),
    'dubins_n16_o4_b3': dict(env='DubinsCar', n=16, obs=4, graphs=3, area=2.0, seed=12),
    'drone_n8_b2': dict(env='SimpleDrone', n=8, obs=8, graphs=2, area=1.0, seed=13),
    'dubins_n16_o4_b1_freeze': dict(env='DubinsCar', n=16, obs=4, graphs=1, area=3.0, seed=14),
    'simplecar_c1': dict(env='SimpleCar', n=16, obs=0, graphs=1, area=4.0, seed=1001),
    'simplecar_isolated': dict(env='SimpleCar', n=4, obs=0, graphs=2, area=50.0, seed=15),
}
# MACBF baseline (SURVEY 8f-4): env built with max_neighbors = 12, per-edge h and masks; the nets are small, so the fixtures carry
# the full initial state dicts (final ones as digests)
MACBF_CASES = {
    'macbf_dubins_n24_o6_b3': dict(env='DubinsCar', n=24, obs=6, graphs=3, area=1.6, seed=21),       # dense: the top-12 filter cuts
    'macbf_simplecar_n20_b3': dict(env='SimpleCar', n=20, obs=0, graphs=3, area=1.2, seed=22),       # dense: torch_cluster's cap cuts
    'macbf_drone_n10_b2': dict(env='SimpleDrone', n=10, obs=10, graphs=2, area=0.8, seed=23),
    'macbf_dubins_sparse_b2': dict(env='DubinsCar', n=16, obs=4, graphs=2, area=6.0, seed=24),       # nodes without incoming edges
    'macbf_dubins_single': dict(env='DubinsCar', n=16, obs=4, graphs=1, area=2.0, seed=25),          # one graph: reach-freeze branch
}
INIT_SEED = 0
STEPS = 2
# intra-op threads of every fixture run: MKL's QR inside the seeded orthogonal_ initialisation rounds differently at other thread
# counts, so tests/test_oracle_cpu.py runs the port at this count too
THREADS = 8
# one train step from seed 5, compared bit for bit (tests/test_oracle_cpu.py::test_port_matches_live_reference); the post-step
# state dicts are stored as per-tensor SHA-256 of their float32 bytes, which keeps the comparison exact at a few kB
LIVE_CASES = [('SimpleCar', 12, 0, 2, 2.0), ('DubinsCar', 10, 3, 2, 2.0), ('SimpleDrone', 6, 6, 2, 1.0)]
LIVE_SEED = 5


def digest(sd):
    return {k: dict(sum=float(v.double().sum()), abssum=float(v.double().abs().sum()),
                    head=v.reshape(-1)[:4].clone()) for k, v in sd.items()}


def sha256(t):
    import hashlib
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


def main():
    synth = ref_harness._load_synth()
    out_dir = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)
    for name, c in CASES.items():
        sb = synth.make_states(c['env'], c['n'], c['obs'], c['graphs'], c['area'], c['seed'])
        if c['env'] == 'DubinsCar' and name.endswith('freeze'):
            # put two agents on their goals so the single-graph reach-freeze branch is exercised
            sb.states[0, :2] = sb.goals[0, :2]
            sb.states[3, :2] = sb.goals[3, :2] + 0.01
        res = ref_harness.run_reference(sb, INIT_SEED, None, STEPS)
        fix = dict(
            meta=dict(c, init_seed=INIT_SEED, steps=STEPS, num_obs=sb.num_obs, case=name),
            states=sb.states, goals=sb.goals,
            edge_index=res['edge_index'], u_ref=res['u_ref'], edge_attr=res['edge_attr'],
            h_probe=res['h_probe'], u_probe=res['u_probe'], unsafe_mask=res['unsafe_mask'],
            safe_mask=res['safe_mask'], states_next_probe=res['states_next_probe'], apply_action=res['apply_action'],
            steps=res['steps'], cbf_init=digest(res['cbf_init']), actor_init=digest(res['actor_init']),
            cbf_final=digest(res['cbf_final']), actor_final=digest(res['actor_final']),
        )
        path = os.path.join(out_dir, name + '.pt')
        torch.save(fix, path)
        s = res['steps'][-1]['scalars']
        print(f'{name}: E={res["edge_index"].shape[1]} unsafe={int(res["unsafe_mask"].sum())} '
              f'safe={int(res["safe_mask"].sum())} loss_hdot={s["loss/derivative"]:.6f} -> {os.path.getsize(path)} B')


def main_macbf():
    synth = ref_harness._load_synth()
    out_dir = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
    for name, c in MACBF_CASES.items():
        sb = synth.make_states(c['env'], c['n'], c['obs'], c['graphs'], c['area'], c['seed'])
        if name.endswith('single'):
            sb.states[0, :2] = sb.goals[0, :2]
        res = ref_harness.run_reference(sb, INIT_SEED, None, STEPS, algo_name='macbf')
        fix = dict(meta=dict(c, init_seed=INIT_SEED, steps=STEPS, num_obs=sb.num_obs, case=name, algo='macbf', max_neighbors=12),
                   states=sb.states, goals=sb.goals, **{k: res[k] for k in (
                       'edge_index', 'u_ref', 'edge_attr', 'h_probe', 'u_probe', 'unsafe_mask', 'safe_mask', 'states_next_probe',
                       'apply_action', 'steps', 'cbf_init', 'actor_init')},
                   cbf_final=digest(res['cbf_final']), actor_final=digest(res['actor_final']))
        path = os.path.join(out_dir, name + '.pt')
        torch.save(fix, path)
        s = res['steps'][-1]['scalars']
        deg = torch.bincount(res['edge_index'][1]).max() if res['edge_index'].numel() else 0
        print(f'{name}: E={res["edge_index"].shape[1]} max in-degree={int(deg)} unsafe={int(res["unsafe_mask"].sum())} '
              f'safe={int(res["safe_mask"].sum())} loss_hdot={s["loss/derivative"]:.6f} -> {os.path.getsize(path)} B')


def reference_buffer_sampling():
    """The reference's replay buffer (gcbf/algo/buffer.py): appends, seeded segment sampling (balanced and not), a merge."""
    import random
    import numpy as np
    from ref_loader import load_reference
    load_reference()
    from gcbf.algo.buffer import Buffer
    buf, other = Buffer(), Buffer()
    for i in range(90):
        buf.append(i, i % 4 != 0)
    for i in range(200, 230):
        other.append(i, i % 3 == 0)
    out = []
    for seed, (n, m, bal) in enumerate([(12, 3, False), (16, 3, True), (7, 1, False), (20, 5, True)]):
        np.random.seed(seed)
        random.seed(seed)
        out.append(buf.sample(n, m, bal))
    buf.merge(other)
    np.random.seed(9)
    random.seed(9)
    out.append(buf.sample(24, 3, True))
    out.append([buf.size, buf.safe_data[-3:], buf.unsafe_data[-3:]])
    return out


def main_live():
    """tests/golden/reference_runs.json: what the CPU tests compare the port and the replay buffers against."""
    import json
    synth = ref_harness._load_synth()
    cases = []
    for env_name, n, obs, graphs, area in LIVE_CASES:
        sb = synth.make_states(env_name, n, obs, graphs, area, LIVE_SEED)
        res = ref_harness.run_reference(sb, 0, None, 1)
        cases.append(dict(env=env_name, n=n, obs=obs, graphs=graphs, area=area, seed=LIVE_SEED,
                          edge_index=res['edge_index'].tolist(), h_probe=res['h_probe'].tolist(), u_probe=res['u_probe'].tolist(),
                          cbf_final_sha256={k: sha256(v) for k, v in res['cbf_final'].items()},
                          actor_final_sha256={k: sha256(v) for k, v in res['actor_final'].items()}))
        print(f'{env_name}: E={res["edge_index"].shape[1]} agents={res["h_probe"].shape[0]}')
    path = os.path.join(os.path.dirname(HERE), 'tests', 'golden', 'reference_runs.json')
    with open(path, 'w') as f:
        json.dump(dict(train_step=cases, buffer_sampling=reference_buffer_sampling()), f, indent=1)
        f.write('\n')
    print(f'{path}: {os.path.getsize(path)} B')


if __name__ == '__main__':
    torch.set_num_threads(THREADS)
    if len(sys.argv) > 1 and sys.argv[1] == 'macbf':
        main_macbf()
    elif len(sys.argv) > 1 and sys.argv[1] == 'live':
        main_live()
    else:
        main()
