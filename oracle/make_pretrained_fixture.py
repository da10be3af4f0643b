"""TEST INFRASTRUCTURE ONLY (build container only: needs /root/reference).

Known-answer fixtures on the reference's SHIPPED, TRAINED checkpoints (pretrained/<env>/models/step_500000/{cbf,actor}.pkl,
SURVEY 8a row a13): the unmodified reference (on oracle/shim) evaluates h and u with the trained weights on a seeded
synthetic batch large enough for the tensor-core layers of the product (>= 256 edges and agents).

Writes
  tests/golden/pretrained_<env>.pt          inputs' seeds, edge_index, h, u, masks (small, committed)
  tests/golden/pretrained_stats.pt          per-tensor statistics of all six checkpoints (shape, mean, std, absmax, row-norm range,
                                            quantiles) -- lets a test synthesise "trained-like" weights where the 98 MB files
                                            are absent
  tests/golden/pretrained_checkpoints.json  layout of all six checkpoint files (key order, shapes, state-dict metadata, file size)
                                            -- lets a test write checkpoints the shipped files' shape without their weights
  tests/golden/_pretrained/<env>/*.pkl      a byte copy of the checkpoint files for ONE env (git-ignored: weights are data, not
                                            history; the directory travels to the GPU box with the working tree)

    python oracle/make_pretrained_fixture.py
    python oracle/make_pretrained_fixture.py manifest     # only tests/golden/pretrained_checkpoints.json
"""
import os
import shutil
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import ref_harness  # noqa: E402

REF = '/root/reference'
CASES = {
    'DubinsCar': dict(n=64, obs=8, graphs=6, area=3.0, seed=501),
    'SimpleCar': dict(n=96, obs=0, graphs=4, area=3.5, seed=502),
    'SimpleDrone': dict(n=48, obs=48, graphs=4, area=1.6, seed=503),
}
SHIP_WEIGHTS = ('DubinsCar',)


def tensor_stats(t):
    t = t.double().reshape(t.shape[0], -1) if t.dim() > 1 else t.double().reshape(1, -1)
    flat = t.reshape(-1)
    q = torch.quantile(flat.abs()[:: max(1, flat.numel() // 200000)], torch.tensor([0.5, 0.9, 0.99, 0.999], dtype=torch.float64))
    rn = t.norm(dim=1)
    return dict(shape=tuple(t.shape), mean=float(flat.mean()), std=float(flat.std()) if flat.numel() > 1 else 0.0,
                absmax=float(flat.abs().max()), q_abs=q.tolist(), rownorm_min=float(rn.min()), rownorm_max=float(rn.max()),
                sigma_max=float(torch.linalg.matrix_norm(t, 2)) if min(t.shape) > 1 else float(rn.max()))


def main():
    synth = ref_harness._load_synth()
    out_dir = os.path.join(ROOT, 'tests', 'golden')
    stats = {}
    for env_name, c in CASES.items():
        ckpt = os.path.join(REF, 'pretrained', env_name, 'models', 'step_500000')
        sb = synth.make_states(env_name, c['n'], c['obs'], c['graphs'], c['area'], c['seed'])
        env, algo, graphs = ref_harness.build_reference(sb, 0, ckpt)
        from torch_geometric.data import Batch
        batch = Batch.from_data_list(graphs)
        with torch.no_grad():
            h = algo.cbf(batch).clone()          # one power iteration on the loaded u / v, as the reference's first forward does
            u = algo.actor(batch).clone()
            um, sm = env.unsafe_mask(batch).clone(), env.safe_mask(batch).clone()
        fix = dict(meta=dict(env=env_name, n=c['n'], obs=sb.num_obs, graphs=c['graphs'], area=c['area'], seed=c['seed'],
                             checkpoint=f'pretrained/{env_name}/models/step_500000'),
                   edge_index=batch.edge_index.clone(), u_ref=batch.u_ref.clone(), h=h, u=u, unsafe_mask=um, safe_mask=sm)
        torch.save(fix, os.path.join(out_dir, f'pretrained_{env_name}.pt'))
        st = {}
        for net in ('cbf', 'actor'):
            sd = torch.load(os.path.join(ckpt, f'{net}.pkl'), map_location='cpu')
            st[net] = {k: tensor_stats(v) for k, v in sd.items()}
        stats[env_name] = st
        print(f'{env_name}: E={batch.edge_index.shape[1]} agents={h.shape[0]} |h|max={h.abs().max():.4f} |u|max={u.abs().max():.4f} '
              f'unsafe={int(um.sum())} safe={int(sm.sum())} h>=0: {(h >= 0).float().mean():.3f}')
        if env_name in SHIP_WEIGHTS:
            dst = os.path.join(out_dir, '_pretrained', env_name)
            os.makedirs(dst, exist_ok=True)
            for f in ('cbf.pkl', 'actor.pkl'):
                shutil.copyfile(os.path.join(ckpt, f), os.path.join(dst, f))
                os.chmod(os.path.join(dst, f), 0o644)
    torch.save(stats, os.path.join(out_dir, 'pretrained_stats.pt'))
    checkpoint_manifest()


def checkpoint_manifest():
    import json
    out = {}
    for env_name in CASES:
        ckpt = os.path.join(REF, 'pretrained', env_name, 'models', 'step_500000')
        out[env_name] = {}
        for net in ('cbf', 'actor'):
            path = os.path.join(ckpt, f'{net}.pkl')
            sd = torch.load(path, map_location='cpu')
            assert all(v.dtype == torch.float32 for v in sd.values())
            out[env_name][net] = dict(file_bytes=os.path.getsize(path), keys=[[k, list(v.shape)] for k, v in sd.items()],
                                      metadata=getattr(sd, '_metadata', {}))
    path = os.path.join(ROOT, 'tests', 'golden', 'pretrained_checkpoints.json')
    with open(path, 'w') as f:
        json.dump(out, f, indent=1)
        f.write('\n')
    print(f'{path}: {os.path.getsize(path)} B')


if __name__ == '__main__':
    if sys.argv[1:] == ['manifest']:
        checkpoint_manifest()
    else:
        main()
