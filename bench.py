#!/usr/bin/env python
"""bench.py -- agent*steps/sec of the GCBF train step (one inner iteration of GCBF.update, reference
gcbf/algo/gcbf.py:158-226) on synthetic BASELINE.json configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C3] [--also C2,...|none] [--impl own|reference] [--dump-outputs DIR]

Workload     : `value` / `e2e` / `roofline` are measured on --config, by default C3 (DubinsCar n=1024, obs=32, B=64 per GPU) -- the
               largest single-GPU configuration of BASELINE.json.  `config.also` carries the same device-timed and end-to-end
               numbers for further BASELINE configs measured in the same run: C2 at every N, and under --gpus 8 the two
               configurations BASELINE.json defines over 8 GPUs -- C4 (SimpleDrone n=1024, 16 replicas = 2 per GPU) and C5
               (DubinsCar n=4096 dense, 8 graphs = 1 per GPU, gradient all-reduce).

own arm      : gcbf_b200 (sm_100a kernels through the C ABI).  `value` = device-timed throughput with the batch
               resident in HBM; `e2e` = the same step driven from pinned HOST buffers (H2D of the states, graph
               build, train step, D2H of the scalars) per step.
reference arm: the reference algorithm on the host CPU cores.  The reference is pure Python on torch_geometric, which
               cannot be installed on the GPU box, so this arm times oracle/gcbf_oracle.py (a port validated
               bit-for-bit against the reference in the build container) -- kind "port".
Outputs      : --dump-outputs DIR writes what the last timed step of --config handed its caller (rank 0's share) as DIR/<name>.npy,
               see step_outputs().  That step starts from the seeded weights and optimiser state (restored before it, outside the
               timed interval), so the same arguments give the same inputs on every run and two builds can be compared output for
               output: the weight-gradient reductions add in a run-dependent order, and clipped Adam grows those last-bit
               differences into visibly different weights within a few steps.
Multi-GPU    : one process per GPU (torchrun), environment-parallel: every rank trains on its own B graphs (weak
               scaling), one NCCL all-reduce of the flat gradient bucket per step.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.join(ROOT, 'gcbf-pytorch_b200'),):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

METRIC = 'agent*steps/sec (train step, device-timed)'
UNIT = 'agent*steps/s'


def read_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p['hbm_gbs'], bf16_tflops=p['bf16_tflops'], bf16_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """SM clock / throttle reasons sampled during the timed region.  In-process NVML polling thread (nvidia_ml_py, 20 ms
    period: an ioctl per sample, no process spawn inside the timed region); falls back to `nvidia-smi -lms 200`."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None
        self.thread, self.stop_flag, self.samples, self.reasons, self.max_mhz = None, False, [], set(), None

    def _nvml_loop(self, nv, handle):
        bits = {'hw_slowdown': getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8),
                'hw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
                'sw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20),
                'sw_power_cap': getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4)}
        get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(handle))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[self.index]) if vis and all(x.strip().isdigit() for x in vis.split(',')) else self.index
            handle = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '200',
                                          '-i', str(self.index)], stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            sm = self.samples
            return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': self.max_mhz, 'samples': len(sm),
                    'reasons': sorted(self.reasons), 'source': 'nvml thread, 20 ms'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            f = [x.strip() for x in line.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        os.unlink(self.path)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons), 'source': 'nvidia-smi -lms 200'}


def build_case(cfg_name, device, rank):
    from gcbf_b200 import synth
    from gcbf_b200.synth import seeded_algo
    c = dict(synth.CONFIGS[cfg_name])
    c['num_graphs'] = synth.GRAPHS_PER_GPU[cfg_name]
    c['seed'] = c['seed'] + 7919 * rank            # every rank owns different graphs (environment-parallel)
    sb = synth.make_states(**c)
    env, algo = seeded_algo(sb.env, sb.num_agents, device, 0, {'num_obs': sb.num_obs, 'area_size': sb.area_size})
    env.set_goal(sb.goals)
    if sb.env == 'DubinsCar':
        env._obs = sb.obs.to(device)
    return sb, env, algo


DUMP_MAX_ELEMS = 1 << 20        # per array: larger outputs are dumped as a fixed, seeded sample (all arrays together stay under 64 MB)


def step_outputs(res, algo):
    """What one train step hands its caller, copied to the host before the next step reuses the step's workspace: every tensor of
    the result dict (integer / float64 tensors as float64, the rest as float32) and the updated parameters (the flat bucket).
    An array of more than DUMP_MAX_ELEMS elements is replaced by the elements at a fixed, seeded, sorted set of flat indices."""
    arrays = dict(res, params=algo._bucket.flat)
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t.cpu()
        out[name] = (t.double() if t.dtype in (torch.int32, torch.int64, torch.float64) else t.float()).numpy()
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def train_state(algo):
    """Copies of everything a train step reads and rewrites: parameters, spectral-norm vectors, Adam moments and step count."""
    b = algo._ensure_bucket()
    return ([{k: v.clone() for k, v in m.state_dict().items()} for m in (algo.cbf, algo.actor)], b.exp_avg.clone(),
            b.exp_avg_sq.clone(), b.step)


def restore_train_state(algo, state):
    sds, exp_avg, exp_avg_sq, step = state
    for m, sd in zip((algo.cbf, algo.actor), sds):
        m.load_state_dict(sd)          # in-place copies: the library sees new weight versions and refreshes its fp16 companions
    b = algo._bucket
    b.exp_avg.copy_(exp_avg)
    b.exp_avg_sq.copy_(exp_avg_sq)
    b.step = step


def measure(cfg_name, args, dev, rank, world, dist, with_roofline, sampler=None, dump=False):
    """Device-timed and end-to-end throughput of one BASELINE config on this rank's share (max over ranks taken by the caller).
    With `dump`, the last timed step starts from the seeded state and its outputs are returned (step_outputs)."""
    from gcbf_b200 import _C, ops
    sb, env, algo = build_case(cfg_name, dev, rank)
    algo.process_group = None
    B, n = sb.num_graphs, sb.num_agents
    data = env.graph_from_states(sb.states.to(dev))
    E = int(data.edge_index.shape[1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    seeded = train_state(algo) if dump else None
    # ---- device-timed region: batch resident in HBM ---------------------------------------------------------
    for _ in range(args.warmup):
        algo.train_step(data)
    barrier()
    if sampler is not None:
        sampler.start()
    _C.reset_counters()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pause0, pause1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        if seeded is not None and i == args.steps - 1:
            pause0.record()
            restore_train_state(algo, seeded)
            pause1.record()
        res = algo.train_step(data)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1) - (pause0.elapsed_time(pause1) if seeded is not None else 0.0)
    launches = _C.kernel_launches()
    clocks = sampler.stop() if sampler is not None else None
    scal = res['scalars'].tolist()
    outputs = step_outputs(res, algo) if dump else None
    # ---- end-to-end: host buffers in, scalars out, every step ---------------------------------------------------
    host_states = sb.states.pin_memory()
    h2d = host_states.numel() * 4
    out_host = torch.empty(args.steps + 2, 8, dtype=torch.float32).pin_memory()   # one pinned row per step

    def e2e_step(i=0):
        st = host_states.to(dev, non_blocking=True)
        g = env.graph_from_states(st)                    # radius graph + edge features + u_ref (K1, K2, K5); syncs on the edge count
        r = algo.train_step(g)
        # D2H read of the step's result: an asynchronous copy into this step's pinned row (as a training loop logs its
        # losses); every row has landed when the timed region is closed by the synchronize below
        out_host[i].copy_(r['scalars'], non_blocking=True)

    e2e_runs = []
    if not args.no_e2e:
        for i in range(2):
            e2e_step(i)
        # this leg synchronises with the host every step (edge counts), so one host hiccup on a shared box moves a K = 10 total
        # by tens of percent: the K steps are timed three times back to back and the MEDIAN total is reported (all are kept)
        for _rep in range(3):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                e2e_step(2 + i)
            e1.record()
            barrier()
            e2e_runs.append(e0.elapsed_time(e1))
            assert bool(torch.isfinite(out_host[2:2 + args.steps]).all()), 'e2e results did not reach the host'
    ms_e2e = statistics.median(e2e_runs) if e2e_runs else 0.0

    gemm, ms_instr = None, None
    if with_roofline:
        # roofline pass: the same steps again with a CUDA-event pair around every GEMM launch (the event records slow the host
        # down, so this pass is kept out of the throughput measurement above).  The side stream is switched off here: with two
        # streams the GEMMs of the two nets overlap and a per-launch event pair would time the kernel plus whatever shares the
        # GPU with it.
        two_streams = os.environ.get('GCBF_TWO_STREAMS')
        os.environ['GCBF_TWO_STREAMS'] = '0'
        algo.train_step(data)
        ops.GEMM_TIMER.enable()
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record()
        for _ in range(args.steps):
            algo.train_step(data)
        ev3.record()
        barrier()
        ms_instr = ev2.elapsed_time(ev3)
        gemm = ops.GEMM_TIMER.summary()
        ops.GEMM_TIMER.disable()
        if two_streams is None:
            del os.environ['GCBF_TWO_STREAMS']
        else:
            os.environ['GCBF_TWO_STREAMS'] = two_streams

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    # edges of all ranks (every rank owns different graphs)
    et = torch.tensor([E], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(et)
    del algo, data
    return dict(sb=sb, B=B, n=n, E=E, E_total=int(et.item()), ms=ms, ms_e2e=ms_e2e, e2e_runs=e2e_runs, h2d=h2d, launches=launches, clocks=clocks,
                scal=scal, gemm=gemm, ms_instr=ms_instr, outputs=outputs)


def rollout_leg(cfg_name, dev, steps=20):
    """Vectorised data collection (SURVEY 8f-2, gcbf_b200/algo/rollout.py): all graphs of the config as independent environments,
    one vector step = u_ref + ONE radius graph + ONE actor forward + masks + dynamics + replay append for all of them.  The
    reference steps one 16-agent env per ~5 ms of host time (SURVEY section 6)."""
    from gcbf_b200.algo.rollout import VectorRollout
    sb, env, algo = build_case(cfg_name, dev, 0)
    B, n = sb.num_graphs, sb.num_agents
    algo.use_device_replay(capacity=(steps + 4) * B)      # ring sized up front: no regrowth inside the timed loop
    goals = sb.goals.repeat(B, 1)
    vr = VectorRollout(env, algo, B, states=sb.states, goals=goals)
    for _ in range(3):
        vr.step(prob=0.5)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        vr.step(prob=0.5)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    ms = e0.elapsed_time(e1) / steps
    return {'workload': f'{cfg_name}: {B} environments x {n} agents per vector step (actor forward, env step, masks, replay append)',
            'ms_per_vector_step': round(ms, 4), 'wall_ms_per_vector_step': round(wall, 4), 'env_steps_per_s': round(B / (wall / 1e3), 1),
            'agent_steps_per_s': round(B * n / (wall / 1e3), 1), 'host_syncs_per_vector_step': 1}


def controller_leg(cfg_name, dev, calls=5):
    """Test-time controller (SURVEY 8f-1, GCBF.apply = gcbf_apply in csrc/apply.cu) on ONE graph of the config: wall time per call
    with the reference's settings (lr 0.1, rand 30, up to 31 Adam rounds); random-init weights violate the h_dot condition
    somewhere, so the refinement loop runs (rounds reported)."""
    sb, env, algo = build_case(cfg_name, dev, 0)
    single = env.graph_from_states(sb.states[:sb.nodes_per_graph].to(dev))
    algo.apply(single)
    torch.cuda.synchronize()
    rounds = []
    t0 = time.perf_counter()
    for _ in range(calls):
        algo.apply(single)
        rounds.append(getattr(algo, 'last_apply_rounds', -1))
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / calls * 1e3
    per_round = wall / max(1.0, sum(rounds) / len(rounds) + 2)      # + the two passes before the loop
    return {'workload': f'{cfg_name}: GCBF.apply on one graph ({sb.num_agents} agents, {int(single.edge_index.shape[1])} edges)',
            'wall_ms_per_call': round(wall, 3), 'adam_rounds': rounds, 'wall_ms_per_round': round(per_round, 3)}


def shape_traffic(dom):
    """DRAM bytes per launch of the dominant launch shape from the committed `ncu --set full` capture of exactly that shape
    (profiles/r02_gemm_h_ncu_full.json: {"launches": [{"product", "M", "N", "K", "dram_read_bytes", "dram_write_bytes"}, ...]});
    None when no capture of this shape exists -- never a number taken from a different launch."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r02_gemm_h_ncu_full.json')) as f:
            caps = json.load(f)['launches']
    except Exception:
        return None, None
    for c in caps:
        if c.get('product') == dom['product'] and (c.get('M'), c.get('N'), c.get('K')) == (dom['M'], dom['N'], dom['K']):
            return int(c['dram_read_bytes'] + c['dram_write_bytes']), c.get('source', 'profiles/r02_gemm_h_ncu_full.json')
    return None, None


def run_own(args):
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    main_cfg = args.config
    if args.also == 'auto':
        # one GPU: every other BASELINE config as its per-GPU share (C1; C2; C4 = 2 of the 16 replicas; C5 = 1 of the 8 dense graphs), so
        # that the single-GPU line carries the whole config table; 8 GPUs: the two configs BASELINE defines over 8 GPUs
        extra_cfgs = ['C2', 'C1', 'C4', 'C5'] if world == 1 else (['C2', 'C4', 'C5'] if world == 8 else ['C2'])
        also = [c for c in extra_cfgs if c != main_cfg]
    else:
        also = [c for c in args.also.split(',') if c and c != 'none' and c != main_cfg]

    gpu_leg_threads()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    m = measure(main_cfg, args, dev, rank, world, dist, True, sampler, dump=args.dump_outputs is not None)
    extra = {}
    for c in also:
        if world == 1:
            try:                                                  # an extra config never costs the headline line (single process: no
                r = measure(c, args, dev, rank, world, dist, False, None)      # collective another rank could be left waiting in)
            except Exception as ex:
                extra[c] = {'error': repr(ex)[:300]}
                continue
        else:
            r = measure(c, args, dev, rank, world, dist, False, None)
        agents_c = r['B'] * r['n'] * world
        extra[c] = {'workload': f"{c}: {r['sb'].env} n={r['n']} obs={r['sb'].num_obs} B={r['B']}/GPU area={r['sb'].area_size}",
                    'agents_per_step': agents_c, 'edges_per_step': r['E_total'], 'ms_per_step': round(r['ms'] / args.steps, 4),
                    'value': round(agents_c * args.steps / (r['ms'] / 1e3), 1), 'unit': UNIT,
                    'e2e': ({'value': round(agents_c * args.steps / (r['ms_e2e'] / 1e3), 1), 'ms_per_step': round(r['ms_e2e'] / args.steps, 4),
                             'h2d_bytes_per_step': r['h2d'], 'd2h_bytes_per_step': 32} if r['e2e_runs'] else None),
                    'gpu_launches': r['launches'], 'loss': round(r['scal'][6], 6)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    sb, B, n, E, ms, ms_e2e, gemm, ms_instr = m['sb'], m['B'], m['n'], m['E'], m['ms'], m['ms_e2e'], m['gemm'], m['ms_instr']
    peaks = read_peaks()
    agents = B * n * world
    value = agents * args.steps / (ms / 1e3)
    # dominant kernel: gemm_h_kernel (tcgen05 kind::f16).  Peak = measured dense bf16/fp16 tensor throughput inside a long
    # step (sustained).  `achieved` counts the ALGORITHMIC fp32 FLOPs (2*M*N*K per product); the kernel issues 3 fp16 MMAs
    # per product (hi*hi + hi*lo + lo*hi), so the tensor pipe itself runs at 3x that: `frac_issued`.
    f16_peak = peaks['bf16_sustained']
    achieved_tflops = gemm['flops'] / max(gemm['ms'], 1e-9) / 1e9
    incl_prep = gemm['flops'] / max(gemm['ms'] + gemm.get('prep_ms', 0.0), 1e-9) / 1e9
    roofline = {'bound': 'tensor', 'kernel': gemm['kernel'], 'achieved': round(achieved_tflops, 2), 'peak': round(f16_peak, 1),
                'unit': 'TFLOP/s', 'frac': round(achieved_tflops / f16_peak, 4),
                'frac_issued': round(3 * achieved_tflops / f16_peak, 4) if gemm['tensor'] else None,
                'achieved_incl_operand_prep': round(incl_prep, 2),
                'peak_source': f"{peaks['source']}: bf16_tflops_sustained = dense 16-bit tensor throughput",
                'launches_timed': gemm['launches'], 'gemm_share_of_step': round(gemm['ms'] / ms_instr, 4),
                'prep_share_of_step': round(gemm.get('prep_ms', 0.0) / ms_instr, 4),
                'instrumented_ms_per_step': round(ms_instr / args.steps, 4),
                'whole_step_flops': gemm['flops'] / args.steps,
                'whole_step_frac': round(gemm['flops'] / args.steps / (ms / args.steps) / 1e9 / f16_peak, 4),
                'instrumented_pass': 'single stream, CUDA-event pair per GEMM / operand-prep launch', 'traffic': None}
    dom = gemm.get('dominant')
    if dom:
        # the launch shape that takes the most GEMM time: algorithmic FLOPs and bytes per launch (companions in: 2 planes x
        # 2 B per element of each operand; fp32 out) against its CUDA-event duration; DRAM traffic only from a committed
        # `ncu --set full` capture of exactly this launch shape
        M_, N_, K_ = dom['M'], dom['N'], dom['K']
        out_elems = {'forward': M_ * N_, 'data-grad': M_ * K_, 'weight-grad': N_ * K_}[dom['product']]
        in_elems = {'forward': M_ * K_ + N_ * K_, 'data-grad': M_ * N_ + N_ * K_, 'weight-grad': M_ * N_ + M_ * K_}[dom['product']]
        alg_bytes = 4 * in_elems + 4 * out_elems
        tf = dom['flops_per_launch'] / dom['ms_per_launch'] / 1e9
        roofline['dominant_launch'] = {
            'shape': f"{dom['product']} M={M_} N={N_} K={K_}", 'launches': dom['launches'],
            'flops_per_launch': dom['flops_per_launch'], 'ms_per_launch': round(dom['ms_per_launch'], 4),
            'achieved': round(tf, 1), 'frac': round(tf / f16_peak, 4), 'frac_issued': round(3 * tf / f16_peak, 4),
            'algorithmic_bytes_per_launch': alg_bytes}
        roofline['traffic'], src = shape_traffic(dom)
        if src:
            roofline['traffic_source'] = src
    line = {
        'metric': METRIC, 'value': round(value, 1), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': round(ms / args.steps, 4), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 via 3xfp16 tensor-core products (fp32 accumulate)' if gemm['tensor'] else 'f32', 'data': 'synthetic',
        'config': {'workload': f'{main_cfg}: {sb.env} n={n} obs={sb.num_obs} B={B}/GPU area={sb.area_size}',
                   'agents_per_step': agents, 'edges_per_gpu': E, 'parallelism': f'dp{world}',
                   'l2': 'no flush: per-step working set (>= 0.2 GB of activations per 2048-wide layer + 98 MB weights) '
                         'exceeds the 126 MB L2',
                   'also': extra},
        'clocks': m['clocks'],
        'e2e': ({'value': round(agents * args.steps / (ms_e2e / 1e3), 1), 'unit': UNIT, 'h2d_bytes_per_step': m['h2d'],
                 'd2h_bytes_per_step': 32, 'ms_per_step': round(ms_e2e / args.steps, 4), 'statistic': 'median of 3 timed K-step runs',
                 'ms_per_step_runs': [round(x / args.steps, 4) for x in m['e2e_runs']]} if m['e2e_runs'] else None),
        'gpu_launches': m['launches'],
        'roofline': roofline,
        'loss': round(m['scal'][6], 6),
    }
    if world == 1 and not args.no_e2e:
        try:
            line['rollout'] = [rollout_leg(main_cfg, dev), rollout_leg('C1x256', dev)]
            line['controller'] = [controller_leg('C1', dev), controller_leg(main_cfg, dev)]
        except Exception as ex:                                   # the rollout leg is an extra: never lose the bench line over it
            line['rollout'] = {'error': repr(ex)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        line['cpu_baseline'] = cpu_baseline(main_cfg, budget_s=25.0)
    if args.dump_outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in m['outputs'].items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def cpu_quota():
    """CPUs this container may use per scheduler period (cgroup v2 cpu.max, v1 cpu.cfs_quota_us), or None if unlimited.  The GPU
    boxes of this pool report 128 logical CPUs but a quota of 16: threads beyond it only get the whole process group throttled
    (measured: 50 ms stalls every 100 ms period in the rollout loop, /sys/fs/cgroup/cpu.stat nr_throttled)."""
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            q, p = f.read().split()[:2]
        if q != 'max':
            return float(q) / float(p)
    except Exception:
        pass
    try:
        with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
            q = int(f.read())
        with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
            p = int(f.read())
        if q > 0:
            return q / p
    except Exception:
        pass
    return None


def host_threads():
    """torch intra-op threads for the CPU legs: the physical cores of the box, capped by the container's CPU quota (torchrun
    exports OMP_NUM_THREADS=1, which would pin the reference arm to a single core)."""
    n = max(1, (os.cpu_count() or 2) // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    q = cpu_quota()
    if q:
        n = max(1, min(n, int(q)))
    torch.set_num_threads(n)
    return torch.get_num_threads()


def gpu_leg_threads():
    """The GPU legs need one host thread; torch's default (one intra-op thread per logical CPU, spinning after every parallel region)
    burns the container's CPU quota and gets the launching thread throttled with it."""
    q = cpu_quota()
    torch.set_num_threads(max(1, min(4, int(q) if q else 4)))


def cpu_sample_step(cfg_name, graphs):
    """Callable running ONE reference train step (oracle port) on the first `graphs` graphs of the config."""
    host_threads()
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import gcbf_oracle as O                      # the ONLY use of oracle/ in bench.py: the CPU baseline
    from gcbf_b200 import synth
    from helpers import oracle_batch, sd_clone, seeded_algo
    c = dict(synth.CONFIGS[cfg_name])
    c['num_graphs'] = graphs
    sb = synth.make_states(**c)
    _, algo = seeded_algo(sb.env, sb.num_agents, torch.device('cpu'), 0, {'num_obs': sb.num_obs, 'area_size': sb.area_size})
    cbf, act = sd_clone(algo.cbf), sd_clone(algo.actor)
    ob = oracle_batch(sb)
    oc, oa = {}, {}

    def step():
        O.update_step(sb.env, cbf, act, oc, oa, sb.states, sb.goals, ob['edge_index'], ob['u_ref'], sb.num_graphs,
                      sb.num_agents, sb.num_obs, K=ob['K'])
    return step, sb


def cpu_baseline(cfg_name, budget_s=20.0):
    from gcbf_b200 import synth
    full = synth.GRAPHS_PER_GPU[cfg_name]
    graphs = max(1, min(full, 4))
    step, sb = cpu_sample_step(cfg_name, graphs)
    step()                                       # warm-up
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < 3 or (time.perf_counter() < t_end and len(times) < 10):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() > t_end and len(times) >= 2:
            break
    t = statistics.median(times)
    return {'value': round(graphs * sb.num_agents / t, 1), 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': f'{graphs} of {full} graphs of {cfg_name} ({sb.env} n={sb.num_agents}), median of {len(times)} steps, '
                      f'{t:.2f} s/step; host has {os.cpu_count()} logical CPUs, container CPU quota {cpu_quota()}',
            'seconds_per_step': round(t, 3)}


def run_reference(args):
    """Reference arm: the reference's algorithm (oracle port, kind "port": torch_geometric cannot be installed on the box) on
    the host cores, same config / metric / K / W as the own arm.  Every step runs as many of the config's graphs as fit a
    ~150 s budget for the whole K + W run (all of them when that fits: C2 does, C3's 64 graphs do not)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from gcbf_b200 import synth
    full = synth.GRAPHS_PER_GPU[args.config]
    steps, warmup = args.steps, args.warmup
    probe = min(full, 2)
    step, sb = cpu_sample_step(args.config, probe)
    step()
    t0 = time.perf_counter()
    step()
    per_graph = (time.perf_counter() - t0) / probe
    budget = float(os.environ.get('GCBF_REF_BUDGET_S', '150'))
    graphs = int(max(1, min(full, budget / max(1, steps + warmup) / per_graph)))
    if graphs != probe:
        step, sb = cpu_sample_step(args.config, graphs)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    value = graphs * sb.num_agents * steps / dt
    world = int(os.environ.get('WORLD_SIZE', '1'))
    sample = ((f'all {full} graphs per step' if graphs == full else f'{graphs} of {full} graphs per step (bounded sample)') + f', {steps} steps'
              + f'; host has {os.cpu_count()} logical CPUs, container CPU quota {cpu_quota()}')
    line = {'impl': 'reference', 'metric': METRIC, 'value': round(value, 1), 'unit': UNIT, 'n_gpus': world, 'steps': steps,
            'warmup': warmup, 'ms_per_step': round(dt / steps * 1e3, 2), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'{args.config}: {sb.env} n={sb.num_agents} obs={sb.num_obs} B={full}/GPU area={sb.area_size}',
                       'graphs_per_step': graphs, 'graphs_in_config': full, 'same_config': graphs == full},
            'cpu_baseline': {'value': round(value, 1), 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port', 'sample': sample},
            'e2e': {'value': round(value, 1), 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def run_macbf(args):
    """`--macbf`: the MACBF baseline's train step (SURVEY 8f-4; not the headline metric) at the reference's own training scale and at
    C3's shape, device-timed (tools/macbf_probe.py), with the CPU port of the same step timed beside it on the first workload."""
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import macbf_probe
    dev = torch.device('cuda', 0)
    out = {}
    for name in macbf_probe.WORKLOADS:
        rec, (sb, algo, data) = macbf_probe.measure(name, dev, steps=args.steps, warmup=args.warmup)
        if name == 'ref' and not args.no_cpu_baseline:
            host_threads()
            sys.path.insert(0, os.path.join(ROOT, 'oracle'))
            import macbf_oracle as MO                # CPU baseline leg: the only use of oracle/ on this path
            cbf = {k: v.detach().cpu().clone() for k, v in algo.cbf.state_dict().items()}
            act = {k: v.detach().cpu().clone() for k, v in algo.actor.state_dict().items()}
            ei, ur = data.edge_index.cpu(), data.u_ref.cpu()
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                MO.update_step(sb.env, cbf, act, {}, {}, sb.states, sb.goals, ei, ur, sb.num_graphs, sb.num_agents, sb.num_obs)
                ts.append(time.perf_counter() - t0)
            t = statistics.median(ts)
            rec['cpu_baseline'] = {'value': round(rec['agents'] / t, 1), 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
                                   'sample': f'the same batch (graph given), median of 5 steps, {t:.3f} s/step'}
        out[name] = rec
    print(json.dumps({'metric': 'agent*steps/sec (MACBF train step, device-timed)', 'unit': UNIT, 'n_gpus': 1, 'higher_is_better': True,
                      'data': 'synthetic', 'dtype': 'f32', 'value': out['ref']['agent_steps_per_s'], 'ms_per_step': out['ref']['train_step_ms'],
                      'config': {'workload': 'MACBF ' + out['ref']['workload'], 'also': {'C3': out['C3']}},
                      'gpu_launches': out['ref']['gpu_launches_per_step'], 'cpu_baseline': out['ref'].get('cpu_baseline'), 'detail': out['ref']}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--config', default='C3', help='BASELINE config `value` is measured on (default: the largest single-GPU one)')
    ap.add_argument('--also', default='auto', help="further configs reported under config.also: comma list, 'none', or 'auto' (C2; plus C4, C5 at 8 GPUs)")
    ap.add_argument('--impl', default='own', choices=['own', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true', help='skip the host-buffer leg (profiling runs under ncu only)')
    ap.add_argument('--macbf', action='store_true', help='measure the MACBF baseline train step instead (SURVEY 8f-4; single GPU, own arm only)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed train step of --config as DIR/<name>.npy (own arm, GCBF only)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs is not None and (args.impl != 'own' or args.macbf):
        ap.error('--dump-outputs writes the outputs of the GCBF train step of the own arm (not with --impl reference or --macbf)')
    if args.impl == 'reference':
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py (own arm) needs a CUDA device: the gcbf_b200 path has no CPU fallback')
        if args.macbf:
            run_macbf(args)
        else:
            run_own(args)


if __name__ == '__main__':
    main()
