#!/usr/bin/env python
"""Benchmark of the HandyRL learner hot path on B200 (DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one learner step on one replay batch: Batcher output -> net forward -> fused loss
fwd+bwd kernel -> net backward -> [all-reduce SUM] -> clip + Adam.
metric = learner samples/s = B*T*steps/s over all GPUs (BASELINE.json).

  value        inputs already resident in HBM (a ring of distinct batches larger than L2)
  e2e          the same step through LearnerStep.step() with HOST (pinned) batches: one H2D copy per step (on a copy
               stream, one step ahead of the compute) and a D2H read of the step's loss sums inside the timed region
  e2e_trainer  (N=1) the whole drop-in Trainer fed by a deque of episodes in the reference's wire format: episode
               decode + upload by the feeder thread, window sampling, gather/pad kernel, step, epoch hand-offs --
               the part `e2e` starts after (Batcher.batch, reference train.py:317-318, 358)
  roofline     the fused loss kernel: algorithmic bytes / CUDA-event duration measured live in the timed region,
               against the measured HBM copy bandwidth (MEASURED_PEAKS.json); roofline_wide_rows: the same kernel alone
               at the wide-row shape (roofline_wide_rows_bf16: with bf16 logit / gradient I/O); roofline_k2: the replay
               gather/pad kernel alone; roofline_net_gemm (nets on the fused tower engine): the three tensor-core products
               of one tower layer alone, bound = tensor, against the measured bf16 peak and the 3xTF32 ceiling peak/6
  cpu_baseline / --impl reference: the eager-PyTorch CPU port of the reference learner step (oracle/torch_learner.py,
               pinned to the reference's golden vectors) on the host cores: ALWAYS the workload's full batch, a fixed
               thread count, 3+ warm-ups, min / median / mean, loss-only and full step reported separately.

--dump-outputs DIR writes what the last timed step of `value` handed back -- its six loss sums and the model state --
as DIR/<name>.npy; the inputs depend on the arguments only, so two builds run with the same arguments can be compared.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[0]: the reference's own config.yaml shape -- TicTacToe episodes, batch_size 64, forward_steps 16,
    # V-Trace (CPU-runnable case; episodes from handyrl_b200.synthetic.tictactoe_episodes in the reference's wire format)
    'cfg1': dict(B=64, T=16, P=2, A=9, turn_based=True, observation=False, obs_shape=(3, 3, 3), net='tictactoe',
                 policy_target='VTRACE', value_target='VTRACE', reward_kind='zero', episodes=True,
                 desc='configs[0]: TicTacToe net (29,006 params), self-play episodes, batch_size=64 forward_steps=16, V-Trace'),
    # BASELINE.json configs[1]: TicTacToe net, synthetic replay (T=32,B=512,P=2), V-Trace + UPGO
    'cfg2': dict(B=512, T=32, P=2, A=9, turn_based=True, observation=False, obs_shape=(3, 3, 3), net='tictactoe',
                 policy_target='UPGO', value_target='VTRACE', reward_kind='zero',
                 desc='configs[1]: TicTacToe net (29,006 params), synthetic replay T=32 B=512/GPU P=2 Pa=1 A=9, '
                      'policy UPGO + value V-Trace'),
    # BASELINE.json configs[2]: the Geister architecture (DRC ConvLSTM 3 layers x 3 repeats, 231,604 params; dict observation;
    # policy/value/return heads), TD(lambda), batch 256, burn-in 4 + 16 forward steps
    'cfg3': dict(B=256, T=20, P=2, A=214, turn_based=True, observation=True, obs_shape=None, net='geister', burn_in=4,
                 policy_target='TD', value_target='TD', reward_kind='step',
                 desc='configs[2]: Geister net (DRC ConvLSTM, 231,604 params, recurrent path), TD(lambda), B=256/GPU, '
                      'T=4 burn-in + 16, P=Pa=2, A=214, dict observation {scalar 18, board 7x6x6}'),
    # BASELINE.json configs[3]: Hungry Geese architecture (12-block torus tower, 116,928 params), V-Trace, batch 1024 over 4 GPUs
    'cfg4': dict(B=256, T=32, P=4, A=4, turn_based=False, observation=False, obs_shape=(17, 7, 11), net='geese',
                 policy_target='VTRACE', value_target='VTRACE', reward_kind='zero',
                 desc='configs[3]: Hungry Geese net (torus conv tower, 116,928 params), V-Trace, B=256/GPU (1024 over 4 GPUs), '
                      'T=32, P=Pa=4, A=4, obs 17x7x11'),
    # per-GPU shard of BASELINE.json configs[4]: 64x64 obs, 512 actions, T=64, B=4096/8
    'cfg5shard': dict(B=512, T=64, P=2, A=512, turn_based=True, observation=False, obs_shape=(1, 64, 64), net='wide',
                      policy_target='UPGO', value_target='VTRACE', reward_kind='zero',
                      desc='configs[4] per-GPU shard: 64x64 obs / 512 actions, T=64 B=512/GPU P=2 Pa=1'),
}
L2_BYTES = 126e6
DUMP_BYTES = 64 << 20
CPU_THREADS = max(1, min(64, (os.cpu_count() or 2) // 2))       # fixed: the host's physical cores, at most 64


def train_args(w):
    return {'turn_based_training': w['turn_based'], 'observation': w['observation'], 'gamma': 0.8, 'lambda': 0.7,
            'burn_in_steps': w.get('burn_in', 0), 'forward_steps': w['T'] - w.get('burn_in', 0), 'entropy_regularization': 0.1,
            'entropy_regularization_decay': 0.1, 'policy_target': w['policy_target'], 'value_target': w['value_target'],
            'batch_size': w['B'], 'compress_steps': 4, 'maximum_episodes': 100000, 'minimum_episodes': 400, 'num_batchers': 1,
            'seed': 0}


def make_net(w):
    from handyrl_b200 import nets
    torch.manual_seed(0)
    return {'tictactoe': nets.tictactoe_net, 'geister': nets.geister_net, 'geese': nets.geese_net, 'wide': nets.WideActionNet}[w['net']]()


_EPISODES = {}


def episodes_for(w, n=2000):
    from handyrl_b200.synthetic import tictactoe_episodes
    if n not in _EPISODES:
        _EPISODES[n] = tictactoe_episodes(n, seed=123)
    return _EPISODES[n]


def make_batch(w, seed):
    """One replay batch of the workload at its FULL batch size."""
    from handyrl_b200 import synthetic
    if w.get('episodes'):           # windows drawn from real episodes by the host batcher (reference sampling law)
        import random
        from collections import deque
        from handyrl_b200.train import Batcher
        random.seed(seed)
        return Batcher(train_args(w), deque(episodes_for(w)))._make()
    if w['net'] == 'geister':
        return synthetic.synthetic_geister_batch(w['B'], w['T'], w['P'], w['A'], turn_based=w['turn_based'], observation=w['observation'],
                                                 burn_in=w.get('burn_in', 0), seed=seed)
    if w['net'] == 'geese':
        return synthetic.synthetic_geese_batch(w['B'], w['T'], w['P'], w['A'], seed=seed)
    return synthetic.synthetic_batch(w['B'], w['T'], w['P'], w['A'], turn_based=w['turn_based'], observation=w['observation'],
                                     reward_kind=w['reward_kind'], seed=seed, obs_shape=w['obs_shape'])


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU while the timed region runs (NVML, the
    same source nvidia-smi reads)."""

    def __init__(self, index, period=0.05):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.stop_flag = threading.Event()
        self.sm_max = None
        self.th = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
                getattr(nv, 'nvmlClocksThrottleReasonHwSlowdown', 0x8): 'hw_slowdown',
                getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
                getattr(nv, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
                getattr(nv, 'nvmlClocksThrottleReasonHwPowerBrakeSlowdown', 0x80): 'hw_power_brake',
            }
            get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                getattr(nv, 'nvmlDeviceGetCurrentClocksThrottleReasons')
            while not self.stop_flag.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get_reasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # noqa: BLE001
            self.reasons.add('sampler_error:%s' % type(e).__name__)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *exc):
        self.stop_flag.set()
        self.th.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.sm_max, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def physical_device_index(local):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------ CPU arm

def run_cpu_port(w, steps, warmup, threads, loss_only_too=True):
    """The eager-PyTorch CPU port of the reference learner step on the workload's FULL batch (never a smaller one):
    per-step wall times of `steps` steps after `warmup` untimed ones, plus the loss-only part (mask epilogue +
    compute_loss + autograd through it, net outputs given) timed the same way."""
    from oracle.torch_learner import CpuLearner, loss_from_raw
    torch.set_num_threads(threads)
    args = train_args(w)
    lrn = CpuLearner(make_net(w), args, lr=3e-8 * w['B'] * w['T'])
    batches = [make_batch(w, 2000 + i) for i in range(4)]
    for i in range(warmup):
        lrn.step(batches[i % 4])
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        lrn.step(batches[i % 4])
        times.append(time.perf_counter() - t0)
    out = {'ms_mean': 1e3 * sum(times) / len(times), 'ms_min': 1e3 * min(times), 'ms_median': 1e3 * statistics.median(times),
           'value': w['B'] * w['T'] * len(times) / sum(times), 'cores': torch.get_num_threads(), 'steps': steps, 'warmup': warmup,
           'total_s': sum(times)}
    if loss_only_too:
        from handyrl_b200.synthetic import synthetic_outputs
        b = batches[0]
        has_ret = w['net'] == 'geister'
        lt = []
        for i in range(warmup + steps):
            raw = {k: v.requires_grad_(True) for k, v in synthetic_outputs(b, has_return=has_ret, seed=i).items()}
            t0 = time.perf_counter()
            losses, _ = loss_from_raw(raw, b, args)
            losses['total'].backward()
            if i >= warmup:
                lt.append(time.perf_counter() - t0)
        out['loss_only'] = {'ms_min': 1e3 * min(lt), 'ms_median': 1e3 * statistics.median(lt), 'ms_mean': 1e3 * sum(lt) / len(lt)}
    return out


def cpu_baseline_block(w, r, kind_note=''):
    return {'value': r['value'], 'unit': 'samples/s', 'cores': r['cores'], 'kind': 'port',
            'sample': '%d timed steps (after %d warm-ups) of the FULL B=%d x T=%d batch, eager-PyTorch CPU port of the reference '
                      'step (oracle/torch_learner.py)%s' % (r['steps'], r['warmup'], w['B'], w['T'], kind_note),
            'ms_per_step': {'min': r['ms_min'], 'median': r['ms_median'], 'mean': r['ms_mean']},
            'loss_only_ms': r.get('loss_only'), 'host_cores': os.cpu_count()}


def reference_arm(opt, w):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return      # the host has one set of cores: rank 0 alone measures it
    steps, warmup = max(1, opt.steps), max(3, opt.warmup)
    # a probe step decides only whether the run fits the time box; the batch is never shrunk
    probe = run_cpu_port(w, 1, 1, CPU_THREADS, loss_only_too=False)
    est = probe['ms_mean'] * 1e-3 * (steps + warmup) * 1.3
    if est > opt.cpu_budget_s:
        fit = int(opt.cpu_budget_s / (probe['ms_mean'] * 1e-3 * 1.3)) - warmup
        if fit < 3:
            print(json.dumps({'impl': 'reference', 'unavailable': 'one CPU step of %s takes %.1f s: %d+%d steps do not fit %d s'
                              % (opt.workload, probe['ms_mean'] * 1e-3, steps, warmup, opt.cpu_budget_s)}), flush=True)
            return
        steps = fit
    r = run_cpu_port(w, steps, warmup, CPU_THREADS)
    line = {
        'impl': 'reference', 'metric': 'learner_samples_per_sec', 'value': r['value'], 'unit': 'samples/s',
        'n_gpus': opt.gpus, 'steps': steps, 'warmup': warmup, 'ms_per_step': r['ms_mean'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
        'config': {'workload': w['desc'], 'global_batch': w['B'], 'seq_len': w['T'], 'parallelism': 'cpu', 'threads': r['cores']},
        'cpu_baseline': cpu_baseline_block(w, r),
        'e2e': {'value': r['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ B200 arm

def dump_outputs(path, stepper):
    """The last step's loss sums (p, v, r, ent, total, dcnt) as losses.npy and every entry of the model's state_dict
    after it as state.<key>.npy; float32 stays float32, everything else is written as float64."""
    import numpy as np
    stepper.stream.synchronize()
    arrays = {'losses': stepper.last_losses.cpu()}
    arrays.update(('state.' + k, v) for k, v in stepper.cpu_state_dict().items())
    arrays = {k: (t if t.dtype == torch.float32 else t.double()).numpy() for k, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit('bench.py: --dump-outputs would write %d bytes (limit %d)' % (total, DUMP_BYTES))
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + '.npy'), a)


def loss_kernel_name(A):
    """Which variant hrl_loss_fwd_bwd dispatches to for this action count (csrc/loss_kernel.cu)."""
    return 'hrl::loss_group_kernel' if A <= 32 else ('hrl::loss_bulk_kernel' if (A > 256 and A % 4 == 0) else 'hrl::loss_rows_kernel')


def time_loss_alone(B, T, P, A, turn_based, observation, args, device, reps, bf16=False):
    """Average device time (ms) of hrl_loss_fwd_bwd launched back to back over input sets that together exceed L2."""
    from handyrl_b200 import ops
    from handyrl_b200.synthetic import synthetic_batch, synthetic_outputs, bytes_per_cell
    Pa = 1 if (turn_based and not observation) else P
    per_set = (bytes_per_cell(P, Pa, A, T, 0) - (4 * Pa * A if bf16 else 0)) * B * T     # bf16 logits + gradients: 8 not 12 bytes / action
    n = max(2, min(64, int(2 * L2_BYTES / per_set) + 1))
    sets = []
    for i in range(n):
        b = synthetic_batch(B, T, P, A, turn_based=turn_based, observation=observation, seed=300 + i, with_obs=False)
        o = synthetic_outputs(b, seed=400 + i)
        o = {k: v.to(device) for k, v in o.items()}
        if bf16:
            o['policy'] = o['policy'].to(torch.bfloat16)
        sets.append((o, {k: v.to(device) for k, v in b.items()},
                     ops.LossBuffers(B, T, P, Pa, A, True, False, device, policy_dtype=o['policy'].dtype)))
    for o, b, buf in sets:
        ops.loss_fwd_bwd(o, b, args, buffers=buf)
    torch.cuda.synchronize()
    # one launch per input set captured in a CUDA graph: no host launch overhead between kernels
    side = torch.cuda.Stream(device=device)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            for o, b, buf in sets:
                ops.loss_fwd_bwd(o, b, args, buffers=buf)
        rounds = max(1, reps // n)
        graph.replay()
        side.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for _ in range(rounds):
            graph.replay()
        e1.record(side)
        side.synchronize()
    return {'ms': e0.elapsed_time(e1) / (rounds * n), 'bytes': per_set, 'sets': n}


def time_tower_products(engine, device):
    """The three tcgen05 3xTF32 products of one layer of the fused tower engine (handyrl_b200/tower.py), each alone: 20 launches
    captured in a CUDA graph, replayed 5 times.  flops = 2 M N K of the fp32 product the kernel computes (the hardware executes three
    TF32 instructions per product at half the bf16 rate, i.e. a ceiling of 1/6 of the bf16 peak)."""
    M, D = engine.M, engine.D
    f = dict(dtype=torch.float32, device=device)
    X, Y, out = torch.randn(M, D, **f), torch.randn(M, D, **f), torch.empty(M, D, **f)
    c = [torch.rand(D, **f) for _ in range(5)]
    sp = engine.splits['tower']
    ws = engine.ws
    cases = {
        'forward (A = relu(bn(y)) on the fly, packed weights, BN-statistics epilogue)':
            lambda: engine._gemm(dict(t=X, consts=(c[0], c[1]), relu=True), dict(t=engine.Wf[0], packed=True), out, K=D, N=D, epilogue='stats'),
        'input gradient (A = BN backward of two sources on the fly, ReLU-mask + BN-sums epilogue)':
            lambda: engine._gemm(dict(t=X, t2=Y, consts=(c[0], c[1], c[2])), dict(t=engine.Wb[0], packed=True), out, K=D, N=D,
                                 epilogue='mask_stats', ep=dict(y=Y, scale=c[0], shift=c[1], mean=c[2], rstd=c[3])),
        'weight gradient (both operands transformed, %d K slices)' % sp:
            lambda: engine._gemm(dict(t=X, t2=Y, consts=(c[0], c[1], c[2]), kmajor=False, by_row=True),
                                 dict(t=Y, consts=(c[3], c[4]), relu=True, kmajor=False, by_row=True), None, K=M, N=D, M=D, splits=sp,
                                 partial=True, ws=ws),
    }
    res = {}
    side = torch.cuda.Stream(device=device)
    for name, fn in cases.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for _ in range(20):
                    fn()
            graph.replay()
            side.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(side)
            for _ in range(5):
                graph.replay()
            e1.record(side)
            side.synchronize()
        us = e0.elapsed_time(e1) / 100 * 1e3
        res[name] = {'kernel_us': us, 'flops': 2.0 * M * D * D, 'achieved': 2.0 * M * D * D / (us * 1e-6) / 1e12}
    return res


def time_gather_alone(w, device, reps=20):
    """The replay gather/pad kernel (K2) alone: episodes of the workload's shape resident in the device ring, B windows per
    launch into distinct output batches that together exceed L2.  Algorithmic bytes = batch bytes written + stored rows read
    (batch bytes x live fraction)."""
    import numpy as np
    from handyrl_b200.batch import FlatEpisode
    from handyrl_b200.replay import DeviceReplay
    g = np.random.default_rng(0)
    B, T, P, A = w['B'], w['T'], w['P'], w['A']
    args = train_args(w)
    obs_elems = int(np.prod(w['obs_shape']))
    steps = 3 * T
    n_eps = max(8, min(64, int(1.5e9 / (steps * P * (obs_elems + A) * 4))))
    rp = DeviceReplay(capacity_steps=n_eps * steps + 1, max_episodes=n_eps + 1, device=device)
    fes = []
    for _ in range(n_eps):
        fe = FlatEpisode()
        fe.steps, fe.players = steps, list(range(P))
        fe.obs = (g.random((steps, P) + tuple(w['obs_shape'])) < 0.3).astype(np.float32)
        fe.prob = g.random((steps, P), dtype=np.float32)
        fe.action = g.integers(0, A, (steps, P)).astype(np.int32)
        fe.amask = np.where(g.random((steps, P, A)) < 0.7, 0, 1e32).astype(np.float32)
        fe.value = g.random((steps, P, 1), dtype=np.float32)
        fe.reward = np.zeros((steps, P), np.float32)
        fe.ret = np.zeros((steps, P), np.float32)
        fe.flags = np.full((steps, P), 3, np.uint8)
        fe.turn = (np.arange(steps) % P).astype(np.int32)
        fe.outcome = np.zeros(P, np.float32)
        fes.append(fe)
    rp.add_flat_many(fes)
    probe = rp.empty_batch(B, args)
    batch_bytes = sum(t.numel() * t.element_size() for t in probe.values())
    n_out = max(2, min(16, int(2 * L2_BYTES / batch_bytes) + 1))
    outs = [probe] + [rp.empty_batch(B, args) for _ in range(n_out - 1)]
    wins = [rp.sample_windows(B, args, g) for _ in range(n_out)]
    wdev = [torch.from_numpy(x.view(np.uint8).reshape(B, -1)).to(device) for x in wins]
    live = float(np.mean([(x['end'] - x['start']).sum() / (B * T) for x in wins]))
    for wd, out in zip(wdev, outs):
        rp.gather(wd, args, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for wd, out in zip(wdev, outs):
            rp.gather(wd, args, out=out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (reps * n_out)
    return {'ms': ms, 'bytes': batch_bytes * (1 + live), 'batch_bytes': batch_bytes, 'live': live, 'outputs': n_out}


def trainer_leg(w, steps, warm_steps=100):
    """samples/s through the drop-in Trainer: episodes (reference wire format) -> feeder thread decode + upload -> window
    sampling -> gather/pad kernel -> learner step, with epoch hand-offs (update()) going on, over >= `steps` steps."""
    from handyrl_b200.train import Trainer
    from handyrl_b200.synthetic import tictactoe_episodes
    args = dict(train_args(w), minimum_episodes=2000, maximum_episodes=20000, gpu_replay=True, num_gpus=1, forward_steps=w['T'])
    tr = Trainer(args, make_net(w))
    tr.episodes.extend(tictactoe_episodes(4000, seed=7))
    stop = threading.Event()

    def learner_side():          # what Learner.feed_episodes / Learner.update do while the trainer runs
        fresh = tictactoe_episodes(2000, seed=8)
        i = 0
        while not stop.is_set():
            tr.episodes.extend(fresh[i % 2000:i % 2000 + 20])
            i += 20
            while len(tr.episodes) > args['maximum_episodes']:
                tr.episodes.popleft()
            time.sleep(0.01)

    th = threading.Thread(target=tr.run, daemon=True)
    th.start()
    tr.update()                                    # first epoch: builds + captures the step
    feeder = threading.Thread(target=learner_side, daemon=True)
    feeder.start()
    while tr.steps < warm_steps:
        time.sleep(0.001)
    tr.stepper.stream.synchronize()
    s0, t0 = tr.steps, time.perf_counter()
    handoffs = 0
    while tr.steps - s0 < steps:
        time.sleep(0.05)
        if handoffs < 3 and tr.steps - s0 > (handoffs + 1) * steps // 4:
            tr.update()                            # an epoch hand-off in the middle of the timed region
            handoffs += 1
    tr.stepper.stream.synchronize()
    dt, n = time.perf_counter() - t0, tr.steps - s0
    stop.set()
    feeder.join(timeout=5)
    fed = tr.gpu_batcher.fed
    tr.stop()
    th.join(timeout=20)
    return {'value': w['B'] * w['T'] * n / dt, 'unit': 'samples/s', 'ms_per_step': 1e3 * dt / n, 'steps': n, 'epoch_handoffs': handoffs,
            'episodes_uploaded': fed, 'timing': 'host wall clock around the steps, stream synchronised on both sides',
            'path': 'Trainer.run: EpisodeDeque -> GpuBatcher (feeder thread, vectorised window sampling, hrl_gather_pad) -> LearnerStep'}


def b200_arm(opt, w):
    import torch.distributed as dist
    from handyrl_b200 import multigpu, ops
    from handyrl_b200.synthetic import bytes_per_cell
    from handyrl_b200.train import LearnerStep, PackedBatch

    rank, world, local = multigpu.init_from_env('nccl')
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    pinned_cpus = multigpu.pin_to_gpu_numa(local) if world > 1 else None
    pg = dist.group.WORLD if world > 1 else None

    args = train_args(w)
    B, T, P, A = w['B'], w['T'], w['P'], w['A']
    example = make_batch(w, 10_000 + rank)
    stepper = LearnerStep(make_net(w), args, example, lr=3e-8 * B * T * world, device=device, process_group=pg,
                          use_graph=True, time_loss_kernel=True)
    nbytes = stepper.layout.nbytes
    R = max(8, int(2 * L2_BYTES / nbytes) + 1)
    R = min(R, 96)
    host_ring = [PackedBatch(stepper.layout).fill(make_batch(w, 20_000 + rank * 1000 + i)) for i in range(R)]
    dev_ring = torch.empty((R, nbytes), dtype=torch.uint8, device=device)
    for i, pk in enumerate(host_ring):
        dev_ring[i].copy_(pk.buffer)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n_warm, n_steps):
        for i in range(n_warm):
            fn(i)
        stepper.loss_kernel_ms()            # drop warm-up kernel timings
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        with torch.cuda.stream(stepper.stream):
            e0.record()
        for i in range(n_steps):
            fn(n_warm + i)
        t_launched = time.perf_counter() - t0
        with torch.cuda.stream(stepper.stream):
            e1.record()
        barrier()
        wall = time.perf_counter() - t0
        mine = e0.elapsed_time(e1)
        ms, per_rank = mine, None
        if world > 1:
            t = torch.tensor([mine, wall * 1e3, t_launched * 1e3], device=device)
            allt = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            ms = max(float(x[0]) for x in allt)
            per_rank = [{'device_ms': float(x[0]), 'wall_ms': float(x[1]), 'host_launch_ms': float(x[2])} for x in allt]
        return ms, wall, per_rank

    warm = max(3, opt.warmup)
    # ---- value: inputs resident in HBM
    with ClockSampler(physical_device_index(local)) as clocks:
        ms, wall, per_rank_value = timed(lambda i: stepper.step_resident(dev_ring[i % R]), warm, opt.steps)
    kernel_ms, n_k = stepper.loss_kernel_ms()
    value = B * T * world * opt.steps / (ms * 1e-3)
    if opt.dump_outputs and rank == 0:
        dump_outputs(opt.dump_outputs, stepper)

    # ---- e2e: host batches, H2D inside (copy stream, one step ahead), loss read back every step (lagged by one step)
    pending = []

    def e2e_step(i):
        stepper.step(host_ring[i % R])
        pending.append(stepper.fetch_losses_async())
        if len(pending) > 1:
            pending.pop(0)()

    ms_e2e, wall_e2e, per_rank_e2e = timed(e2e_step, warm, opt.steps)
    last = pending.pop()()
    stepper.loss_kernel_ms()
    e2e_value = B * T * world * opt.steps / (ms_e2e * 1e-3)

    # ---- every rank must hold the same weights (identical clip + Adam on the all-reduced bucket)
    ranks_identical = None
    if world > 1:
        if stepper.peer is not None:
            stepper.peer.check()
        flat = stepper.state.flat_param
        digest = torch.stack([flat.double().sum(), (flat.double() * torch.arange(flat.numel(), device=device, dtype=torch.float64)).sum()])
        alld = [torch.empty_like(digest) for _ in range(world)]
        dist.all_gather(alld, digest)
        ranks_identical = all(torch.equal(d, alld[0]) for d in alld)
        assert ranks_identical, 'ranks hold different weights after %d steps: %s' % (stepper.steps, [d.tolist() for d in alld])

    # ---- the loss kernel alone on cold inputs (distinct input sets larger than L2), at the bench shape and at the
    #      wide-row shape of configs[4]'s per-GPU shard (where an HBM roofline is physically meaningful); K2 alone
    alone, wide, wide16, k2, gemm = None, None, None, None, None
    if rank == 0 and not opt.quick:
        alone = time_loss_alone(B, T, P, A, w['turn_based'], w['observation'], args, device, reps=200)
        if stepper.engine is not None:
            gemm = time_tower_products(stepper.engine, device)
        if not opt.no_wide:
            ww = WORKLOADS['cfg5shard']
            wide = time_loss_alone(ww['B'], ww['T'], ww['P'], ww['A'], ww['turn_based'], ww['observation'], train_args(ww),
                                   device, reps=40)
            wide16 = time_loss_alone(ww['B'], ww['T'], ww['P'], ww['A'], ww['turn_based'], ww['observation'], train_args(ww),
                                     device, reps=40, bf16=True)
            k2 = {'cfg5shard': time_gather_alone(ww, device, reps=5)}
            if w['obs_shape'] is not None and opt.workload != 'cfg5shard':
                k2[opt.workload] = time_gather_alone(w, device, reps=20)

    launches_per_step = stepper.launches_per_step
    if rank != 0:
        shutdown(stepper, world)
        return

    peak, peak_src = measured_peak()
    Pa = example['action_mask'].shape[2]
    alg_bytes = bytes_per_cell(P, Pa, A, T, 1 if w['net'] == 'geister' else 0) * B * (T - w.get('burn_in', 0))
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_all = None, None
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            traffic_all = json.load(f)
            traffic = traffic_all.get(opt.workload)
    except Exception:
        pass
    line = {
        'metric': 'learner_samples_per_sec', 'value': value, 'unit': 'samples/s', 'n_gpus': world, 'steps': opt.steps,
        'warmup': warm, 'ms_per_step': ms / opt.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
        'config': {'workload': w['desc'], 'global_batch': B * world, 'seq_len': T, 'parallelism': 'dp%d' % world,
                   'tf32': 'single-pass TF32 disabled; the small-board dense layers run 3xTF32 (hi/lo split, fp32 accumulate) on tcgen05',
                   'cuda_graph': True,
                   'l2': 'inputs rotate over a ring of %d distinct resident batches (%.0f MB > 126 MB L2)' % (R, R * nbytes / 1e6),
                   'batchnorm': 'per-shard statistics (as the reference DataParallel)'},
        'clocks': clocks.summary(),
        'e2e': {'value': e2e_value, 'unit': 'samples/s', 'ms_per_step': ms_e2e / opt.steps,
                'h2d_bytes_per_step': nbytes * world, 'd2h_bytes_per_step': 24 * world,
                'wall_s': wall_e2e, 'last_losses': last},
        # this library's kernels per step, counted by the Python wrappers while the step was captured (ops.LAUNCHES)
        'gpu_launches': launches_per_step * opt.steps,
        'gpu_launches_per_step': launches_per_step,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'kernel': loss_kernel_name(A) + ' (hrl_loss_fwd_bwd)', 'kernel_us': kernel_ms * 1e3,
                     'launches_timed': n_k, 'algorithmic_bytes': alg_bytes, 'peak_source': peak_src,
                     'alone_cold_us': None if alone is None else alone['ms'] * 1e3,
                     'alone_cold_gbs': None if alone is None else alg_bytes / (alone['ms'] * 1e-3) / 1e9,
                     'note': 'event-bracketed single launch inside the step (events + the graph boundary around it add ~10 us to a '
                             'launch of this size, see DESIGN.md section 4); %.2f MB per launch = %.2f us at peak%s'
                             % (alg_bytes / 1e6, alg_bytes / peak / 1e3,
                                ' (latency-bound: below one DRAM round trip + launch)' if alg_bytes < 2e7 else '')},
        'wall_s': wall,
    }
    if world > 1:
        line['ranks_identical'] = ranks_identical
        line['per_rank'] = {'value': per_rank_value, 'e2e': per_rank_e2e, 'numa_pinned_cpus': None if pinned_cpus is None else len(pinned_cpus)}
    if wide is not None:
        gbs = wide['bytes'] / (wide['ms'] * 1e-3) / 1e9
        line['roofline_wide_rows'] = {
            'workload': WORKLOADS['cfg5shard']['desc'] + ' (loss kernel alone, %d cold input sets)' % wide['sets'],
            'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s', 'frac': gbs / peak,
            'kernel': loss_kernel_name(WORKLOADS['cfg5shard']['A']) + ' (hrl_loss_fwd_bwd)', 'kernel_us': wide['ms'] * 1e3,
            'algorithmic_bytes': wide['bytes'], 'traffic': None if traffic_all is None else traffic_all.get('cfg5shard')}
    if wide16 is not None:
        gbs = wide16['bytes'] / (wide16['ms'] * 1e-3) / 1e9
        line['roofline_wide_rows_bf16'] = {
            'workload': 'the same shape with HrlLossArgs.io_bf16: logits read and policy gradient written as bf16 (8 instead of 12 bytes '
                        'per action), all arithmetic fp32 (tests/test_loss_gpu.py: losses bit-identical to the fp32 pass)',
            'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s', 'frac': gbs / peak, 'kernel_us': wide16['ms'] * 1e3,
            'algorithmic_bytes': wide16['bytes'], 'speedup_vs_fp32_io': None if wide is None else wide['ms'] / wide16['ms']}
    if gemm is not None:
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                tpeak, tsrc = float(json.load(f)['bf16_tflops']), 'measured (MEASURED_PEAKS.json bf16_tflops, burst)'
        except Exception:
            tpeak, tsrc = 2250.0, 'fallback (nominal dense bf16)'
        line['roofline_net_gemm'] = {
            'kernel': 'hrl::gemm_tf32x3_kernel (hrl_gemm_fused): the net of this workload, 14 launches / ~75% of the step', 'bound': 'tensor',
            'unit': 'TFLOP/s', 'peak': tpeak, 'peak_source': tsrc,
            'note': 'M x 288 x 288 products of one tower layer, alone; fp32-class accuracy = 3 TF32 tensor instructions per product at half '
                    'the bf16 rate: ceiling peak/6; a single 128-row tile per CTA (prologue/epilogue not overlapped)',
            'products': {k: dict(v, frac=v['achieved'] / tpeak, frac_of_3xtf32_ceiling=v['achieved'] / (tpeak / 6)) for k, v in gemm.items()}}
    if k2:
        line['roofline_k2'] = {
            name: {'bound': 'hbm', 'kernel': 'hrl::gather_pad_kernel (hrl_gather_pad)', 'achieved': r['bytes'] / (r['ms'] * 1e-3) / 1e9,
                   'peak': peak, 'unit': 'GB/s', 'frac': r['bytes'] / (r['ms'] * 1e-3) / 1e9 / peak, 'kernel_us': r['ms'] * 1e3,
                   'algorithmic_bytes': r['bytes'], 'batch_bytes': r['batch_bytes'], 'live_fraction': r['live'],
                   'traffic': None if traffic_all is None else traffic_all.get('k2_' + name),
                   'note': 'alone, back to back into %d output batches (> L2); algorithmic = batch bytes written + live rows read' % r['outputs']}
            for name, r in k2.items()}
    if world == 1 and not opt.no_trainer and not opt.quick and w['net'] == 'tictactoe':
        try:
            import contextlib
            with contextlib.redirect_stdout(sys.stderr):        # the Trainer prints the reference's progress lines
                line['e2e_trainer'] = trainer_leg(w, steps=opt.steps)
        except Exception as e:  # noqa: BLE001
            line['e2e_trainer'] = {'error': '%s: %s' % (type(e).__name__, e)}
    if world == 1 and not opt.no_cpu and not opt.quick:
        probe = run_cpu_port(w, 1, 1, CPU_THREADS, loss_only_too=False)
        n = max(3, min(20, int(25.0 / (probe['ms_mean'] * 1e-3)) - 3))
        r = run_cpu_port(w, steps=n, warmup=3, threads=CPU_THREADS)
        line['cpu_baseline'] = cpu_baseline_block(w, r)
        if probe['ms_mean'] < 4000:
            r1 = run_cpu_port(w, steps=3, warmup=1, threads=1, loss_only_too=False)
            line['cpu_baseline']['as_shipped_1_thread'] = {'value': r1['value'], 'ms_median': r1['ms_median']}
    print(json.dumps(line), flush=True)
    shutdown(stepper, world)


def shutdown(stepper, world):
    """Tear down NCCL after the captured graphs are gone; never let a teardown hang eat the run."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush()
    killer = threading.Timer(20.0, lambda: os._exit(0))
    killer.daemon = True
    killer.start()
    stepper.close()
    dist.barrier()
    torch.cuda.synchronize()
    dist.destroy_process_group()
    killer.cancel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=1000)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-wide', action='store_true', help='skip the wide-row loss-kernel and gather-kernel measurements')
    ap.add_argument('--no-trainer', action='store_true', help='skip the Trainer (e2e_trainer) leg')
    ap.add_argument('--quick', action='store_true', help='value and e2e only')
    ap.add_argument('--cpu-budget-s', type=int, default=240, help='time box of --impl reference (steps are dropped, never the batch)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed step\'s loss sums and model state to DIR/<name>.npy')
    opt = ap.parse_args()
    if opt.steps < 1:
        ap.error('--steps must be at least 1')
    if opt.dump_outputs and opt.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    w = WORKLOADS[opt.workload]
    if opt.impl == 'reference':
        reference_arm(opt, w)
    else:
        if not torch.cuda.is_available():
            raise SystemExit('bench.py: no CUDA device; the learner hot path has no CPU fallback '
                             '(use --impl reference for the CPU port)')
        b200_arm(opt, w)


if __name__ == '__main__':
    main()
