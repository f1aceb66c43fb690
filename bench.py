#!/usr/bin/env python
""" bench.py — collocation points/sec of the pydens fit step on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port), rank 0
    python bench.py ... --dump-outputs DIR                    # also write the timed path's last-step outputs as .npy

A "step" is one optimizer step of `Solver.fit` on one batch: fused kernel (sample/read points, forward
jets, residual, MSE, backward) + all-reduce (N>1) + Adam + loss record.  Workload = BASELINE.json
configs[1]: 2-D Poisson, 4-layer [10,12,15,1] tanh MLP, batch 100 000 per GPU (weak scaling).

Numbers in the JSON line:
  value      points/s, device-timed (CUDA events, max over ranks) over EXACTLY K steps replayed from a
             CUDA graph; every step reads its own batch from an HBM-resident pool of distinct batches
             (pool > L2 when K >= 160), so no step sees its input warm in L2.
  e2e        the same metric through the public call `Solver.fit(niters=K, batch_size=B, sampler=...)`
             with HOST batches: per step one H2D copy of the batch from pinned memory and one D2H read of
             the loss, all inside the timed region.
  roofline   the fused kernel alone (CUDA events around K back-to-back launches): algorithmic bytes
             (4*total B/point) over time against the measured HBM peak — the path is FP32-FMA bound
             (SURVEY.md 8d), so `fp32` carries the meaningful fraction: algorithmic flops (6*C*M per
             point) over time against 148 SMs x 128 lanes x 2 flop x the measured SM clock.
  cpu_baseline  oracle/autograd_port.py (the reference algorithm on PyTorch-CPU autograd) timed on this
             box's host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

import numpy as np          # noqa: E402
import torch                # noqa: E402

METRIC = 'collocation points/sec (fit step)'
WORKLOADS = {
    # name: (problem in tests/problems.py, per-GPU batch, lr)
    'cfg2': ('poisson2d', 100000, 0.005),
    'cfg3': ('ode_param', 1000000, 0.01),
    'cfg4': ('heat2d', 1000000, 0.001),
    'cfg5': ('wave3d', 500000, 0.001),
}


def describe(workload, n_gpus):
    import problems as P
    name, batch, lr = WORKLOADS[workload]
    cfg = P.PROBLEMS[name]
    return {'workload': '%s: %s, MLP %s %s, batch_size=%d per GPU' % (
        workload, name, [cfg['ndims'] + cfg['nparams']] + cfg['features'], cfg['activation'], batch),
        'global_batch': batch * n_gpus, 'optimizer': 'Adam lr=%g' % lr, 'parallelism': 'dp%d' % n_gpus}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return None
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if (t0 is None or t >= t0 - 0.05) and (t1 is None or t <= t1 + 0.1)] \
            or [r for _, r in self.rows]
        if not rows:
            return None
        try:
            sm = sorted(float(r[0]) for r in rows)
            reasons = []
            for i, nm in enumerate(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')):
                if any(r[3 + i].lower().startswith('active') for r in rows):
                    reasons.append(nm)
            return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(rows[0][1]), 'reasons': reasons,
                    'samples': len(rows), 'power_w_max': max(float(r[2]) for r in rows)}
        except (ValueError, IndexError):
            return None


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port of the reference loop on host cores
# ------------------------------------------------------------------------------------------------
def cpu_reference(workload, n_gpus, steps, warmup, budget_s=None):
    import problems as P
    from oracle import autograd_port as ap
    name, batch, lr = WORKLOADS[workload]
    cfg = P.PROBLEMS[name]
    cores = os.cpu_count() or 1
    torch.manual_seed(0)
    prob = ap.Problem(lambda u, *xs, D, V: cfg['equation'](u, *xs, D=D, V=V), ndims=cfg['ndims'],
                      nparams=cfg['nparams'], initial_condition=cfg['ic'], boundary_condition=cfg['bc'],
                      domain=cfg['domain'], features=cfg['features'], activation=cfg['activation'],
                      variables=cfg.get('variables'))
    gbatch = batch * n_gpus
    # bound the sample so the run ends within minutes: cap points per step
    sample_batch = min(gbatch, 100000 if name != 'wave3d' else 20000)
    ranges = cfg['ranges']

    def stream(i):
        cols = [torch.rand((sample_batch, 1)) * (hi - lo) + lo for lo, hi in ranges]
        return torch.cat(cols, dim=1)
    # the reference leaves threading to PyTorch; on a many-core host the default (all cores) can be far
    # from the best setting for these small ops, so give the baseline its best thread count
    best, best_t = None, None
    for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(nt)
        ap.fit(prob, 1, sample_batch, lr=lr, point_stream=stream)
        t = time.perf_counter()
        ap.fit(prob, 2, sample_batch, lr=lr, point_stream=stream)
        t = time.perf_counter() - t
        if best_t is None or t < best_t:
            best, best_t = nt, t
    torch.set_num_threads(best)
    ap.fit(prob, warmup, sample_batch, lr=lr, point_stream=stream)
    t0 = time.perf_counter()
    done = 0
    chunk = max(1, min(steps, 5))
    while done < steps:
        n = min(chunk, steps - done)
        ap.fit(prob, n, sample_batch, lr=lr, point_stream=stream)
        done += n
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {'value': done * sample_batch / dt, 'unit': 'points/s', 'cores': best, 'kind': 'port',
            'sample': '%d steps of batch %d (of the global %d) through oracle/autograd_port.py (reference loop '
                      'on PyTorch-CPU autograd; %d threads = best of a sweep on this %d-core host)'
                      % (done, sample_batch, gbatch, best, cores),
            'ms_per_step': 1e3 * dt / done, 'steps': done}


# ------------------------------------------------------------------------------------------------
# our arm: device-timed steps of one workload
# ------------------------------------------------------------------------------------------------
def make_solver(workload, dev):
    import problems as P
    from pydens_b200 import Solver, D, V
    name, batch, lr = WORKLOADS[workload]
    cfg = P.PROBLEMS[name]
    torch.manual_seed(0)
    solver = Solver(P.bind(name, D, lambda n, init: V(n, data=torch.Tensor([init]))), ndims=cfg['ndims'],
                    nparams=cfg['nparams'], initial_condition=cfg['ic'], boundary_condition=cfg['bc'],
                    domain=cfg['domain'], layout=cfg['layout'], features=cfg['features'],
                    activation=cfg['activation'], device=dev, backend='fused', seed=123)
    return solver, cfg, lr


class Timed:
    """ One workload on this rank's shard: an HBM-resident pool of distinct batches, the step function, and
    device-timed runs of EXACTLY K steps (CUDA events, max over ranks), repeated `reps` times. """

    def __init__(self, workload, gbatch, dev, rank, world, K, W, pool_cap_bytes=2 << 30):
        import ctypes as C
        from pydens_b200 import _native
        from pydens_b200.engine import shard_batch
        import torch.distributed as dist
        self.dist, self.world, self.rank, self.dev, self.K, self.W = dist, world, rank, dev, K, W
        self.solver, self.cfg, self.lr = make_solver(workload, dev)
        self.eng = eng = self.solver._get_engine()
        self.info = eng.info
        self.total = self.cfg['ndims'] + self.cfg['nparams']
        self.gbatch = gbatch
        self.local_n, self.offset = shard_batch(gbatch, world, rank)
        self.inv_n = 1.0 / gbatch
        bytes_per_batch = self.local_n * self.total * 4
        # >= 160 distinct batches at cfg2 (the pool then exceeds the 126 MB L2); big batches are each > L2 already
        self.pool_n = int(max(2, min(max(K, 160), 256, pool_cap_bytes // max(bytes_per_batch, 1))))
        gen = torch.Generator(device=dev).manual_seed(1000 + rank)
        self.pool = torch.empty((self.pool_n, self.local_n, self.total), device=dev)
        for k, (lo, hi) in enumerate(self.cfg['ranges']):
            self.pool[:, :, k] = torch.rand((self.pool_n, self.local_n), generator=gen, device=dev) * (hi - lo) + lo
        self.solver._make_optimizer('Adam', self.lr, fused_hint=True)
        self.opt = self.solver.optimizer
        self.ring = torch.zeros(4096, device=dev)
        self._C, self._native = C, _native
        # the engine's default step: optimizer.step() and the loss log in the tail of the step kernel (pinn_step_adam)
        self.fused_adam = os.environ.get('PYDENS_B200_FUSED_ADAM', '1') != '0' and (world == 1 or eng.comm is not None)
        self.adam = None
        if self.fused_adam:
            g0 = self.opt.param_groups[0]
            mask = eng._bind_adam_state(self.opt)
            m, v, steps, _ = eng._adam_flat
            self.adam = _native.PinnAdam(m.data_ptr(), v.data_ptr(), mask.data_ptr(), steps.data_ptr(), steps.numel(),
                                         float(g0['lr']), float(g0['betas'][0]), float(g0['betas'][1]), float(g0['eps']),
                                         float(g0['weight_decay']), self.ring.data_ptr(), self.ring.numel())

    def step(self, pts):
        C, eng = self._C, self.eng
        if self.fused_adam:
            eng._step_adam(pts, None, self.local_n, self.inv_n, self.offset, self.adam, allreduce=self.world > 1)
            return
        eng._step(pts, None, self.local_n, self.inv_n, self.offset, allreduce=self.world > 1)
        if self.world > 1 and eng.comm is None:
            self.dist.all_reduce(eng.out)
        self.opt.step()
        self._native.check(eng.lib.pinn_record_loss(eng.plan, C.c_void_p(eng.out.data_ptr()), C.c_void_p(self.ring.data_ptr()),
                                                    C.c_int64(self.ring.numel()), C.c_void_p(eng.step_counter.data_ptr()),
                                                    eng._stream()))

    def run(self, reps=10, sampled=False):
        """ -> (list of ms for K steps, one per repetition; graphed?) """
        K, dist, world, dev = self.K, self.dist, self.world, self.dev
        for i in range(self.W):
            self.step(None if sampled else self.pool[i % self.pool_n])
        torch.cuda.synchronize()
        graph, graphed = torch.cuda.CUDAGraph(), True
        try:
            with torch.cuda.graph(graph):
                for i in range(K):
                    self.step(None if sampled else self.pool[i % self.pool_n])
        except Exception as exc:            # noqa: BLE001
            graphed = False
            torch.cuda.synchronize()
            sys.stderr.write('graph capture failed (%s): timing plain launches\n' % exc)
        if graphed:
            graph.replay()                  # one untimed replay (uploads the graph)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(reps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0.record()
            if graphed:
                graph.replay()
            else:
                for i in range(K):
                    self.step(None if sampled else self.pool[i % self.pool_n])
            e1.record()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            times.append(float(ms.item()))
        del graph
        return times, graphed

    def kernel_ms(self, reps=5):
        """ the fused kernel alone: CUDA events around K back-to-back launches on the launching stream """
        eng, K = self.eng, self.K
        if self.fused_adam and self.world == 1:         # the launch of the timed region: Adam + loss log in its tail
            def launch(pts):
                eng._step_adam(pts, None, self.local_n, self.inv_n, self.offset, self.adam)
        else:
            def launch(pts):
                eng._step(pts, None, self.local_n, self.inv_n, self.offset)
        for i in range(3):
            launch(self.pool[i % self.pool_n])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = []
        for _ in range(reps):
            e0.record()
            for i in range(K):
                launch(self.pool[i % self.pool_n])
            e1.record()
            torch.cuda.synchronize()
            best.append(e0.elapsed_time(e1) / K)
        return sorted(best)[len(best) // 2]

    def allreduce_check(self):
        """ one step through the in-kernel peer all-reduce and through pinn_step + NCCL all_reduce on the same batch """
        eng, dist = self.eng, self.dist
        if self.world <= 1 or eng.comm is None:
            return None
        pts = self.pool[0]
        eng._step(pts, None, self.local_n, self.inv_n, self.offset, allreduce=True)
        torch.cuda.synchronize()
        fused = eng.out.clone()
        eng._step(pts, None, self.local_n, self.inv_n, self.offset, allreduce=False)
        dist.all_reduce(eng.out)
        torch.cuda.synchronize()
        ref = eng.out.clone()
        num = (fused - ref).abs().max()
        den = ref.abs().max().clamp_min(1e-30)
        d = (num / den).reshape(1)
        dist.all_reduce(d, op=dist.ReduceOp.MAX)
        return {'max_rel_diff': float(d.item()), 'vector_floats': int(fused.numel()),
                'paths': 'pinn_step_allreduce (NVLink peer memory, in-kernel) vs pinn_step + NCCL all_reduce'}


def dump_outputs(t, outdir):
    """ What the timed path hands its caller after its last step, as DIR/<name>.npy (float32): the updated flat
    parameters, the gradient that step applied and its loss.  Inputs are seeded, so two builds run with the same
    arguments can be compared output for output. """
    eng = t.eng
    torch.cuda.synchronize()
    os.makedirs(outdir, exist_ok=True)
    for name, v in (('params', eng.flat), ('grads', eng.out[:eng.n_params]),
                    ('loss', eng.out[eng.n_params:eng.n_params + 1])):
        np.save(os.path.join(outdir, name + '.npy'), v.detach().cpu().numpy().astype(np.float32))


def roofline_blocks(t, kern_ms, step_ms, clk, peaks, workload):
    """ roofline of the fused kernel: the binding roof (FP32 FMA for the thread kernel, tensor cores for the tile
    kernel) first, the HBM fraction BASELINE.json asks for beside it. """
    info = t.info
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if 'hbm_gbs' in peaks else 'fallback (B200_PROFILING.md)'
    flops = info.flops_per_point * t.local_n
    byts = info.bytes_per_point * t.local_n
    ach_tf = flops / (kern_ms * 1e-3) / 1e12
    ach_gbs = byts / (kern_ms * 1e-3) / 1e9
    sm_mhz = (clk or {}).get('sm_mhz') or float(peaks.get('sm_max_mhz', 1965.0))
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get(workload)
    except (OSError, ValueError):
        pass
    if info.tensor_core:
        bf16 = float(peaks.get('bf16_tflops_sustained', peaks.get('bf16_tflops', 1590.0)))
        peak = bf16 / 2.0
        roof = {'bound': 'tensor', 'achieved': ach_tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach_tf / peak,
                'traffic': traffic, 'kernel': 'wide_step_kernel (tcgen05 kind::tf32, 3xTF32)', 'kernel_ms': kern_ms,
                'share_of_step': kern_ms / step_ms, 'flops_per_point': int(info.flops_per_point),
                'peak_source': 'dense TF32 = measured cuBLAS bf16 (sustained) / 2, ' + peak_src,
                'note': 'achieved counts the ALGORITHMIC 6*C*M flops per point once; the tensor cores execute 3x that '
                        '(3xTF32 split for fp32-grade results), so the pipe utilisation is ~3x frac'}
    else:
        peak = info.sm_count * 128 * 2 * sm_mhz * 1e6 / 1e12
        roof = {'bound': 'fp32', 'achieved': ach_tf, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach_tf / peak,
                'traffic': traffic, 'kernel': 'step_kernel', 'kernel_ms': kern_ms, 'share_of_step': kern_ms / step_ms,
                'flops_per_point': int(info.flops_per_point),
                'peak_source': '%d SMs x 128 FMA lanes x 2 x %.0f MHz (SM clock sampled under load)' % (info.sm_count, sm_mhz)}
    hbm = {'achieved': ach_gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach_gbs / hbm_peak, 'peak_source': peak_src,
           'bytes_per_point': int(info.bytes_per_point),
           'note': 'reported because BASELINE.json asks for it: the path is compute bound (flop/byte ~1e3-4e4)'}
    return roof, hbm


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument('--gpus', type=int, default=1)
    ap_.add_argument('--steps', type=int, default=200)
    ap_.add_argument('--warmup', type=int, default=5)
    ap_.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap_.add_argument('--workload', default='cfg2', choices=list(WORKLOADS))
    ap_.add_argument('--global-batch', type=int, default=0,
                     help='fix the GLOBAL batch (strong scaling); default: per-GPU batch of the workload (weak)')
    ap_.add_argument('--no-cpu-baseline', action='store_true')
    ap_.add_argument('--no-e2e', action='store_true')
    ap_.add_argument('--no-extras', action='store_true', help='skip strong_cfg5 / other_configs')
    ap_.add_argument('--reps', type=int, default=10, help='repetitions of the K-step timed region (min/median/max)')
    ap_.add_argument('--dump-outputs', metavar='DIR', default=None,
                     help='after the timed steps, write what their last step computed to DIR/<name>.npy')
    args = ap_.parse_args()
    K, W = args.steps, max(args.warmup, 3)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    os.environ.setdefault('PYDENS_B200_PROGRESS', '0')

    if args.impl == 'reference':
        if rank != 0:
            return
        res = cpu_reference(args.workload, args.gpus, K, W)
        line = {'impl': 'reference', 'metric': METRIC, 'value': res['value'], 'unit': 'points/s',
                'n_gpus': args.gpus, 'steps': res['steps'], 'warmup': W, 'ms_per_step': res['ms_per_step'],
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
                'data': 'synthetic', 'config': describe(args.workload, args.gpus),
                'cpu_baseline': {k: res[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
                'e2e': {'value': res['value'], 'unit': 'points/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device — the fused fit step has no CPU fallback '
                         '(use --impl reference for the CPU baseline)')
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    dev = torch.device('cuda', local_rank)

    name, batch, lr = WORKLOADS[args.workload]
    gbatch = args.global_batch if args.global_batch else batch * world

    clocks = ClockSampler(local_rank) if rank == 0 else None
    if clocks:
        clocks.start()

    # ---------------- value: K graph-replayed steps over an HBM-resident pool of batches, `reps` times ----------
    t = Timed(args.workload, gbatch, dev, rank, world, K, W)
    eng, info, total, local_n = t.eng, t.info, t.total, t.local_n
    check = t.allreduce_check()
    t_load0 = time.time()
    times, graphed = t.run(reps=args.reps)
    ms_sorted = sorted(times)
    ms_total = ms_sorted[len(ms_sorted) // 2]                       # median of the repetitions
    value = gbatch * K / (ms_total * 1e-3)
    last_loss = float(eng.out[eng.n_params].item())
    if args.dump_outputs and rank == 0:                             # before the runs below advance the parameters
        dump_outputs(t, args.dump_outputs)

    # ---------------- in-kernel sampling variant (the default `fit(sampler=None)` mode) ----------------
    sampled_value = None
    try:
        ts, _ = t.run(reps=3, sampled=True)
        sampled_value = gbatch * K / (sorted(ts)[1] * 1e-3)
    except Exception as exc:            # noqa: BLE001
        torch.cuda.synchronize()
        sys.stderr.write('sampled-variant run failed: %s\n' % exc)

    # ---------------- roofline: the fused kernel alone ----------------
    kern_ms = t.kernel_ms()
    kern_src = 'CUDA events around K back-to-back plain launches of the step kernel'
    if t.fused_adam and world == 1 and graphed and ms_total / K < kern_ms:
        # one launch per step: the timed region IS K launches of this kernel, and the graph replays them with a smaller
        # inter-launch gap than plain launches leave — the per-launch duration is the step time
        kern_ms = ms_total / K
        kern_src = 'the timed region itself: one launch of this kernel per graph-replayed step'
    t_load1 = time.time()

    # ---------------- e2e: Solver.fit with host batches (pinned H2D per step, loss D2H per step) --------
    e2e = None
    if not args.no_e2e:
        solver, cfg = t.solver, t.cfg
        host_pool = [torch.empty((gbatch, total)).pin_memory() for _ in range(min(max(K, 8), 32))]
        for hp in host_pool:
            for k, (lo, hi) in enumerate(cfg['ranges']):
                hp[:, k] = torch.rand(gbatch) * (hi - lo) + lo

        class HostBatches:
            i = 0

            def sample(self, size):
                self.i += 1
                return host_pool[self.i % len(host_pool)]
        hb = HostBatches()
        solver.fit(niters=max(W, 8), batch_size=gbatch, sampler=hb, lr=lr)      # warm-up: also builds the step graphs
        e2e_times = []
        for _ in range(max(3, args.reps // 2)):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            solver.fit(niters=K, batch_size=gbatch, sampler=hb, lr=lr)
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            e2e_times.append(float(dt.item()))
        dt_med = sorted(e2e_times)[len(e2e_times) // 2]
        e2e = {'value': gbatch * K / dt_med, 'unit': 'points/s',
               'h2d_bytes_per_step': int(local_n * total * 4) * world, 'd2h_bytes_per_step': 4 * world,
               'ms_per_step': 1e3 * dt_med / K,
               'ms_per_step_min_median_max': [1e3 * min(e2e_times) / K, 1e3 * dt_med / K, 1e3 * max(e2e_times) / K],
               'repetitions': len(e2e_times),
               'api': 'Solver.fit(niters=K, batch_size=B, sampler=<host batches in pinned memory>), wall clock around the '
                      'call incl. its final synchronisation; every step: one H2D copy of the batch, one D2H read of the loss'}

    clk = clocks.stop(t_load0, t_load1) if clocks else None

    # ---------------- the other BASELINE configurations (N=1) and cfg5 strong scaling (4 M points over N GPUs) --------
    other, strong = None, None
    if not args.no_extras and args.workload == 'cfg2' and not args.global_batch:
        kk = max(3, min(K, 10))
        del t.pool
        torch.cuda.empty_cache()
        try:
            ts5 = Timed('cfg5', 4000000, dev, rank, world, kk, 3, pool_cap_bytes=1 << 30)
            tms, _ = ts5.run(reps=3)
            med = sorted(tms)[1]
            strong = {'workload': 'cfg5 wave3d, MLP [4, 64, 64, 64, 64, 1] Tanh', 'global_batch': 4000000, 'n_gpus': world,
                      'scaling': 'strong', 'steps': kk, 'ms_per_step': med / kk, 'value': 4000000 * kk / (med * 1e-3),
                      'unit': 'points/s', 'kernel': 'tcgen05 tile kernel' if ts5.info.tensor_core else 'thread kernel',
                      'allreduce_check': ts5.allreduce_check(),
                      'note': 'same code at every N: the driver can form the 1->N strong-scaling ratio from these lines'}
            del ts5
            torch.cuda.empty_cache()
        except Exception as exc:        # noqa: BLE001
            strong = {'error': str(exc)[:200]}
        if world == 1:
            other = {}
            for wl in ('cfg3', 'cfg4', 'cfg5'):
                try:
                    tw = Timed(wl, WORKLOADS[wl][1], dev, rank, world, kk, 3, pool_cap_bytes=1 << 30)
                    tms, _ = tw.run(reps=3)
                    med = sorted(tms)[1] / kk
                    km = min(tw.kernel_ms(reps=3), med) if tw.fused_adam else tw.kernel_ms(reps=3)
                    roof, _ = roofline_blocks(tw, km, med, clk, _peaks(), wl)
                    other[wl] = {'workload': describe(wl, 1)['workload'], 'ms_per_step': med,
                                 'value': WORKLOADS[wl][1] / (med * 1e-3), 'unit': 'points/s', 'steps': kk,
                                 'roofline': {k: roof[k] for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic', 'kernel_ms')}}
                    del tw
                    torch.cuda.empty_cache()
                except Exception as exc:        # noqa: BLE001
                    other[wl] = {'error': str(exc)[:200]}

    torch.cuda.synchronize()
    if rank != 0:
        _shutdown(dist, world)
        return

    peaks = _peaks()
    roof, hbm = roofline_blocks(t, kern_ms, ms_total / K, clk, peaks, args.workload)
    roof['kernel_ms_source'] = kern_src
    n_ctas = min(info.sm_count, (local_n + 127) // 128) if info.tensor_core else \
        min(info.sm_count, (local_n + info.threads_per_cta - 1) // info.threads_per_cta)
    line = {
        'metric': METRIC, 'value': value, 'unit': 'points/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms_total / K, 'higher_is_better': True,
        'scaling': 'strong' if args.global_batch else 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'timing': {'repetitions': len(times), 'ms_per_step_min': ms_sorted[0] / K, 'ms_per_step_median': ms_total / K,
                   'ms_per_step_max': ms_sorted[-1] / K, 'value_is': 'median over repetitions of K graph-replayed steps'},
        'config': dict(describe(args.workload, world), global_batch=gbatch,
                       inputs='HBM-resident pool of %d distinct batches (%.0f MB%s), one per step; '
                              'in-kernel Philox sampling variant reported as value_sampled'
                              % (t.pool_n, t.pool_n * local_n * total * 4 / 1e6,
                                 ' > L2' if t.pool_n * local_n * total * 4 > 126e6 else ''),
                       cuda_graph=graphed, final_loss=last_loss,
                       optimizer_step=('torch.optim.Adam update in the tail of the step kernel (pinn_step_adam): one launch '
                                       'per step' if t.fused_adam else 'torch fused Adam kernels + pinn_record_loss'),
                       allreduce=('in-kernel over NVLink peer memory (pinn_step_allreduce)' if eng.comm is not None
                                  else ('NCCL' if world > 1 else 'none')),
                       kernel='%s<NF=%d,NS=%d> %d threads/CTA x %d CTAs, %d B smem, %d regs, per-point state in %s'
                              % ('wide_step_kernel' if info.tensor_core else 'step_kernel', info.nf, info.ns,
                                 info.threads_per_cta, n_ctas, info.smem_bytes, info.regs_per_thread,
                                 'TMEM + L2 slab' if info.tensor_core else ('smem' if info.activations_in_smem else 'gmem'))),
        'value_sampled': sampled_value,
        'gpu_launches': (1 if t.fused_adam else 2) * K,
        'clocks': clk,
        'roofline': roof,
        'hbm': hbm,
        'e2e': e2e,
    }
    if check is not None:
        line['allreduce_check'] = check
    if strong is not None:
        line['strong_cfg5'] = strong
    if other is not None:
        line['other_configs'] = other
    if not args.no_cpu_baseline and world == 1:
        cb = cpu_reference(args.workload, 1, 40, 2, budget_s=20.0)
        line['cpu_baseline'] = {k: cb[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
    print(json.dumps(line), flush=True)
    _shutdown(dist, world)


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except (OSError, ValueError):
        return {}


def _shutdown(dist, world):
    """ Tear the process group down; never let a stuck NCCL teardown keep the job alive. """
    if world <= 1:
        return
    t = threading.Thread(target=lambda: (dist.barrier(), dist.destroy_process_group()), daemon=True)
    t.start()
    t.join(20.0)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == '__main__':
    main()
