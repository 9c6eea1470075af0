#!/usr/bin/env python
"""bench.py — SCoNe train trajectories/s on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg5|cfg4|cfg1|cfg3-ebli|cfg3-bunch]
                    [--scaling strong|weak] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one optimizer step of the 3-layer model over one batch of synthetic trajectories on the named complex: plan (cone &
support -> live rows + gather programs) -> fused forward / readout / NLL / backward per trajectory -> partial reduce -> (all-reduce
of the flat [grads | nll | count] buffer when N > 1) -> Adam.  Every trajectory of the batch contributes to the loss (mask all ones).

  cfg5 (default)  1M-edge complex, GLOBAL batch 32768 (BASELINE.json config 5).  --scaling strong (default): 32768 / N trajectories
                  per GPU, the same global batch at every N; --scaling weak: 4096 per GPU.
  value           whole-job trajectories/s with the batch already resident in HBM (device-timed with CUDA events, max over ranks)
  e2e             same metric through the public host API (SconeModel.loss_grad + adam_step on pinned HOST buffers, H2D of the batch
                  and D2H of the loss inside the timed region)
  roofline        the dominant tensor-moving kernel, timed live with CUDA events on its launching stream in a SEPARATE profiled pass
                  (the value loop runs with profiling off); bytes = device-counted live rows x SURVEY 8(d)'s per-row figures
  roofline_dense  the contracted dense-tile measurement: one fused 32->32 layer on dense random features [E][64][32], no pruning
  parity_check    the GPU's log-probs / NLL / gradients for the cpu_baseline sample against the oracle (1e-5 / 1e-4)
  cpu_baseline    the oracle's CPU port on a bounded sample, rank 0, N = 1 only
--impl reference times that CPU port as the whole arm (jax is not installable offline and the dense E x E formulation cannot be
instantiated at E = 1M — DESIGN.md), with every host thread.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    'cfg5': dict(n_nodes=370000, global_batch=32768, weak_batch=4096, hidden=32, model='scone', cuts=8,
                 desc='1M-edge synthetic holed Delaunay complex, global batch 32768 trajectories, 3-layer SCoNe hidden 32'),
    'cfg4': dict(n_nodes=110000, global_batch=4096, weak_batch=4096, hidden=32, model='scone', cuts=1,
                 desc='~300k-edge synthetic complex, batch 4096, 3-layer SCoNe hidden 32'),
    'cfg1': dict(n_nodes=400, global_batch=1000, weak_batch=1000, hidden=16, model='scone', cuts=1,
                 desc='default synthetic complex (400 nodes), 1000 trajectories, 3-layer SCoNe hidden 16'),
    'cfg3-ebli': dict(n_nodes=400, global_batch=1000, weak_batch=1000, hidden=16, model='ebli', cuts=1,
                      desc='default synthetic complex (400 nodes), 1000 trajectories, 3-layer SNN (-model ebli) hidden 16'),
    'cfg3-bunch': dict(n_nodes=400, global_batch=1000, weak_batch=1000, hidden=16, model='bunch', cuts=1,
                       desc='default synthetic complex (400 nodes), 1000 trajectories, SCCONV (-model bunch) 7_16_7_16_7_16'),
}
KIND_NAMES = ['layer_fwd', 'layer_bwd', 'layer0_fwd', 'layer0_bwd', 'readout', 'flows_to_dense', 'zero_fill', 'cone']
PIPELINES = {4: 'trajectory-fused kernels: plan + fused forward/backward + partial reduce', 3: 'row lists over the readout cone, compact tensors',
             2: 'row lists, compact tensors', 1: 'row lists, dense tensors', 0: 'unit kernels, byte flags'}


def load_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).  The timed region can be
    shorter than one `nvidia-smi` invocation, so the sampler polls NVML in-process (nvidia_ml_py, ~1 kHz, own thread);
    `nvidia-smi -lms` is the fallback when NVML cannot be loaded."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.rows, self.proc, self.index, self.nv, self.h = [], None, index, None, None
        self.running, self.th, self.source = False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(',')[self.index])
                except Exception:
                    idx = self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.running, self.source = True, 'nvml'
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = 'nvidia-smi'
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        bits = [(getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8), 'hw_slowdown'),
                (getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40), 'hw_thermal_slowdown'),
                (getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20), 'sw_thermal_slowdown'),
                (getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4), 'sw_power_cap')]
        get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons

        def once():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = int(get_reasons(self.h))
                self.rows.append([sm, self.mx, 0.0] + ['Active' if r & bit else 'Not Active' for bit, _ in bits])
            except Exception:
                pass
        self._once = once
        while self.running:
            once()
            time.sleep(0.001)

    def sample_while(self, busy):
        """Poll from the CALLING thread while busy() holds (the timed steps are enqueued and the GPU is working through them): the
        background thread alone can be starved by the interpreter lock and leave a single sample."""
        once = getattr(self, '_once', None)
        while busy():
            if once is not None and self.nv is not None:
                once()
            time.sleep(0.001)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.nv is not None:
            self.running = False
            self.th.join(timeout=2)
        elif self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        else:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no NVML, no nvidia-smi'], 'samples': 0}
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nme, v in zip(self.NAMES, r[3:7]):
                    if str(v).lower().startswith('active'):
                        reasons.add(nme)
            except Exception:
                pass
        sm.sort()
        load = [x for x in sm if mx and x > 0.3 * mx] or sm
        return {'sm_mhz': (load[len(load) // 2] if load else None), 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm), 'source': self.source}


def ncu_traffic(kernel_pattern, tag, launches_per_step=1):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set full` capture
    of this round (profiles/prof_<tag>_raw.csv) — only quoted when the capture was taken on the same launch shape.  A kernel that runs
    as several launches per step (the fused compute kernel: its small and its big row-store class) is summed over them, like `achieved`."""
    path = os.path.join(ROOT, 'profiles', 'prof_%s_raw.csv' % tag)
    if not os.path.exists(path):
        return None
    try:
        import csv
        rows = list(csv.reader(open(path)))
        hdr, unit = rows[0], rows[1]
        kn = hdr.index('Kernel Name')
        scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
        tot, n = 0.0, 0
        for val in rows[2:]:
            if len(val) < len(hdr) or kernel_pattern not in val[kn]:
                continue
            for name in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                i = hdr.index(name)
                tot += float(val[i]) * scale[unit[i]]
            n += 1
        return tot / (n / float(launches_per_step)) if n else None
    except Exception:
        return None


def make_dataset(name, cfg, n_traj, seed):
    from scone_gcn_b200 import synthetic_data_gen as sdg
    if cfg['n_nodes'] <= 1000:
        sys.path.insert(0, os.path.join(ROOT, 'tests'))
        from golden_util import Dataset
        ds = Dataset('dataset_default.npz')
        return sdg.SparseDataset.from_dense(ds.flows, ds.B1, ds.B2, ds.targets, ds.train_mask, ds.test_mask, ds.last_nodes, ds.target_nodes), ds
    return sdg.generate_sparse_dataset(cfg['n_nodes'], n_traj, seed=seed, n_waypoints=24, cuts_per_walk=cfg['cuts']), None


def dump_outputs(path, grad_buffer, weights=None):
    """What a caller of the timed step receives from its last run: the flat [grads | nll_sum | count] buffer of that step and, when
    the step ends with an Adam update, the flat weights after it.  The inputs are seeded, so two builds run with the same arguments
    compare file for file."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, 'grad_buffer.npy'), np.asarray(grad_buffer, np.float32))
    if weights is not None:
        np.save(os.path.join(path, 'weights.npy'), np.asarray(weights, np.float32))


def tri_lists(sp):
    from scone_gcn_b200.complex import incidence_lists_from_simplices
    return incidence_lists_from_simplices(sp.edges, sp.faces)


def oracle_sample(sp, model, W, n_sample, repeats, dtype=None):
    """Oracle port (CPU, torch sparse, all host threads) over the first n_sample trajectories: (log-probs, nll, grads, times)."""
    import numpy as np
    import torch
    from oracle import scone_oracle as so
    torch.set_num_threads(os.cpu_count() or 1)
    en, es, te, ts = tri_lists(sp)
    orc = so.SparseOracle(model, sp.edges, te, ts, int(sp.n_nodes), dtype=dtype or np.float32)
    E = len(sp.edges)
    X = np.zeros((E, n_sample), np.float32)
    for t in range(n_sample):
        sl = slice(sp.traj_ptr[t], sp.traj_ptr[t + 1])
        X[sp.flow_edge[sl], t] = sp.flow_val[sl]
    times, nll, grads = [], None, None
    for _ in range(repeats):
        t0 = time.perf_counter()
        nll, grads = orc.loss_and_grads(W, X, sp.last_nodes[:n_sample], sp.target_idx[:n_sample], np.ones(n_sample, np.float32))
        times.append(time.perf_counter() - t0)
    lp = orc.forward(W, X, sp.last_nodes[:n_sample])
    return lp, nll, grads, times, torch.get_num_threads()


def sample_size(E):
    return 2 if E > 500000 else (8 if E > 2000 else 64)


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    import numpy as np
    sp, _ = make_dataset(args.config, cfg, 64, 1030)
    E = len(sp.edges)
    model = cfg['model'] if cfg['model'] != 'bunch' else 'scone'
    C = cfg['hidden']
    rs = np.random.RandomState(1030)
    W = [0.01 * rs.randn(*s) for s in [(1, C)] * 3 + [(C, C)] * 6 + [(C, 1)]]
    n_sample = sample_size(E)
    lp, nll, grads, times, threads = oracle_sample(sp, model, W, n_sample, args.warmup + args.steps)
    if args.dump_outputs:                                  # the oracle step has no optimizer update: gradients and loss only
        dump_outputs(args.dump_outputs, np.concatenate([g.ravel() for g in grads] + [np.array([nll, n_sample])]))
    times = times[args.warmup:] or times
    tps = n_sample / (sum(times) / len(times))
    sample = '%d trajectories fwd+bwd per step on the same complex (E=%d), sparse CSR CPU port of the reference maths' % (n_sample, E)
    out = {'impl': 'reference', 'metric': 'SCoNe train trajectories/sec', 'value': tps, 'unit': 'trajectories/s',
           'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(times) / len(times),
           'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
           'config': {'workload': args.config + ': ' + cfg['desc'], 'E': int(E), 'N': int(sp.n_nodes), 'F': int(len(sp.faces)),
                      'global_batch': cfg['global_batch'], 'sample_trajectories_per_step': n_sample},
           'cpu_baseline': {'value': tps, 'unit': 'trajectories/s', 'cores': threads, 'kind': 'port', 'sample': sample},
           'e2e': {'value': tps, 'unit': 'trajectories/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
           'gpu_launches': 0,
           'note': 'jax is not installable offline and the dense E x E reference formulation cannot be instantiated at this size; this is '
                   'the oracle port (oracle/scone_oracle.py SparseOracle) on torch CPU sparse kernels with torch.set_num_threads(os.cpu_count())'}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='cfg5', choices=sorted(CONFIGS))
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'])
    ap.add_argument('--batch', type=int, default=0, help='override the per-GPU batch')
    ap.add_argument('--micro-batch', type=int, default=0)
    ap.add_argument('--pipeline', type=int, default=-1, help='force a model-level pipeline (default: the library\'s choice)')
    ap.add_argument('--exchange', default='peer', choices=['peer', 'nccl'],
                    help='N > 1: gradient exchange fused with Adam over NVLink peer memory (one kernel), or NCCL all-reduce + Adam kernel')
    ap.add_argument('--e2e-steps', type=int, default=10)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', dest='extras', action='store_false', help='skip the dense-tile roofline measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed (grad_buffer.npy, and weights.npy after the Adam update; '
                         'float32) to DIR')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    cfg = dict(CONFIGS[args.config])
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        return run_reference(args, cfg, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import _lib, dp
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    saved_stdout = None
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner to fd 1 at the first collective, so fd 1 points at
        # stderr until the result is printed
        os.environ['NCCL_DEBUG_FILE'] = '/dev/stderr'
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=dev)
    L = sg.lib()

    t_setup = time.time()
    # strong scaling: ONE global batch (same seed on every rank), rank r owns the contiguous shard dp.shard_range gives it;
    # weak scaling: weak_batch trajectories per GPU, generated per rank
    if args.scaling == 'strong':
        gb = cfg['global_batch'] if not args.batch else args.batch * world
        sp, dense_ds = make_dataset(args.config, cfg, gb, 1030)
        gb = min(gb, sp.n_traj)
        lo, hi = dp.shard_range(gb, rank, world)
    else:
        per = args.batch or cfg['weak_batch']
        sp, dense_ds = make_dataset(args.config, cfg, per, 1030 + rank)
        per = min(per, sp.n_traj)
        lo, hi, gb = 0, per, per * world
    B = hi - lo
    model = cfg['model']
    C = cfg['hidden']
    p0, p1 = int(sp.traj_ptr[lo]), int(sp.traj_ptr[hi])
    ptr = (sp.traj_ptr[lo:hi + 1] - sp.traj_ptr[lo]).astype(np.int32)

    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h = dict(ptr=pinned(ptr), edge=pinned(sp.flow_edge[p0:p1].astype(np.int32)), val=pinned(sp.flow_val[p0:p1].astype(np.float32)),
             last=pinned(sp.last_nodes[lo:hi].astype(np.int32)), tgt=pinned(sp.target_idx[lo:hi].astype(np.int32)),
             mask=pinned(np.ones(B, np.float32)))
    h2d_bytes = sum(v.numel() * v.element_size() for v in h.values())
    hp = {k: v.numpy() for k, v in h.items()}
    stream = torch.cuda.current_stream().cuda_stream
    lr, wd = 1e-3, 5e-5
    step_no = [0]
    rs = np.random.RandomState(1030)                       # same init on every rank

    if model == 'bunch':
        return bench_bunch(args, cfg, sp, dense_ds, hp, h2d_bytes, B, gb, world, rank, dev, stream, t_setup)

    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, model)
    mb = min(args.micro_batch or B, B)
    net = sg.SconeModel(cx, [C, C, C], micro_batch=mb)
    if args.pipeline >= 0:
        net.set_pipeline(args.pipeline)
    net.set_weights([0.01 * rs.randn(*s) for s in net.shapes])
    E, N, F, D = cx.E, cx.N, cx.F, cx.D
    d = {k: v.to(dev) for k, v in h.items()}
    gbuf = net.grads_tensor()

    exchange = None
    if world > 1 and args.exchange == 'peer':
        os.environ.pop('SCONE_DP_EXCHANGE', None)
        exchange = dp.make_exchange(net.n_params + 2, dev)   # None (with a message on stderr) if the peers cannot be mapped

    def optimizer_step():
        if exchange is not None:                           # sum over ranks + Adam: one kernel over NVLink peer memory
            exchange.adam_step(net, step_no[0], lr, wd, stream)
        else:
            if world > 1:
                dist.all_reduce(gbuf)
            net.adam_step(step_no[0], lr, wd, stream)
        step_no[0] += 1

    def step_dev():
        _lib.check(L.scone_model_loss_grad_dev(net.handle, B, _lib.dptr(d['ptr']), _lib.dptr(d['edge']), _lib.dptr(d['val']),
                                               _lib.dptr(d['last']), _lib.dptr(d['tgt']), _lib.dptr(d['mask']), 1, stream))
        optimizer_step()

    def step_e2e():
        net.loss_grad(hp['ptr'], hp['edge'], hp['val'], hp['last'], hp['tgt'], hp['mask'], zero_first=True, stream=stream, read=False)
        optimizer_step()
        buf = net.read_grads(stream)                       # D2H of [grads | nll_sum | count]: the step's loss
        return float(buf[-2] / buf[-1])

    # The same step, software-pipelined by the caller: every step's H2D copies, kernels and the D2H of its loss are enqueued before
    # the host looks at the PREVIOUS step's loss, so the GPU never waits for the host and the library copies the next batch's flow
    # arrays under the current compute kernel.  Every step still moves its own inputs and its own result.
    gpin = [torch.empty(net.n_params + 2, dtype=torch.float32).pin_memory() for _ in range(2)]
    gev = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_enqueue(k):
        net.loss_grad(hp['ptr'], hp['edge'], hp['val'], hp['last'], hp['tgt'], hp['mask'], zero_first=True, stream=stream, read=False)
        optimizer_step()
        net.read_grads_async(gpin[k & 1], stream)
        gev[k & 1].record()

    def e2e_collect(k):
        gev[k & 1].synchronize()
        g = gpin[k & 1]
        return float(g[-2] / g[-1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        step_dev()
    barrier()
    net.check_overflow(stream)
    setup_s = time.time() - t_setup

    # ---- value: profiling OFF, batch resident ----
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = L.scone_launch_count()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step_dev()
    ev1.record()
    launches = L.scone_launch_count() - launches0
    clocks.sample_while(lambda: not ev1.query())           # (host-side polling of NVML: nothing is enqueued on the GPU)
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    clk = clocks.stop()
    net.check_overflow(stream)                             # a truncated step would have been timed silently otherwise
    if exchange is not None:
        exchange.status(stream)                            # ... and so would a step whose peers never delivered their gradients
    if args.dump_outputs and rank == 0:                    # before the passes below run more steps on the same model
        dump_outputs(args.dump_outputs, net.read_grads(stream), net.flatten(net.get_weights()))
    ms_per_step = ms_total / args.steps
    value = gb * args.steps / (ms_total / 1e3)

    # ---- separate profiled pass: per-kernel-family device time (CUDA events around each launch on the launching stream) ----
    prof_steps = min(args.steps, 5)
    L.scone_profile_reset()
    L.scone_profile_enable(1)
    done = (ctypes.c_int64 * 2)()
    L.scone_model_read_rows_done(net.handle, done)
    for _ in range(prof_steps):
        step_dev()
    barrier()
    L.scone_profile_enable(0)
    fam = {}
    for k, nme in enumerate(KIND_NAMES):
        n_l, t_ms = ctypes.c_int64(), ctypes.c_double()
        L.scone_profile_read(k, n_l, t_ms)
        fam[nme] = (n_l.value, t_ms.value)
    L.scone_model_read_rows_done(net.handle, done)
    rows = {'layer_fwd': int(done[0]), 'layer_bwd': int(done[1])}
    pipeline_id = net.pipeline
    if pipeline_id != 4:
        for k, nme in ((0, 'layer_fwd'), (1, 'layer_bwd')):
            r = ctypes.c_int64()
            L.scone_profile_read_rows(k, r)
            rows[nme] = r.value
    peak, peak_src = load_peaks()
    # ALGORITHMIC bytes (DESIGN.md 4): per produced live row a fused layer forward reads one input row and writes one output row
    # (4*(Cin+Cout) bytes), a backward reads G and Hin rows and writes Gprev (4*(2*Cin+Cout)) — SURVEY 8(d)'s per-row figures;
    # the fused compute kernel does both passes in one launch, so its bytes are the sum
    alg = {}
    if pipeline_id == 4:
        if fam['layer_bwd'][0]:
            alg['layer_bwd'] = (rows['layer_fwd'] * 4.0 * 2 * C + rows['layer_bwd'] * 4.0 * 3 * C) / fam['layer_bwd'][0]
    else:
        if fam['layer_fwd'][0]:
            alg['layer_fwd'] = rows['layer_fwd'] * 4.0 * 2 * C / fam['layer_fwd'][0]
        if fam['layer_bwd'][0]:
            alg['layer_bwd'] = rows['layer_bwd'] * 4.0 * 3 * C / fam['layer_bwd'][0]
    tot_ms = sum(t for _, t in fam.values()) or 1.0
    table_plan = pipeline_id == 4 and bool((net.fused_info() or {}).get('table_plan_mb'))
    names = {'layer_bwd': 'fused_traj_kernel (small + big row-store launches; + cost sort, fused_reduce_kernel)',
             'cone': 'table_plan_kernel (three tiers)' if table_plan else 'fused_plan_kernel (two tiers)'} if pipeline_id == 4 else {}
    kernels = {}
    for nme, (n_l, t_ms) in fam.items():
        if n_l:
            avg = t_ms / n_l
            kernels[nme] = {'kernel': names.get(nme, nme), 'launches': n_l, 'avg_ms': avg, 'share_of_kernel_time': t_ms / tot_ms}
            if nme in alg:
                kernels[nme].update({'algorithmic_bytes_per_launch': alg[nme], 'achieved_gbs': alg[nme] / avg / 1e6, 'frac': alg[nme] / avg / 1e6 / peak})
    with_bytes = [k_ for k_ in kernels if 'achieved_gbs' in kernels[k_]]
    dom = max(with_bytes or kernels, key=lambda k_: kernels[k_]['share_of_kernel_time'])
    largest = max(kernels, key=lambda k_: kernels[k_]['share_of_kernel_time'])
    dense_bytes_per_traj = 4.0 * E * (15 * C + 2)
    step_alg_bytes = (rows['layer_fwd'] * 4.0 * 2 * C + rows['layer_bwd'] * 4.0 * 3 * C) / prof_steps
    roofline = {'bound': 'hbm', 'kernel': kernels[dom]['kernel'], 'achieved': kernels[dom].get('achieved_gbs'), 'peak': peak, 'unit': 'GB/s',
                'frac': kernels[dom].get('frac'),
                'traffic': ncu_traffic('fused_traj_kernel', 'fused_r2_' + args.config, 2) if pipeline_id == 4 else None,
                'peak_source': peak_src, 'largest_family': kernels[largest]['kernel'],
                'algorithmic_bytes_per_launch': kernels[dom].get('algorithmic_bytes_per_launch'),
                'whole_step': {'algorithmic_bytes': step_alg_bytes, 'achieved_gbs': step_alg_bytes / ms_per_step / 1e6,
                               'frac': step_alg_bytes / ms_per_step / 1e6 / peak},
                'rows_per_step': {k_: v_ / prof_steps for k_, v_ in rows.items()},
                'dense_rows_per_step': float(E) * B * 2,
                'kernels': kernels,
                'dense_equivalent': {'bytes_per_trajectory': dense_bytes_per_traj,
                                     'effective_gbs': dense_bytes_per_traj * value / world / 1e9,
                                     'note': 'SURVEY 8(d) dense formula 4*E*(15C+2) bytes per trajectory times the measured per-GPU '
                                             'trajectories/s: what a dense-streaming implementation would have to move to match'},
                'bytes_model': 'live rows produced (device-counted) x 4*(Cin+Cout) per forward row and 4*(2*Cin+Cout) per backward row '
                               '(SURVEY 8(d) per-row figures; index arrays and the gather programs excluded, as there).  The fused compute kernel '
                               'keeps those rows in shared memory, so its real DRAM traffic (roofline.traffic, ncu) is far BELOW the algorithmic '
                               'bytes: it is bound by instruction issue / mma.sync rate and smem latency, the plan kernel by dependent L2 loads — '
                               'neither by HBM.  The contracted dense-tile figure is roofline_dense.',
                'pipeline': PIPELINES.get(pipeline_id, str(pipeline_id))}

    # ---- epoch >= 2 of a training run: the batch's plans are already on the device (weight-independent: Scone_GCN.train plans its
    # dataset once, scone_model_plan_*), a step runs only the compute kernel + reduce (+ all-reduce) + Adam.  Reported next to
    # `value`, never instead of it: `value` plans every step. ----
    plans_cached = None
    if pipeline_id == 4:
        _lib.check(L.scone_model_plan_dev(net.handle, B, _lib.dptr(d['ptr']), _lib.dptr(d['edge']), _lib.dptr(d['val']), _lib.dptr(d['last']), stream))

        def step_planned():
            _lib.check(L.scone_model_loss_grad_planned_dev(net.handle, B, None, _lib.dptr(d['tgt']), _lib.dptr(d['mask']), 1, stream))
            if world > 1:
                dist.all_reduce(gbuf)
            net.adam_step(step_no[0], lr, wd, stream)
            step_no[0] += 1
        for _ in range(3):
            step_planned()
        barrier()
        ev0.record()
        for _ in range(args.steps):
            step_planned()
        ev1.record()
        barrier()
        pc_ms = max_over_ranks(ev0.elapsed_time(ev1))
        plans_cached = {'value': gb * args.steps / (pc_ms / 1e3), 'unit': 'trajectories/s', 'ms_per_step': pc_ms / args.steps, 'steps': args.steps,
                        'note': 'the same step with the plans of the batch kept from an earlier step (a dataset revisited every epoch is planned '
                                'once); compute kernel + partial reduce + Adam only'}

    # ---- end to end through the host API ----
    barrier()
    e2e_steps = max(1, args.e2e_steps)
    step_e2e()
    barrier()
    ev0.record()
    loss = None
    for k in range(e2e_steps):
        e2e_enqueue(k)
        if k:
            loss = e2e_collect(k - 1)
    loss = e2e_collect(e2e_steps - 1)
    ev1.record()
    barrier()
    e2e_ms = max_over_ranks(ev0.elapsed_time(ev1))
    net.check_overflow(stream)
    # the unpipelined variant (the host reads every step's loss before it enqueues the next step), for comparison
    barrier()
    ev0.record()
    for _ in range(e2e_steps):
        step_e2e()
    ev1.record()
    barrier()
    e2e_sync_ms = max_over_ranks(ev0.elapsed_time(ev1))
    e2e = {'value': gb * e2e_steps / (e2e_ms / 1e3), 'unit': 'trajectories/s', 'h2d_bytes_per_step': h2d_bytes,
           'd2h_bytes_per_step': int(4 * (net.n_params + 2)), 'steps': e2e_steps, 'last_loss': loss,
           'note': 'host API with pinned host buffers; per step: H2D of the batch, plan + compute + optimizer step, D2H of [grads | nll | count]; '
                   'the caller enqueues step k + 1 before it reads the loss of step k (scone_model_read_grads_async)',
           'unpipelined_value': gb * e2e_steps / (e2e_sync_ms / 1e3)}

    # ---- the contracted DENSE-tile measurement (north-star / SURVEY 8d): one fused 32->32 layer on dense random features,
    # no pruning, algorithmic bytes 4*E*b*(Cin+Cout) fwd and 4*E*b*(2*Cout+Cin) bwd ----
    roofline_dense = None
    if args.extras and rank == 0 and E > 100000:
        roofline_dense = dense_tile_roofline(L, cx, E, C, dev, stream, peak)

    # ---- parity on THIS workload + CPU baseline (rank 0, N = 1): the oracle port on a bounded sample ----
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_sample = sample_size(E)
        W_now = net.get_weights()
        lp_o, nll_o, g_o, times, threads = oracle_sample(sp, model, W_now, n_sample, 2)
        tps = n_sample / min(times)
        cpu_baseline = {'value': tps, 'unit': 'trajectories/s', 'cores': threads, 'kind': 'port',
                        'sample': '%d trajectories fwd+bwd on the same complex (E=%d), best of 2; sparse CSR CPU port '
                                  '(oracle/scone_oracle.py), torch CPU sparse kernels' % (n_sample, E)}
        nz = int(sp.traj_ptr[n_sample])
        a = (sp.traj_ptr[:n_sample + 1].astype(np.int32), sp.flow_edge[:nz].astype(np.int32), sp.flow_val[:nz].astype(np.float32),
             sp.last_nodes[:n_sample].astype(np.int32))
        lp_g = net.forward(*a)
        buf = net.loss_grad(*a, sp.target_idx[:n_sample].astype(np.int32), np.ones(n_sample, np.float32))
        g_g = net.unflatten(buf[:net.n_params])
        lp_err = float(np.abs(lp_g - lp_o).max() / max(1.0, np.abs(lp_o).max()))
        gmax = max(float(np.abs(y).max()) for y in g_o)
        g_err = max(float(np.abs(x - y).max() / max(np.abs(y).max(), 1e-3 * gmax, 1e-30)) for x, y in zip(g_g, g_o))
        nll_err = float(abs(buf[net.n_params] - nll_o) / max(1.0, abs(nll_o)))
        parity = {'against': 'oracle/scone_oracle.py SparseOracle (fp32)', 'trajectories': n_sample, 'weights': 'after the timed Adam steps',
                  'logprob_max_err': lp_err, 'grad_max_rel_err': g_err, 'nll_rel_err': nll_err,
                  'tolerance': {'logprob': 1e-5, 'grad': 1e-4}, 'ok': bool(lp_err <= 1e-5 and g_err <= 1e-4 and nll_err <= 1e-5)}

    if rank == 0:
        nnz = p1 - p0
        info = net.fused_info() if pipeline_id == 4 else None
        touched = 8.0 * nnz + 16.0 * B * 4 + (step_alg_bytes if pipeline_id != 4 else 0.0)
        if pipeline_id == 4:
            # ncu (profiles/prof_r2*): the plan kernels read ~0.24 GB and write ~0.48 GB of DRAM per 32768 trajectories (node-table rows of
            # 32768 random nodes out of a %d MB table; programs written), the compute kernel reads ~0.44 GB (programs back)
            tb_mb = (info or {}).get('table_plan_mb', 0)
            per_step = touched + B * 20e3 + B * 8e3
            l2_policy = ('inputs larger than L2: a step reads %.0f MB of flows / last nodes / targets, the node-table rows of the %d last nodes '
                         '(~20 KB each, random rows of a %d MB table) and writes + re-reads the gather programs (~8 KB per trajectory): ~%.0f MB per '
                         'step, %s the 126 MB L2; no explicit flush'
                         % (touched / 1e6, B, tb_mb, per_step / 1e6, 'larger than' if per_step > 126e6 else 'SMALLER than'))
        else:
            l2_policy = 'no explicit flush; compact row tensors of ~%.0f MB per step' % (touched / 1e6)
        out = {'metric': 'SCoNe train trajectories/sec', 'value': value, 'unit': 'trajectories/s', 'n_gpus': world,
               'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_per_step, 'higher_is_better': True,
               'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
               'config': {'workload': args.config + ': ' + cfg['desc'] + (' (%d per GPU)' % B if world > 1 else ''),
                          'N': N, 'E': E, 'F': F, 'D': D, 'model': model, 'per_gpu_batch': B, 'global_batch': gb, 'hidden': C,
                          'layers': 3, 'micro_batch': mb,
                          'parallelism': 'dp%d (trajectory shards, complex replicated, one sum of %d floats over ranks per step: %s)' % (
                              world, net.n_params + 2, 'none at N = 1' if world == 1 else
                              ('NVLink peer-memory push + Adam in one kernel (scone_dp.cu)' if exchange is not None else 'NCCL all-reduce, then the Adam kernel')),
                          'l2_policy': l2_policy, 'generator_seed': 1030, 'mean_flow_nnz': nnz / B,
                          'trajectories': ('prefixes of %d BEGIN->A->B->END walks cut at %d random points each' % (-(-gb // cfg['cuts']), cfg['cuts']))
                          if cfg['n_nodes'] > 1000 else 'the reference generator\'s 1000 trajectories (tests/golden/dataset_default.npz)'},
               'roofline': roofline, 'roofline_dense': roofline_dense, 'plans_cached': plans_cached, 'e2e': e2e,
               'cpu_baseline': cpu_baseline, 'parity_check': parity, 'gpu_launches': int(launches),
               'clocks': clk, 'setup_s': setup_s, 'fused_info': info}
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(out), flush=True)
        if parity is not None and not parity['ok']:
            sys.stderr.write('bench parity check FAILED: %s\n' % parity)
            sys.exit(3)
    if world > 1:
        dist.destroy_process_group()


def dense_tile_roofline(L, cx, E, C, dev, stream, peak):
    import torch
    from scone_gcn_b200 import _lib
    bd = 64
    Hd = torch.randn(E, bd, C, device=dev)
    Od = torch.empty_like(Hd)
    Wd = [torch.randn(C, C, device=dev) * 0.2 for _ in range(3)]
    wsd = torch.empty(L.scone_layer_backward_workspace_bytes(C, C) // 4 + 16, device=dev)
    dWd = torch.zeros(3, C, C, device=dev)

    def t_of(fn, it=3):
        fn()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(it):
            a, z = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            z.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(z))
        return best
    def fwd():
        _lib.check(L.scone_layer_forward(cx.handle, 0, bd, C, C, _lib.dptr(Hd), _lib.dptr(Wd[0]), _lib.dptr(Wd[1]), _lib.dptr(Wd[2]), _lib.dptr(Od),
                                         None, None, None, stream))
    fwd_ms = {}
    try:
        for which, nme in ((1, 'slab (mma.sync 3xTF32)'), (3, 'tcgen05 tiles (TMEM operand, 3xTF32)')):
            L.scone_set_dense_kernel(which)
            fwd_ms[nme] = t_of(fwd)
            if which == 3:
                _lib.check(L.scone_umma_status(stream), 'scone_umma_status')
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    best = min(fwd_ms, key=fwd_ms.get)
    f_ms = fwd_ms[best]
    def bwd():
        _lib.check(L.scone_layer_backward(cx.handle, 0, bd, C, C, _lib.dptr(Hd), _lib.dptr(Od), _lib.dptr(Wd[0]), _lib.dptr(Wd[1]), _lib.dptr(Wd[2]),
                                          _lib.dptr(Od), _lib.dptr(dWd), 0, _lib.dptr(wsd), None, None, None, None, stream))
    bwd_ms = {}
    try:
        for which, nme in ((1, 'fp32 SIMT tile kernel'), (3, 'tcgen05 (weight gradient accumulated in TMEM, 3xTF32)')):
            L.scone_set_dense_kernel(which)
            bwd_ms[nme] = t_of(bwd)
            if which == 3:
                _lib.check(L.scone_umma_status(stream), 'scone_umma_status')
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    best_b = min(bwd_ms, key=bwd_ms.get)
    b_ms = bwd_ms[best_b]
    fa, ba = 4.0 * E * bd * 2 * C / f_ms / 1e6, 4.0 * E * bd * 3 * C / b_ms / 1e6
    del Hd, Od
    return {'bound': 'hbm', 'unit': 'GB/s', 'peak': peak, 'b': bd, 'tensor_bytes': 4.0 * E * bd * C,
            'layer_fwd': {'kernel': best, 'ms': f_ms, 'achieved': fa, 'frac': fa / peak, 'algorithmic_bytes': 4.0 * E * bd * 2 * C,
                          'all_kernels_ms': fwd_ms,
                          'traffic': ncu_traffic('layer_fwd_umma_kernel', 'dense_umma_r2j') if 'tcgen05' in best else
                          ncu_traffic('layer_fwd_slab_kernel', 'dense_slab_r2i')},
            'layer_bwd': {'kernel': best_b, 'ms': b_ms, 'achieved': ba, 'frac': ba / peak, 'algorithmic_bytes': 4.0 * E * bd * 3 * C,
                          'all_kernels_ms': bwd_ms, 'traffic': ncu_traffic('layer_bwd_umma_kernel', 'dense_bwd_umma_r2w')},
            'l2_policy': 'tensors of %.1f GB each: larger than L2' % (4.0 * E * bd * C / 1e9),
            'note': 'one fused 32->32 layer on dense random features [E][64][32], every row computed (no flags / pruning), best of 3, CUDA '
                    'events.  All kernels share the gather (13 neighbour rows per output row): what binds is the L1 / shared-memory data '
                    'pipe the gathered rows come through (backward kernel: 83 % of its peak, tensor pipe 33 %, DRAM 19 %; forward: 47-73 %), '
                    'not HBM and not the tensor cores (profiles/prof_dense_*_r2*, DESIGN.md 4.2)'}


def bench_bunch(args, cfg, sp, ds, hp, h2d_bytes, B, gb, world, rank, dev, stream, t_setup):
    """cfg3 / -model bunch: the SCCONV model has host-pointer entry points only; value == e2e (pinned host buffers, copies inside)."""
    import numpy as np
    import torch
    import scone_gcn_b200 as sg
    from scone_gcn_b200.bunch import BunchModel, CsrOperator
    from scone_gcn_b200.bunch_model_matrices import compute_shift_matrices
    L = sg.lib()
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    shifts = [CsrOperator(M) for M in compute_shift_matrices(ds.B1, ds.B2)]
    net = BunchModel(shifts, np.array(cx.nbrhoods), [cfg['hidden']] * 3, micro_batch=min(B, 1024))
    rs = np.random.RandomState(1030)
    net.set_weights([0.01 * rs.randn(*s) for s in net.shapes])
    step_no = [0]

    def step():
        net.loss_grad(hp['ptr'], hp['edge'], hp['val'], hp['last'], hp['tgt'], hp['mask'], zero_first=True, stream=stream, read=False)
        net.adam_step(step_no[0], 1e-3, 5e-5, stream)
        step_no[0] += 1
        buf = net.read_grads(stream)
        return float(buf[-2] / buf[-1])
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    clocks = ClockSampler(int(os.environ.get('LOCAL_RANK', '0')))
    clocks.start()
    launches0 = L.scone_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    loss = None
    for _ in range(args.steps):
        loss = step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, net.read_grads(stream), net.flatten(net.get_weights()))
    value = B * args.steps / (ms / 1e3)
    peak, peak_src = load_peaks()
    out = {'metric': 'SCoNe train trajectories/sec', 'value': value, 'unit': 'trajectories/s', 'n_gpus': world, 'steps': args.steps,
           'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
           'dtype': 'f32', 'data': 'synthetic',
           'config': {'workload': args.config + ': ' + cfg['desc'], 'N': cx.N, 'E': cx.E, 'F': cx.F, 'D': cx.D, 'model': 'bunch',
                      'global_batch': B, 'hidden': cfg['hidden'], 'layers': 4, 'l2_policy': 'dense [rows][batch][C] tensors of %.0f MB each, ~30 of them per step: larger than L2' % (4e-6 * cx.E * min(B, 1024) * cfg['hidden'])},
           'roofline': {'bound': 'hbm', 'kernel': 'bunch_level_fwd/bwd_kernel, outer_tile_spmm_kernel (generic CSR operators)', 'achieved': None, 'peak': peak, 'unit': 'GB/s', 'frac': None,
                        'traffic': None, 'peak_source': peak_src,
                        'note': 'the bunch model runs dense (no pruning) on generic CSR operators; no per-kernel byte model is reported'},
           'e2e': {'value': value, 'unit': 'trajectories/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': int(4 * (net.n_params + 2)),
                   'steps': args.steps, 'last_loss': loss, 'note': 'the bunch model only has host-pointer entry points: value == e2e'},
           'cpu_baseline': None, 'gpu_launches': int(L.scone_launch_count() - launches0), 'clocks': clk, 'setup_s': time.time() - t_setup}
    if rank == 0:
        print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
