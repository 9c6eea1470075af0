"""Trajectories/s of the log-prob VJP (scone_model_vjp_dev, dense random cotangent) against the one-hot loss + gradient
(scone_model_loss_grad_dev) on bench.py's workload shape, inputs resident on the device, the two calls timed alternately with CUDA
events.  A report, not a gate.  Prints one JSON line with the GPU's name and power limit.  --flows times the VJP that also returns
the gradient with respect to the flow values (scone_model_vjp_flows_dev) against scone_model_vjp_dev instead.
    python tools/vjp_bench.py [--config cfg5] [--steps 20] [--warmup 5] [--rounds 3] [--flows]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench


def gpu_identity():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except Exception:
        return 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='cfg5', choices=['cfg5', 'cfg4', 'cfg1'])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--flows', action='store_true', help='vjp_flows_dev against vjp_dev')
    args = ap.parse_args()
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import _lib
    cfg = bench.CONFIGS[args.config]
    B = cfg['global_batch']
    sp, _ = bench.make_dataset(args.config, cfg, B, 1030)
    B = min(B, sp.n_traj)
    dev = torch.device('cuda')
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, cfg['model'])
    C = cfg['hidden']
    net = sg.SconeModel(cx, [C, C, C], micro_batch=B)
    rs = np.random.RandomState(1030)
    net.set_weights([0.01 * rs.randn(*s) for s in net.shapes])
    p1 = int(sp.traj_ptr[B])
    d = {k: torch.as_tensor(np.ascontiguousarray(v), device=dev) for k, v in dict(
        ptr=sp.traj_ptr[:B + 1].astype(np.int32), edge=sp.flow_edge[:p1].astype(np.int32), val=sp.flow_val[:p1].astype(np.float32),
        last=sp.last_nodes[:B].astype(np.int32), tgt=sp.target_idx[:B].astype(np.int32), mask=np.ones(B, np.float32),
        cot=rs.uniform(-0.25, 1.0, size=(B, cx.D)).astype(np.float32), dflow=np.zeros(p1, np.float32)).items()}
    stream = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()
    flows = [_lib.dptr(d[k]) for k in ('ptr', 'edge', 'val', 'last')]
    calls = {
        'loss_grad_dev': lambda: _lib.check(L.scone_model_loss_grad_dev(net.handle, B, *flows, _lib.dptr(d['tgt']), _lib.dptr(d['mask']), 1,
                                                                       stream), 'scone_model_loss_grad_dev'),
        'vjp_dev': lambda: _lib.check(L.scone_model_vjp_dev(net.handle, B, *flows, _lib.dptr(d['cot']), float(B), 1, stream),
                                      'scone_model_vjp_dev'),
    }
    if args.flows:
        del calls['loss_grad_dev']
        calls['vjp_flows_dev'] = lambda: _lib.check(L.scone_model_vjp_flows_dev(net.handle, B, *flows, _lib.dptr(d['cot']), float(B), 1,
                                                                                _lib.dptr(d['dflow']), stream), 'scone_model_vjp_flows_dev')
    for f in calls.values():
        for _ in range(args.warmup):
            f()
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    for _ in range(args.rounds):
        for name, f in calls.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.steps):
                f()
            b.record()
            b.synchronize()
            ms[name].append(a.elapsed_time(b) / args.steps)
    net.check_overflow()
    out = {'metric': 'trajectories/s per call (inputs on the device)', 'config': args.config, 'B': B, 'E': int(cx.E), 'D': int(cx.D),
           'pipeline': net.pipeline, 'gpu': gpu_identity(), 'steps': args.steps, 'rounds': args.rounds}
    for name, v in ms.items():
        out[name] = {'ms_per_call_median': float(np.median(v)), 'ms_per_call_rounds': [round(x, 4) for x in v],
                     'trajectories_per_s': B / (float(np.median(v)) * 1e-3)}
    if args.flows:
        out['vjp_flows_over_vjp_time'] = out['vjp_flows_dev']['ms_per_call_median'] / out['vjp_dev']['ms_per_call_median']
    else:
        out['vjp_over_loss_grad_time'] = out['vjp_dev']['ms_per_call_median'] / out['loss_grad_dev']['ms_per_call_median']
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
