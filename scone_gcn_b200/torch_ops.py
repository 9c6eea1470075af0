"""PyTorch autograd entry to the model's log-probs: any loss built on them trains through the library's VJP.

    lp = torch_ops.logprobs(net, w_flat, traj_ptr, flow_edge, flow_val, last_nodes)     # [B, D] float32
    loss = my_loss(lp)                                   # label smoothing, KL to a soft target, per-slot weights, ...
    loss.backward()                                      # w_flat.grad = dloss/dW through scone_model_vjp_dev

The forward runs scone_model_forward_dev and the backward scone_model_vjp_dev (which recomputes the forward inside the same
fused pass), both on the current torch stream.  When flow_val requires grad (a learned flow encoder, a trained per-edge mask or
scale, a saliency map over the edges of a path, an adversarial perturbation) the backward runs scone_model_vjp_flows_dev instead
and flow_val.grad receives dloss/dflow_val; the weight gradient is the same either way.  The op uses the model's own device
buffers: forward and backward each write w_flat into net.weights_tensor() first, and the backward overwrites the gradient buffer
net.grads_tensor() (zero_first); anything the caller keeps in those buffers across a call is replaced.  traj_ptr, flow_edge and
last_nodes are integer inputs and get no gradient."""
import torch

from . import _lib


def _check_inputs(net, w_flat, traj_ptr, flow_edge, flow_val, last_nodes):
    for name, t, dt in (('w_flat', w_flat, torch.float32), ('traj_ptr', traj_ptr, torch.int32), ('flow_edge', flow_edge, torch.int32),
                        ('flow_val', flow_val, torch.float32), ('last_nodes', last_nodes, torch.int32)):
        if not t.is_cuda or t.dtype != dt:
            raise TypeError('%s must be a CUDA %s tensor (got %s on %s)' % (name, dt, t.dtype, t.device))
    if w_flat.numel() != net.n_params:
        raise ValueError('w_flat has %d elements, the model %d parameters' % (w_flat.numel(), net.n_params))
    if traj_ptr.numel() != last_nodes.numel() + 1:
        raise ValueError('traj_ptr needs B + 1 = %d entries (got %d)' % (last_nodes.numel() + 1, traj_ptr.numel()))


class _LogProbs(torch.autograd.Function):
    @staticmethod
    def forward(ctx, w_flat, traj_ptr, flow_edge, flow_val, last_nodes, net):
        _check_inputs(net, w_flat, traj_ptr, flow_edge, flow_val, last_nodes)
        w_flat, traj_ptr, flow_edge, flow_val, last_nodes = [t.contiguous() for t in (w_flat, traj_ptr, flow_edge, flow_val, last_nodes)]
        B = last_nodes.numel()
        stream = torch.cuda.current_stream().cuda_stream
        net.weights_tensor().copy_(w_flat.detach())
        out = torch.empty((B, net.cx.D), dtype=torch.float32, device=w_flat.device)
        if B > 0:
            _lib.check(_lib.lib().scone_model_forward_dev(net.handle, B, _lib.dptr(traj_ptr), _lib.dptr(flow_edge), _lib.dptr(flow_val),
                                                          _lib.dptr(last_nodes), _lib.dptr(out), stream), 'scone_model_forward_dev')
        ctx.net = net
        ctx.save_for_backward(w_flat, traj_ptr, flow_edge, flow_val, last_nodes)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        w_flat, traj_ptr, flow_edge, flow_val, last_nodes = ctx.saved_tensors
        net = ctx.net
        B = last_nodes.numel()
        stream = torch.cuda.current_stream().cuda_stream
        want_flows = ctx.needs_input_grad[3]
        dflow = torch.zeros_like(flow_val) if want_flows else None      # (entries outside [traj_ptr[0], traj_ptr[B]) stay 0)
        if B == 0:
            return torch.zeros_like(w_flat), None, None, dflow, None, None
        cot = grad_out.to(torch.float32).contiguous()
        net.weights_tensor().copy_(w_flat)                 # the model's weights may have changed since the forward
        if want_flows:
            _lib.check(_lib.lib().scone_model_vjp_flows_dev(net.handle, B, _lib.dptr(traj_ptr), _lib.dptr(flow_edge), _lib.dptr(flow_val),
                                                            _lib.dptr(last_nodes), _lib.dptr(cot), 0.0, 1, _lib.dptr(dflow), stream),
                       'scone_model_vjp_flows_dev')
        else:
            _lib.check(_lib.lib().scone_model_vjp_dev(net.handle, B, _lib.dptr(traj_ptr), _lib.dptr(flow_edge), _lib.dptr(flow_val),
                                                      _lib.dptr(last_nodes), _lib.dptr(cot), 0.0, 1, stream), 'scone_model_vjp_dev')
        return net.grads_tensor()[:net.n_params].clone(), None, None, dflow, None, None


def logprobs(net, w_flat, traj_ptr, flow_edge, flow_val, last_nodes):
    """Differentiable log-probs [B, D] (float32) of a SconeModel at the flat weights w_flat (torch CUDA float32, net.n_params
    elements, list order of net.shapes) for B trajectories in sparse form (CUDA int32 traj_ptr [B + 1], flow_edge, int32
    last_nodes [B], float32 flow_val: scone_gcn_b200.flows_to_csr's layout, caller's edge ids).  Uses the model's weight and
    gradient buffers (module docstring)."""
    return _LogProbs.apply(w_flat, traj_ptr, flow_edge, flow_val, last_nodes, net)
