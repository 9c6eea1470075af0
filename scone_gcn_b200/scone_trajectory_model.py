"""Scone_GCN — host-side mirror of the reference trainer (trajectory_analysis/scone_trajectory_model.py).

Same constructor, methods, argument meaning, printed lines and NumPy RNG stream as the reference class
(:17-368); the arithmetic (vmap'd model, grad(loss), adam) runs in the CUDA library instead of JAX:

  reference                                              here
  self.model = vmap(model, in_axes)            :256  ->  batched op over device-resident index arrays
  grad(self.loss)(weights, inputs, y, mask)    :307  ->  SconeModel.loss_grad (fused fwd+bwd kernels); a y that is not
                                                         one-hot: SconeModel.vjp with cot = -mask * y
  adam(step_size) init/update/get_params       :300  ->  SconeModel.adam_step (device Adam state)

Differences that are deliberate and results-identical:
  * loss/grad only run the masked trajectories (the reference forwards all N and boolean-selects, :46 — Q4);
    `forward_all=True` restores the reference's work for timing comparisons.
  * the four per-epoch metric evaluations share one forward pass (:328-331).
  * nets with fewer than 3 layers train (the reference crashes at :278,:308 — Q5).
"""
import numpy as onp

from . import dp
from .complex import flows_to_csr
from .model import SconeModel
from .bunch import BunchModel

onp.random.seed(1030)          # scone_trajectory_model.py:15 — weight init and batch masks draw from this stream


class _Prepared:
    """Sparse (CSR) view of inputs = [Bconds_func | nbrhoods, last_nodes, X] cached per X array."""

    def __init__(self, inputs):
        X = inputs[-1]
        self.last_nodes = onp.ascontiguousarray(onp.asarray(inputs[1]).astype(onp.int32))
        if isinstance(X, tuple) and len(X) == 3:          # already sparse: (traj_ptr, flow_edge, flow_val)
            self.ptr, self.edge, self.val = [onp.ascontiguousarray(a) for a in X]
        else:
            self.ptr, self.edge, self.val = flows_to_csr(onp.asarray(X))
        self.n = len(self.ptr) - 1

    def select(self, rows):
        rows = onp.asarray(rows)
        lens = (self.ptr[rows + 1] - self.ptr[rows]).astype(onp.int64)
        ptr = onp.zeros(len(rows) + 1, onp.int32)
        onp.cumsum(lens, out=ptr[1:])
        idx = onp.repeat(self.ptr[rows].astype(onp.int64) - ptr[:-1], lens) + onp.arange(int(ptr[-1]))
        return ptr, self.edge[idx], self.val[idx], self.last_nodes[rows]


class Scone_GCN():
    def __init__(self, epochs, step_size, batch_size, weight_decay, verbose=True, micro_batch=None, forward_all=False,
                 data_parallel=None):
        """
        :param epochs: # of training epochs
        :param step_size: step size for use in training model
        :param batch_size: # of data points to train over in each gradient step
        :param verbose: whether to print training progress
        :param weight_decay: ridge regularization constant
        (micro_batch / forward_all / data_parallel: B200-side knobs, not in the reference.  data_parallel=None: on when a
         torch.distributed process group with more than one rank exists — every rank runs the same script with the same RNG
         stream, computes the gradient of its contiguous share of each batch, and the flat [grads | nll | count] buffer is
         summed over ranks and the replicated Adam step applied by one kernel over NVLink peer memory (dp.PeerExchange;
         SCONE_DP_EXCHANGE=nccl: NCCL all-reduce + Adam kernel): SURVEY 8(e))
        """
        self.random_targets = None
        self.trained = False
        self.model = None
        self.model_single = None
        self.shifts = None
        self.weights = None
        self.epochs = int(epochs)
        self.step_size = step_size
        self.batch_size = int(batch_size)
        self.weight_decay = weight_decay
        self.verbose = verbose
        self.micro_batch = micro_batch
        self.forward_all = forward_all
        self.data_parallel = data_parallel
        self._net = None
        self._prep_cache = {}

    # ---- plumbing -----------------------------------------------------------------------------------
    def _prepared(self, inputs):
        key = id(inputs[-1])
        hit = self._prep_cache.get(key)
        if hit is None or hit[0] is not inputs[-1] or len(hit[1].last_nodes) != len(inputs[1]) \
                or not onp.array_equal(hit[1].last_nodes, onp.asarray(inputs[1]).astype(onp.int32)):
            hit = (inputs[-1], _Prepared(inputs))
            self._prep_cache[key] = hit
        return hit[1]

    def _push(self, weights):
        self._net.set_weights([onp.asarray(w) for w in weights], reset_adam=False)

    def _forward(self, weights, inputs, rows=None):
        """log-probs [n, D, 1] float32 for the selected trajectories (all if rows is None)."""
        p = self._prepared(inputs)
        self._push(weights)
        if rows is None:
            lp = self._net.forward(p.ptr, p.edge, p.val, p.last_nodes)
        else:
            lp = self._net.forward(*p.select(rows))
        return lp[:, :, None]

    def _ridge(self, weights):
        # np.linalg.norm over the three stacked groups (:52-56) == sum of squared Frobenius norms
        return self.weight_decay * float(sum((onp.asarray(w, onp.float64) ** 2).sum() for w in weights))

    # ---- reference API ------------------------------------------------------------------------------
    def loss(self, weights, inputs, y, mask):
        """
        Computes cross-entropy loss per flow                              (scone_trajectory_model.py:42-56)
        """
        mask = onp.asarray(mask)
        rows = onp.nonzero(mask == 1)[0]
        yv = onp.asarray(y)
        if hasattr(self._net, 'evaluate') and not self.forward_all and self._is_onehot(yv):
            # forward + masked NLL sum on the device (fixed summation order); only two floats come back
            p = self._prepared(inputs)
            self._push(weights)
            tgt = onp.argmax(yv.reshape(yv.shape[0], -1)[rows], axis=1)
            nll, cnt = self._net.evaluate(*p.select(rows), target_idx=tgt, mask=onp.ones(len(rows), onp.float32), want_nll=True)['nll']
            return onp.float32(nll / onp.sum(mask) + self._ridge(weights))
        if self.forward_all:
            preds = self._forward(weights, inputs)[rows]
        else:
            preds = self._forward(weights, inputs, rows)
        return onp.float32(-onp.sum(preds.astype(onp.float64) * yv[rows]) / onp.sum(mask) + self._ridge(weights))

    @staticmethod
    def _is_onehot(yv):
        flat = yv.reshape(yv.shape[0], -1)
        return bool(onp.all((flat == 0) | (flat == 1)) and onp.all(flat.sum(axis=1) == 1))

    def accuracy(self, shifts, inputs, y, mask, n_nbrs):
        """
        Computes ratio of correct predictions                             (scone_trajectory_model.py:59-71)
        """
        mask = onp.asarray(mask)
        if hasattr(self._net, 'accuracy') and not self.forward_all:
            # forward + mask-to--100 + argmax + compare on the device; only two integers come back.  Only the masked
            # trajectories are run (the same numbers as forwarding all of them and selecting, quirk Q4).
            rows = onp.nonzero(mask == 1)[0]
            p = self._prepared(inputs)
            self._push(self.weights)
            yv = onp.asarray(y)
            tgt = onp.argmax(yv.reshape(yv.shape[0], -1)[rows], axis=1)
            correct, counted = self._net.accuracy(*p.select(rows), onp.asarray(n_nbrs)[rows], tgt, onp.ones(len(rows), onp.float32))
            return onp.float64(correct) / onp.float64(counted) if counted else onp.float64('nan')
        target_choice = onp.argmax(onp.asarray(y)[mask == 1], axis=1)
        preds = onp.array(self._forward(self.weights, inputs))
        return self._accuracy_from(preds, target_choice, mask, n_nbrs)

    @staticmethod
    def _accuracy_from(preds, target_choice, mask, n_nbrs):
        preds = onp.array(preds)
        n_nbrs = onp.asarray(n_nbrs)
        cols = onp.arange(preds.shape[1])[None, :, None]
        preds[onp.broadcast_to(cols >= n_nbrs[:, None, None], preds.shape)] = -100   # preds[i, n_nbrs[i]:] = -100
        pred_choice = onp.argmax(preds[mask == 1], axis=1)
        return onp.mean(pred_choice == target_choice)

    def two_target_accuracy(self, shifts, inputs, y, mask, n_nbrs):
        """
        Ratio of the time the model ranks the true target above a random, different target (:73-108).

        The ranking runs on the device: the forward's log-probs stay there, the argmax predictions come back (N ints), the redraw
        loop of :89-91 runs on the host because it consumes the global NumPy RNG stream, and the true-vs-random comparison goes
        back to the device (two integer counts return).
        """
        mask = onp.asarray(mask)
        n_nbrs = onp.asarray(n_nbrs)
        N = onp.asarray(inputs[1]).shape[0]
        if type(self.random_targets) != onp.ndarray:
            self.random_targets = onp.random.randint(0, high=n_nbrs, size=N)
        yv = onp.asarray(y)
        true_choice = onp.argmax(yv, axis=1).reshape((yv.shape[0],))
        on_device = hasattr(self._net, 'evaluate')
        if on_device:
            p = self._prepared(inputs)
            self._push(self.weights)
            choice_all = self._net.evaluate(p.ptr, p.edge, p.val, p.last_nodes, n_nbrs=n_nbrs, mask=(mask == 1).astype(onp.float32),
                                            want_choice=True)['choice']
            pred_choice = choice_all[mask == 1]
        else:
            preds = onp.array(self._forward(self.weights, inputs))
            for i in range(len(preds)):
                preds[i, n_nbrs[i]:] = -100
            pred_choice = onp.argmax(preds[mask == 1], axis=1)
        # Faithful to :89-91: the loop runs over ALL N rows and pairs row i with the i-th MASKED prediction; in the reference
        # pred_choice is a jax array, whose out-of-range index clamps to the last element (no IndexError).
        last = len(pred_choice) - 1
        for i in range(N):
            pc = pred_choice[min(i, last)] if last >= 0 else -1
            while self.random_targets[i] == pc:
                self.random_targets[i] = onp.random.randint(0, high=n_nbrs[i])
        if on_device:
            gt, eq = self._net.two_target_counts(true_choice, self.random_targets)
            return (gt + 0.5 * eq) / sum(mask)
        all_row_idxs = range(len(self.random_targets))
        random_probs = preds[all_row_idxs, self.random_targets]
        true_probs = preds[all_row_idxs, true_choice]
        correct = 0
        for t, r in zip(true_probs[mask == 1], random_probs[mask == 1]):
            if t > r:
                correct += 1
            elif t == r:
                correct += 0.5
        return correct / sum(mask)

    def generate_weights(self, in_channels, hidden_layers, out_channels):
        """
        Same shapes, order and RNG draws as scone_trajectory_model.py:215-242.
        """
        weight_shapes = []
        if len(hidden_layers) > 0:
            weight_shapes += [(in_channels, hidden_layers[0][1])] * hidden_layers[0][0]
            for i in range(len(hidden_layers) - 1):
                for _ in range(hidden_layers[i + 1][0]):
                    weight_shapes += [(hidden_layers[i][1], hidden_layers[i + 1][1])]
            if self.model_type == 'bunch':
                weight_shapes += [(hidden_layers[-1][1], out_channels)] * hidden_layers[-1][0]
            else:
                weight_shapes += [(hidden_layers[-1][1], out_channels)]
            self.weights = []
            for s in weight_shapes:
                self.weights.append(0.01 * onp.random.randn(*s))
        else:
            self.weights = [(in_channels, out_channels)]
        print('# of parameters: {}'.format(onp.sum([onp.prod(w) for w in weight_shapes])))

    def setup(self, model, hidden_layers, shifts, inputs, y, in_axes, train_mask, model_type='scone'):
        """
        Set up model for training / calling                               (scone_trajectory_model.py:245-262)

        `shifts` are the ShiftHandle objects data_setup returns (they carry the device-resident complex);
        `model` is scone_func / ebli_func from scone_gcn_b200.trajectory_experiments.
        """
        self.model_type = model_type
        if model_type == 'bunch':
            return self._setup_bunch(model, hidden_layers, shifts, inputs, y)
        cx = getattr(shifts[0], 'complex', None) or getattr(inputs[0], 'complex', None)
        if cx is None:
            raise TypeError('setup() needs the shift handles / Bconds returned by scone_gcn_b200.trajectory_experiments.'
                            'data_setup (dense E x E shift matrices do not carry the incidence structure)')
        for k, _ in hidden_layers:
            if k != 3:
                raise AssertionError('wrong number of weights')       # trajectory_experiments.py:142,160
        self.shifts = shifts
        self._cx = cx.with_model(model_type)
        n = len(onp.asarray(inputs[1]))
        widths = [h[1] for h in hidden_layers]
        # widths 16 / 32 run on the compact row-list pipeline (memory follows the trajectories' support): thousands of
        # trajectories per micro-batch; other widths keep dense [E][micro_batch][C] tensors resident
        cap = 4096 if all(w in (16, 32) for w in widths) and self._cx.E * 4096 < 2 ** 32 else 256
        mb = self.micro_batch or min(max(n, 1), cap)
        self._net = SconeModel(self._cx, widths, micro_batch=mb)
        if self.micro_batch is None and mb > 512 and self._net.pipeline in (1, 2):
            # complexes the cone pipelines cannot take (max degree > 32) run on whole-support row lists: ~8000 rows per
            # trajectory against list capacities of 6 M / 32 M rows -> smaller micro-batches instead of error code 4
            self._net = None
            self._net = SconeModel(self._cx, widths, micro_batch=512)
        self.model_single = model

        def batched(weights, *args):
            ins = args[len(self.shifts):]
            return self._forward(weights, list(ins))
        batched.__name__ = getattr(model, '__name__', 'model')
        self.model = batched

        X = inputs[-1]
        in_channels = 1 if isinstance(X, tuple) else onp.asarray(X).shape[-1]
        out_channels = onp.asarray(y).shape[-1]
        assert in_channels == 1 and out_channels == 1, 'the SCoNe path is defined for scalar flows / one-hot targets'
        self.generate_weights(in_channels, hidden_layers, out_channels)

    def _setup_bunch(self, model, hidden_layers, shifts, inputs, y):
        """-model bunch: 7 weighted CSR operators, inputs[0] is the padded neighbour table (trajectory_experiments.py:309)."""
        for k, _ in hidden_layers:
            if k != 7:
                raise AssertionError('wrong number of weights')       # trajectory_experiments.py:178
        if len(shifts) != 7 or not all(hasattr(s, 'handle') for s in shifts):
            raise TypeError('setup(model_type="bunch") needs the 7 CsrOperator shifts returned by data_setup')
        self.shifts = shifts
        n = len(onp.asarray(inputs[1]))
        mb = self.micro_batch or min(max(n, 1), 1024)
        self._net = BunchModel(shifts, onp.asarray(inputs[0]), [h[1] for h in hidden_layers], micro_batch=mb)
        self.model_single = model

        def batched(weights, *args):
            return self._forward(weights, list(args[len(self.shifts):]))
        batched.__name__ = getattr(model, '__name__', 'model')
        self.model = batched
        self.generate_weights(1, hidden_layers, onp.asarray(y).shape[-1])

    def train(self, inputs, y, train_mask, test_mask, n_nbrs):
        """
        Trains the batched model; same step count, batch-mask stream and Adam as scone_trajectory_model.py:264-357.
        """
        train_mask, test_mask = onp.asarray(train_mask), onp.asarray(test_mask)
        p = self._prepared(inputs)
        N = p.n
        n_train_samples = sum(train_mask)
        n_batches = n_train_samples // self.batch_size
        yv = onp.asarray(y)
        target_idx = onp.argmax(yv.reshape(N, -1), axis=1).astype(onp.int32)
        # a soft target (not one-hot) is trained through the VJP of the log-probs with cot = -mask * y, the gradient of
        # -sum(preds * y) that jax.grad takes at :307; one-hot targets keep the loss_grad path
        soft = not self._is_onehot(yv)
        y_flat = onp.ascontiguousarray(yv.reshape(N, -1), onp.float32) if soft else None

        self._net.set_weights([onp.asarray(w) for w in self.weights], reset_adam=True)     # init_fun(self.weights)
        # the batches of every epoch are drawn from the same N trajectories: their plans (receptive cone, live rows, gather
        # programs — weight-independent) are built once; each step then runs only the compute kernel on the rows of its batch
        planned = bool(getattr(self._net, 'plan', None)) and not self.forward_all and self._net.plan(p.ptr, p.edge, p.val, p.last_nodes)
        self.adam_state = self._net
        use_dp = dp.is_distributed() if self.data_parallel is None else bool(self.data_parallel)
        if use_dp and not hasattr(self._net, 'grads_tensor'):
            raise NotImplementedError('data-parallel training is implemented for -model scone / ebli')
        exchange = None
        if use_dp and dp.is_distributed():                 # NVLink peer-memory exchange fused with Adam (None: NCCL all-reduce + Adam)
            import torch
            if torch.cuda.is_available():
                exchange = dp.make_exchange(self._net.n_params + 2, torch.device('cuda', torch.cuda.current_device()))
        unshuffled_batch_mask = onp.array([1] * self.batch_size + [0] * (N - self.batch_size))
        train_loss = train_acc = test_loss = test_acc = None

        for i in range(self.epochs * n_batches):
            batch_mask = onp.array(unshuffled_batch_mask)
            onp.random.shuffle(batch_mask)
            batch_mask = onp.logical_and(batch_mask, train_mask)
            if self.forward_all:
                rows = onp.arange(N)
                m = batch_mask.astype(onp.float32)
            else:
                rows = onp.nonzero(batch_mask)[0]
                m = onp.ones(len(rows), onp.float32)
            if use_dp:                                     # this rank's contiguous share of the batch (same rows on every rank)
                keep = dp.shard_rows(onp.arange(len(rows)))
                rows, m = rows[keep], m[keep]
            if soft:
                cot = -m[:, None] * y_flat[rows]
                if planned:
                    self._net.vjp_planned(rows, cot, m.sum(), zero_first=True, read=False)
                else:
                    self._net.vjp(*p.select(rows), cot, m.sum(), zero_first=True, read=False)
            elif planned:
                self._net.loss_grad_planned(rows, target_idx[rows], m, zero_first=True, read=False)
            else:
                ptr, fe, fv, last = p.select(rows)
                self._net.loss_grad(ptr, fe, fv, last, target_idx[rows], m, zero_first=True, read=False)
            if exchange is not None:                       # the one exchange of the step ([grads | nll_sum | count] summed over ranks)
                exchange.adam_step(self._net, i, self.step_size, self.weight_decay)      # + Adam, one kernel over NVLink peer memory
            else:
                if use_dp:
                    dp.allreduce_sum_(self._net.grads_tensor())
                self._net.adam_step(i, self.step_size, self.weight_decay)

            if i % n_batches == n_batches - 1:
                if exchange is not None:
                    exchange.status()                      # a rank that never delivered its gradients (time-out) is an error, not a hang
                self.weights = self._net.get_weights()
                preds = self._net.forward_planned()[:, :, None] if planned else self._forward(self.weights, inputs)
                ridge = self._ridge(self.weights)

                def _loss(mask):
                    return -onp.sum(preds[mask == 1].astype(onp.float64) * yv[mask == 1]) / onp.sum(mask) + ridge
                train_loss, test_loss = _loss(train_mask), _loss(test_mask)
                tc = onp.argmax(yv, axis=1)
                train_acc = self._accuracy_from(preds, tc[train_mask == 1], train_mask, n_nbrs)
                test_acc = self._accuracy_from(preds, tc[test_mask == 1], test_mask, n_nbrs)
                if self.verbose:
                    print('Epoch {} -- train loss: {:.6f} -- train acc {:.3f} -- test loss {:.6f} -- test acc {:.3f}'
                          .format(i // n_batches, train_loss, train_acc, test_loss, test_acc))
        self.weights = self._net.get_weights()
        self.trained = True
        if self.verbose:
            print("Epochs: {}, learning rate: {}, batch size: {}, model: {}".format(
                self.epochs, self.step_size, self.batch_size, self.model.__name__))
        return train_loss, train_acc, test_loss, test_acc

    def test(self, test_inputs, y, test_mask, n_nbrs):
        """
        Return the loss and accuracy for the given inputs                 (scone_trajectory_model.py:359-368)
        """
        loss = self.loss(self.weights, test_inputs, y, test_mask)
        acc = self.accuracy(self.shifts, test_inputs, y, test_mask, n_nbrs)
        if self.verbose:
            print("Test loss: {:.6f}, Test acc: {:.3f}".format(loss, acc))
        return loss, acc
