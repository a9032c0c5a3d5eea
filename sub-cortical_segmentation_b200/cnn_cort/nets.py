"""build_model -- the three-branch CNN of the reference (``cnn_cort/nets.py:127-255``)
behind the nolearn ``NeuralNet`` duck type, running on hand-written sm_100a kernels.

    net = build_model(weights_path, options)
    net.fit({'in1': ax, 'in2': cor, 'in3': sag, 'in4': atlas}, y)
    net.predict_proba({'in1': ..., 'in2': ..., 'in3': ..., 'in4': ...})  -> float32 [N, 15]
    net.predict(...)                                                     -> int64   [N]

The graph (3 x [5 x (conv3x3 -> BatchNorm -> PReLU), pools after conv2/conv4, dropout,
dense 180 + PReLU] -> concat 540 -> FC1 540 -> concat atlas 15 -> fc_2 270 -> out 15
softmax), its parameter names and the on-disk weight format (``nets/<name>/<name>.pkl``:
OrderedDict{layer name -> [arrays]}, 88 keys) are the reference's; the committed
``nets/miccai2012_v1`` file loads unchanged.  All arithmetic happens in
``libsubcort_b200.so``; this file is host logic only (parameter packing, the nolearn
epoch loop, history, early stopping, checkpointing).
"""
import os
import pickle
import time
from collections import OrderedDict

import numpy as np

from . import _native
from . import parallel

BRANCHES = ('axial', 'coronal', 'saggital')   # reference spelling, nets.py:202
_CONV = ((1, 20), (20, 20), (20, 40), (40, 40), (40, 60))


def layer_table():
    """(layer name, [array shapes]) in the order nolearn's save_params_to writes them."""
    T = []
    for n, b in enumerate(BRANCHES, 1):
        T.append(('in%d' % n, []))
        for i, (ci, co) in enumerate(_CONV, 1):
            T.append(('%s_ch_conv%d' % (b, i), [(co, ci, 3, 3)]))
            T.append(('%s_ch_conv%d_bn' % (b, i), [(co,)] * 4))           # beta, gamma, mean, inv_std
            T.append(('%s_ch_conv%d_bn_nonlin' % (b, i), []))
            T.append(('%s_ch_prelu%d' % (b, i), [(co,)]))
            if i == 2:
                T.append(('%s_max_pool_1' % b, []))
            if i == 4:
                T.append(('%s_max_pool_2' % b, []))
        T.append(('%s_l1drop' % b, []))
        T.append(('%s_d1' % b, [(540, 180), (180,)]))
        T.append(('%s_prelu_d1' % b, [(180,)]))
    T += [('elem_channels', []), ('f1_drop', []), ('FC1', [(540, 540), (540,)]), ('prelu_f1', [(540,)]),
          ('f2_drop', []), ('in4', []), ('elem_channels2', []), ('fc_2', [(555, 270), (270,)]),
          ('prelu_f2', [(270,)]), ('out_layer', [(270, 15), (15,)])]
    return T


def _initial_params(seed=None):
    """What Lasagne would create: GlorotUniform W (gain 1), b = 0, PReLU alpha = .25,
    BN beta 0 / gamma 1 / mean 0 / inv_std 1."""
    rng = np.random.RandomState(seed)
    P = OrderedDict()
    for name, shapes in layer_table():
        arrs = []
        for k, s in enumerate(shapes):
            if name.endswith('_bn'):
                arrs.append(np.ones(s, np.float32) if k in (1, 3) else np.zeros(s, np.float32))
            elif 'prelu' in name:
                arrs.append(np.full(s, 0.25, np.float32))
            elif len(s) == 1:
                arrs.append(np.zeros(s, np.float32))
            else:
                if len(s) == 4:
                    fan_in, fan_out = s[1] * 9, s[0] * 9
                else:
                    fan_in, fan_out = s
                lim = np.sqrt(6.0 / (fan_in + fan_out))
                arrs.append(rng.uniform(-lim, lim, size=s).astype(np.float32))
        P[name] = arrs
    return P


def pack_params(P):
    """OrderedDict -> flat float32 blob in pickle order (the C-ABI's parameter layout)."""
    out = []
    for name, shapes in layer_table():
        arrs = P[name] if name in P else []      # parameter-less layers may be absent
        if len(arrs) != len(shapes):
            raise ValueError("layer %s: expected %d arrays, got %d" % (name, len(shapes), len(arrs)))
        for a, s in zip(arrs, shapes):
            a = np.asarray(a, dtype=np.float32)
            if a.shape != tuple(s):
                raise ValueError("layer %s: expected shape %s, got %s" % (name, s, a.shape))
            out.append(a.ravel())
    blob = np.concatenate(out)
    assert blob.size == _native.PARAM_FLOATS
    return blob


def unpack_params(blob):
    P = OrderedDict()
    o = 0
    for name, shapes in layer_table():
        arrs = []
        for s in shapes:
            n = int(np.prod(s))
            arrs.append(np.array(blob[o:o + n], dtype=np.float32).reshape(s))
            o += n
        P[name] = arrs
    return P


class TrainSplit(object):
    """nolearn.lasagne.TrainSplit(eval_size): the first fold of an unshuffled stratified
    K-fold (K = round(1/eval_size)) is the validation set."""

    def __init__(self, eval_size):
        self.eval_size = eval_size

    def indices(self, y):
        n = len(y)
        if not self.eval_size:
            return np.arange(n), np.arange(0)
        k = int(round(1.0 / self.eval_size))
        valid = np.zeros(n, bool)
        for c in np.unique(y):  # sklearn StratifiedKFold(shuffle=False): per-class contiguous folds
            idx = np.nonzero(y == c)[0]
            fold_sizes = np.full(k, len(idx) // k)
            fold_sizes[:len(idx) % k] += 1
            valid[idx[:fold_sizes[0]]] = True
        return np.nonzero(~valid)[0], np.nonzero(valid)[0]


class Net(object):
    """The object ``build_model`` returns (nolearn ``NeuralNet`` duck type)."""

    def __init__(self, options, weights_file, history_file, update_learning_rate=0.001, seed=None):
        self.options = options
        self.weights_file = weights_file
        self.history_file = history_file
        self.update_learning_rate = update_learning_rate
        self.max_epochs = int(options.get('max_epochs', 100))
        self.patience = int(options.get('patience', 20))
        self.verbose = int(options.get('net_verbose', 0))
        self.batch_size = int(options.get('batch_size', 128))
        self.train_split = TrainSplit(options.get('train_split', 0.25))
        self.train_history_ = []
        self._seed = seed
        self._ctx = None
        self._pending = None
        dev = options.get('device')
        if dev is None:
            from .load_options import device_index
            dev = device_index(options.get('mode', 'cuda0'))
        if dev is None:
            raise _native.NativeError(
                "mode=%r: this implementation has no CPU path (the reference's mode=cpu exists only "
                "as the oracle / CPU baseline); use mode=cudaN" % options.get('mode'))
        self.device = int(os.environ.get('LOCAL_RANK', dev)) if options.get('use_local_rank') else int(dev)

    # -- lifecycle ------------------------------------------------------------------------------
    def initialize(self):
        if self._ctx is None:
            import torch
            torch.cuda.set_device(self.device)
            self._ctx = _native.Context(self.device)
            P = self._pending if self._pending is not None else _initial_params(self._seed)
            self._ctx.load_weights(pack_params(P))
            self._pending = None
        return self

    @property
    def ctx(self):
        return self.initialize()._ctx

    # -- parameters -----------------------------------------------------------------------------
    def get_all_params_values(self):
        if self._ctx is None:
            return self._pending if self._pending is not None else _initial_params(self._seed)
        return unpack_params(self._ctx.get_params())

    def load_params_from(self, source):
        """nolearn semantics: match by layer name, copy array by array when shapes agree,
        ignore unknown names."""
        if isinstance(source, str):
            with open(source, 'rb') as f:
                source = pickle.load(f, encoding='latin1')
        P = self.get_all_params_values()
        for name, arrs in source.items():
            if name not in P:
                continue
            for k, a in enumerate(arrs):
                if k < len(P[name]) and tuple(np.shape(a)) == P[name][k].shape:
                    P[name][k] = np.asarray(a, dtype=np.float32)
        if self._ctx is None:
            self._pending = P
        else:
            self._ctx.load_weights(pack_params(P))

    def save_params_to(self, path):
        with open(path, 'wb') as f:
            pickle.dump(self.get_all_params_values(), f, protocol=2)

    # -- inference ------------------------------------------------------------------------------
    @staticmethod
    def _inputs(X):
        import torch
        xs = [X['in1'], X['in2'], X['in3'], X['in4']]
        if all(isinstance(x, torch.Tensor) and x.is_cuda for x in xs):
            return [x.contiguous().float() for x in xs], True
        return [np.ascontiguousarray(x, dtype=np.float32) for x in xs], False

    def predict_proba(self, X):
        xs, on_dev = self._inputs(X)
        if on_dev:
            return self.ctx.forward(*xs, want_label=False)[0]
        return self.ctx.forward_host(*xs, want_label=False)[0]

    def predict(self, X):
        xs, on_dev = self._inputs(X)
        if on_dev:
            return self.ctx.forward(*xs, want_proba=False)[1].long()
        return self.ctx.forward_host(*xs, want_proba=False)[1].astype(np.int64)

    # -- training (nolearn epoch loop: nets.py:233-246) ---------------------------------------
    def fit(self, X, y=None, epochs=None):
        """nolearn's fit on X = {'in1', 'in2', 'in3', 'in4'} arrays with labels y, or on a base.ScanTrainingSet (y
        omitted), whose minibatches are gathered on the device from the scans.  Same epoch loop either way."""
        import torch
        import torch.distributed as dist
        ctx = self.ctx
        dev = torch.device('cuda', self.device)
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        rank = dist.get_rank() if world > 1 else 0
        scans = hasattr(X, 'gather')
        if scans:
            if y is not None:
                raise ValueError("fit: a ScanTrainingSet carries its own labels; call fit(scans) without y")
            y = X.y
        else:
            y = np.asarray(y).astype(np.uint8)
        if y.size and int(y.max()) > 14:
            raise ValueError("fit: labels must be in 0..14 (generate_training_set maps the boundary label 15 to 0, base.py:89)")
        tr, va = self.train_split.indices(y)
        if not scans:
            xs = [np.ascontiguousarray(X[k], dtype=np.float32) for k in ('in1', 'in2', 'in3', 'in4')]
        if world > 1:
            # data parallel: every rank must hold the SAME training set in the same order (shard_batch strides through the
            # global minibatch) and start from the SAME parameters; neither is true by construction (the reference's
            # negative sampling and its weight initialisation are unseeded), so check the first and enforce the second
            if scans:
                parallel.assert_same_fingerprint(X.fingerprint, dev)
            else:
                parallel.assert_same_dataset(xs, y, dev)
            p = ctx.param_tensor()
            dist.broadcast(p, 0)
            ctx.load_weights(p.cpu().numpy())          # re-derives the inference layouts from the broadcast parameters
            ctx.reset_optimizer()
        # options['sync_bn'] = 'True': BatchNorm statistics over the GLOBAL batch like the single-device reference (30 tiny
        # all-reduces per step); default: per-GPU statistics, the usual data-parallel practice
        ctx.set_sync_bn(world > 1 and str(self.options.get('sync_bn', 'False')) == 'True')
        # options['fused_adam'] = 'True': the gradient all-reduce and the Adam update run as ONE kernel over NVLink peer memory
        # (sc_allreduce_adam_step) instead of NCCL all_reduce + sc_adam_step
        fused = world > 1 and str(self.options.get('fused_adam', 'False')) == 'True'
        if fused:
            ctx.fused_attach()
        batches = self._scan_batches(X, dev) if scans else self._array_batches(xs, y, dev)

        best_valid, best_train = np.inf, np.inf
        best_epoch, best_weights = 0, None
        first = len(self.train_history_)
        bs = self.batch_size
        n_epochs = epochs or self.max_epochs
        grads = ctx.grad_tensor()
        rng = np.random.RandomState(self._seed)
        loss_buf = torch.zeros(1, dtype=torch.float32, device=dev)
        steps = [tr[s:s + bs] for s in range(0, len(tr), bs)]
        local_steps = [parallel.shard_batch(gidx, rank, world) for gidx in steps]
        valid_steps = [va[s:s + bs] for s in range(0, len(va), bs)]
        for ep in range(first + 1, first + n_epochs + 1):
            t0 = time.time()
            losses, sizes = [], []
            for gidx, b in zip(steps, batches(local_steps)):
                if b is not None:
                    ctx.train_forward_backward(*b, n_global=len(gidx), seed=int(rng.randint(1 << 62)) + rank, loss_out=loss_buf)
                else:                      # a last partial batch smaller than the world size: contribute zeros
                    grads.zero_()
                    loss_buf.zero_()
                if fused:
                    ctx.allreduce_adam_step(lr=self.update_learning_rate)
                    if world > 1:
                        dist.all_reduce(loss_buf)
                else:
                    parallel.allreduce_gradients(grads, loss_buf)
                    # the BN-statistics slots hold the SUM of the batch statistics of the ranks that had samples: rank r of
                    # shard_batch has some iff r < len(gidx)
                    ctx.adam_step(lr=self.update_learning_rate, stat_scale=1.0 / min(world, len(gidx)))
                losses.append(loss_buf.clone())
                sizes.append(len(gidx))
            train_loss = float(np.average(torch.cat(losses).cpu().numpy(), weights=sizes)) if losses else float('nan')
            vsum = torch.zeros(2, dtype=torch.float32, device=dev)
            for b in batches(valid_steps):
                vsum += ctx.eval_batch(*b)
            vs = vsum.cpu().numpy()
            valid_loss = float(vs[0] / max(1, len(va)))
            valid_acc = float(vs[1] / max(1, len(va)))
            info = {'epoch': ep, 'train_loss': train_loss, 'valid_loss': valid_loss, 'valid_accuracy': valid_acc,
                    'train_loss_best': train_loss < best_train, 'valid_loss_best': valid_loss < best_valid,
                    'dur': time.time() - t0}
            best_train = min(best_train, train_loss)
            self.train_history_.append(info)
            if self.verbose:
                print("  %4d  train %.5f  valid %.5f  acc %.5f  %.2fs" % (ep, train_loss, valid_loss, valid_acc, info['dur']))
            # on_epoch_finished: SaveWeights(only_best), SaveTrainingHistory, EarlyStopping (nets.py:154-156)
            if valid_loss < best_valid or len(va) == 0:
                best_valid, best_epoch = valid_loss, ep
                best_weights = self.get_all_params_values()
                if rank == 0 and self.weights_file:
                    with open(self.weights_file, 'wb') as f:
                        pickle.dump(best_weights, f, protocol=2)
            if rank == 0 and self.history_file:
                with open(self.history_file, 'wb') as f:
                    pickle.dump(self.train_history_, f, protocol=2)
            if len(va) and best_epoch + self.patience < ep:
                if self.verbose:
                    print("Early stopping. Best valid loss was %.6f at epoch %d." % (best_valid, best_epoch))
                if best_weights is not None:
                    self.load_params_from(best_weights)
                break
        return self

    def _array_batches(self, xs, y, dev):
        """minibatch source of fit on host arrays: batches(index lists) yields the device tensors (in1..in4, y) of each
        list, None for an empty one"""
        import torch
        # the training set lives on the device when it fits (a minibatch is then one index_select per input instead of five
        # pageable host-to-device copies per step); otherwise minibatches are staged through page-locked buffers
        nbytes = sum(a.nbytes for a in xs) + y.nbytes
        free_b = torch.cuda.mem_get_info(dev)[0]
        resident = nbytes < 0.5 * free_b
        if resident:
            d_xs = [torch.from_numpy(a).to(dev) for a in xs]
            d_y = torch.from_numpy(y).to(dev)

            def to_dev(idx):
                di = torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int64)).to(dev)
                return [a.index_select(0, di) for a in d_xs] + [d_y.index_select(0, di)]
        else:
            stage = {}

            def to_dev(idx):
                out = []
                for k, a in enumerate(xs + [y]):
                    need = (len(idx),) + a.shape[1:]
                    buf = stage.get(k)
                    if buf is None or buf.shape[0] < len(idx):
                        buf = torch.empty((max(len(idx), self.batch_size),) + a.shape[1:], dtype=torch.from_numpy(a[:1]).dtype, pin_memory=True)
                        stage[k] = buf
                    np.take(a, idx, axis=0, out=buf.numpy()[:len(idx)])
                    out.append(buf[:len(idx)].to(dev, non_blocking=True))
                torch.cuda.current_stream().synchronize()      # the staging buffers are reused by the next minibatch
                return out

        def batches(index_lists):
            for idx in index_lists:
                yield to_dev(idx) if len(idx) else None
        return batches

    def _scan_batches(self, scans, dev):
        """minibatch source of fit on a ScanTrainingSet: one upload of all row indices of a pass (an epoch's training or
        validation minibatches); every minibatch is then gathered from the scans on the device (sc_gather_samples, on
        this net's context) out of a slice of that upload -- no host synchronise per step"""
        import torch
        ctx = self.ctx

        def batches(index_lists):
            flat = np.concatenate([np.asarray(i, dtype=np.int64) for i in index_lists]) if index_lists else np.zeros(0, np.int64)
            if flat.size and (flat.min() < 0 or flat.max() >= len(scans)):
                raise IndexError("fit: row index out of range [0, %d)" % len(scans))
            d_idx = torch.from_numpy(flat).to(dev)
            off = 0
            for idx in index_lists:
                yield scans.gather(d_idx[off:off + len(idx)], ctx=ctx) if len(idx) else None
                off += len(idx)
        return batches


def build_model(weights_path, options):
    """Build the CNN model and return the net object (reference: nets.py:127-255).

    - weights_path: folder holding ``<experiment>/<experiment>.pkl``
    - options: dict from ``load_options``; used keys: experiment, patch_size, net_verbose,
      train_split, max_epochs, patience, batch_size, load_weights, mode
    """
    name = options['experiment']
    try:
        os.mkdir(os.path.join(weights_path, name))
    except OSError:
        pass
    net_weights = os.path.join(weights_path, name, name + '.pkl')
    net_history = os.path.join(weights_path, name, name + '_history.pkl')
    ps = options['patch_size'][0]
    if ps != 32:
        raise ValueError("patch_size=%d: the kernels (and the committed weights: flatten 540) are built for 32" % ps)
    net = Net(options, net_weights, net_history, update_learning_rate=0.001, seed=options.get('seed'))
    if options['load_weights'] == 'True':
        print("    --> loading weights from ", net_weights)
        if os.path.exists(net_weights):
            net.load_params_from(net_weights)
        else:
            # reference swallows the failure and keeps the random init (nets.py:249-253)
            print("    --> WARNING: %s not found, keeping the random initialisation" % net_weights)
    return net
