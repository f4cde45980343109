"""GraphedTrainStep: the reference's per-minibatch train step (reg_task.py:62-73 / class_task.py:69-79 /
bandits.py:43-51: zero_grad + sample_elbo[_lr] + backward + optimiser step) captured ONCE into a CUDA graph
and replayed, so a step costs one graph launch instead of ~40 host-side kernel launches.

What makes the captured step replayable:
  * eps comes from Philox keyed by a DEVICE step counter (bbb_rng.step_dev) that the graph itself advances,
    so every replay draws fresh, reproducible noise;
  * beta (the per-minibatch KL weight, reg_task.py:63) is read from a device scalar;
  * the optimiser is FusedAdam (one launch, step counter on the device) or a capturable torch optimiser;
  * inputs live in static device buffers that __call__ refills (from pinned host memory if given host tensors).
"""
import torch

from . import _lib as L
from . import rng as R
from . import parallel


class GraphedTrainStep:
    def __init__(self, net, optimizer, x, y, samples, sigma=1.0, beta=1.0, world_size=1, warmup=3, fuse_optimizer=False):
        # The optimiser's update applied inside the backward kernels (in their gradient write-back, or overlapped on a
        # side stream) measured slower than, or no faster than, the stand-alone multi-tensor Adam launch; it was
        # removed (DESIGN.md §4.6).  The keyword stays so that callers which pass fuse_optimizer=False keep working.
        if fuse_optimizer:
            raise ValueError('fuse_optimizer: the optimiser fused into the backward was removed (DESIGN.md §4.6); '
                             'the step runs the backward, then one FusedAdam launch')
        L.require_cuda(x, y)
        self.net, self.opt, self.samples, self.sigma, self.world = net, optimizer, samples, sigma, world_size
        self.x, self.y = x.clone(), y.clone()
        dev = x.device
        self.beta = torch.full((1,), float(beta), dtype=torch.float32, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int32, device=dev)      # read as uint32 by the kernels
        # d loss / d loss, allocated once: loss.backward() would launch a ones_like fill between the head's forward
        # and backward kernels in every step, which also breaks their programmatic-dependent-launch chain
        self._one = torch.ones(1, dtype=torch.float32, device=dev)
        self._elbo = net.sample_elbo_lr if net.local_reparam else net.sample_elbo
        # an optimiser that exchanges the gradients itself (PeerShardedAdam) needs no all-reduce around the backward
        self._ar = parallel.OverlappedAllReduce(1 if getattr(optimizer, 'reduces_gradients', False) else world_size)
        if hasattr(optimizer, 'use_device_step'):
            optimizer.use_device_step(self.counter)
        # Learning-rate schedulers (reg_task.py:53-54 / class_task.py:60-61: StepLR) change param_groups[...]['lr'] on the
        # host; the captured Adam launch has the initial lr baked in and multiplies it by this device scalar, which
        # __call__ refreshes whenever the host value has moved (one tiny fill, only on the steps where it changes)
        self._lr0 = float(optimizer.param_groups[0]['lr'])
        self._lr_seen = self._lr0
        self.lr_scale = None
        if hasattr(optimizer, 'lr_scale_dev') and self._lr0 > 0:
            self.lr_scale = torch.ones(1, dtype=torch.float32, device=dev)
            optimizer.lr_scale_dev = self.lr_scale
        # warm-up and capture must not train the model: snapshot parameters and optimiser state, restore after
        params = [p for g in optimizer.param_groups for p in g['params']]
        p_snap = [p.detach().clone() for p in params]
        s_snap = {id(t): t.clone() for st in optimizer.state.values() for t in st.values() if torch.is_tensor(t)}
        t_base = getattr(optimizer, '_t', 0)       # steps already taken eagerly: the captured launch continues from them
        R.use_device_step(self.counter)
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(warmup):
                    self._step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self.counter.zero_()
            if hasattr(optimizer, '_t'):
                optimizer._t = t_base            # the captured launch bakes host step t_base + 1; the device counter adds replays
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.loss_info = self._step()
        finally:
            R.use_device_step(None)
        with torch.no_grad():
            for p, snap in zip(params, p_snap):
                p.copy_(snap)
            for st in optimizer.state.values():
                for t in st.values():
                    if torch.is_tensor(t):
                        t.copy_(s_snap[id(t)]) if id(t) in s_snap else t.zero_()
        self.counter.zero_()
        if hasattr(optimizer, '_t'):
            optimizer._t = t_base
        torch.cuda.synchronize()

    def _step(self):
        self.net.zero_grad(set_to_none=True)
        with self._ar:
            info = self._elbo(self.x, self.y, self.beta, self.samples, sigma=self.sigma)
            info[0].backward(self._one)
        self._ar.join(self.net)
        self.opt.step()
        L.check(L.lib().bbb_counter_add(self.counter.data_ptr(), 1, L.stream()), 'bbb_counter_add')
        return info

    def __call__(self, x=None, y=None, beta=None):
        """Refill the static inputs (optional), replay the captured step, return the static loss tuple
        (device tensors, overwritten by the next replay)."""
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        if y is not None:
            self.y.copy_(y, non_blocking=True)
        if beta is not None:
            self.beta.fill_(float(beta))
        if self.lr_scale is not None:
            lr = float(self.opt.param_groups[0]['lr'])
            if lr != self._lr_seen:            # a scheduler stepped: every group moves by the same factor (StepLR)
                self._lr_seen = lr
                self.lr_scale.fill_(lr / self._lr0)
        self.graph.replay()
        return self.loss_info
