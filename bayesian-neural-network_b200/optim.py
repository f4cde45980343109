"""FusedAdam: torch.optim.Adam's update (same rule, same state names) for all parameter tensors in ONE
kernel launch (csrc/bbb_adam.cu, SURVEY 8f-1).  Opt-in: the reference's callers keep constructing
torch.optim.Adam; GraphedTrainStep and bench.py use this one because the stock foreach implementation costs
more than the whole fused forward+backward at the MNIST-shape config."""
import ctypes as C
import os
import weakref

import torch

from . import _lib as L


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        self.step_dev = None        # optional device uint32 counter added to the host step (CUDA-graph replay)
        self.lr_scale_dev = None    # optional device fp32 scalar multiplying lr (schedulers under a captured graph)
        self._t = 0

    def use_device_step(self, counter):
        self.step_dev = counter

    def _ensure_state(self, p):
        st = self.state[p]
        if not st:
            st['step'] = torch.tensor(0.0)
            st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return st

    def _mirror_step(self):
        """torch.optim.Adam keeps the step count in state[p]['step']: mirror ours there so a state_dict round trip
        (or handing the state to torch.optim.Adam) continues the bias correction instead of restarting it."""
        for st in self.state.values():
            if 'step' in st:
                st['step'].fill_(float(self._t))

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        steps = [float(st['step']) for st in self.state.values() if 'step' in st]
        self._t = int(max(steps)) if steps else 0

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self._t += 1
        for group in self.param_groups:
            ps = [p for p in group['params'] if p.grad is not None]
            for i in range(0, len(ps), 32):
                self._launch(group, ps[i:i + 32])
        self._mirror_step()
        return loss

    def _launch(self, group, ps):
        n = len(ps)
        if n == 0:
            return
        tabs = [(C.c_void_p * n)() for _ in range(4)]
        sizes = (C.c_int64 * n)()
        for i, p in enumerate(ps):
            st = self._ensure_state(p)
            L.require_cuda(p, p.grad)
            if not (p.is_contiguous() and p.grad.is_contiguous() and p.dtype == torch.float32):
                raise RuntimeError('FusedAdam needs contiguous fp32 parameters and gradients')
            tabs[0][i], tabs[1][i] = p.data_ptr(), p.grad.data_ptr()
            tabs[2][i], tabs[3][i] = st['exp_avg'].data_ptr(), st['exp_avg_sq'].data_ptr()
            sizes[i] = p.numel()
        b1, b2 = group['betas']
        L.check(L.lib().bbb_adam_step(n, tabs[0], tabs[1], tabs[2], tabs[3], sizes, float(group['lr']), float(b1),
                                      float(b2), float(group['eps']), self._t, L.ptr(self.step_dev),
                                      L.ptr(self.lr_scale_dev), L.stream()), 'bbb_adam_step')


_ipc_bases = {}     # CUDA IPC handle bytes -> base pointer mapped in this process (a handle is opened once)


def open_peers(t, group=None):
    """Map the same tensor of every rank of `group` (one node) into this process.  The exporter's handle comes from
    torch (`_share_cuda_`: handle of the cudaMalloc block + byte offset of the tensor inside it); it is opened by
    bbb_ipc_open with THIS rank's device current, so that this device's kernels can load / store it over NVLink.
    Returns the device pointers [rank 0's tensor, rank 1's, ...] as ints (this rank's own: t.data_ptr())."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    shared = t.untyped_storage()._share_cuda_()       # (device, handle, size, offset, ...)
    handle = bytes(shared[1])
    # torch prefixes the 64-byte cudaIpcMemHandle_t with a version / type tag ('c' = plain cudaMalloc block)
    prefix, handle = handle[:-64], handle[-64:]
    if len(handle) != 64 or (prefix and prefix[-1:] != b'c'):
        raise RuntimeError(f'PeerShardedAdam needs cudaMalloc-backed tensors: unexpected CUDA IPC handle '
                           f'(prefix {prefix!r}, {len(handle)} bytes); expandable segments are not shareable here')
    mine = (int(shared[0]), handle, int(shared[3]) + t.storage_offset() * t.element_size())
    every = [None] * world
    dist.all_gather_object(every, mine, group=group)
    ptrs = []
    with torch.cuda.device(t.device):
        for k, (dev_k, handle, off) in enumerate(every):
            if k == rank:
                ptrs.append(t.data_ptr())
                continue
            L.check(L.lib().bbb_enable_peer_access(dev_k), 'bbb_enable_peer_access')
            if handle not in _ipc_bases:
                out = C.c_void_p()
                L.check(L.lib().bbb_ipc_open(handle, 0, C.byref(out)), 'bbb_ipc_open')
                _ipc_bases[handle] = out.value
            ptrs.append(_ipc_bases[handle] + off)
    return ptrs


class PeerShardedAdam(torch.optim.Optimizer):
    """Data-parallel Adam whose gradient exchange rides in the optimiser kernel (csrc/bbb_adam.cu:
    bbb_adam_step_peer): gradient reduce-scatter + Adam + parameter all-gather in ONE launch over NVLink peer
    memory.  Replaces `all_reduce(grads); optimizer.step()`: there is no NCCL call in the step, no separate pass
    over the gradients, and each rank touches 1/world of the optimiser state.

    The parameters are re-homed into one flat buffer (their `.data` become views of it, same values, same
    layout) and the network-level backward writes its gradients into one flat bucket (functional.grad_buckets);
    both are opened by every rank of the node through CUDA IPC.  Every rank must call step() once per step.
    Same update rule and state names as torch.optim.Adam (the per-parameter `exp_avg` / `exp_avg_sq` are views of the
    flat state; only this rank's slice of them is ever non-zero)."""

    reduces_gradients = True      # callers must NOT all-reduce the gradients themselves

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, group=None):
        import torch.distributed as dist
        from . import functional as F
        params = list(params)
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        for p in params:
            L.require_cuda(p)
            if not (p.is_contiguous() and p.dtype == torch.float32):
                raise RuntimeError('PeerShardedAdam needs contiguous fp32 parameters')
        self.group = group
        multi = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if multi else 1
        self.rank = dist.get_rank(group) if multi else 0
        if self.world > 8:
            raise RuntimeError('PeerShardedAdam: at most 8 ranks (one NVLink node)')
        dev = params[0].device
        self.n = sum(p.numel() for p in params)
        npad = (self.n + 3) // 4 * 4
        # NVLS: when torch's symmetric memory comes up on this node WITH a multicast mapping, the parameter buffer and the
        # gradient bucket are allocated from it, and the kernel reads its slice of the gradient sum with multimem.ld_reduce
        # (the NVSwitch adds the ranks' copies: inbound n/W instead of (W-1) n/W) and writes the new parameters with
        # multimem.st.  Measured inside the captured MNIST-shape step (tools/time_peer_adam.py): 8 GPUs 190 us against
        # 207 us with peer loads / stores (the in-switch reduction alone: 196 us); 4 GPUs 191 against 185 us; 2 GPUs 191
        # against 165 us -- so it is used above 4 ranks.  BBB_PEER_NVLS=0: never, =force: at any world size.
        self.mc_p = self.mc_g = 0
        self._symm = None
        mode = os.environ.get('BBB_PEER_NVLS', '1')
        # (buffers above 64 MB -- config 5's 537 MB -- keep the peer path: the exchange is a per-cent of that step, and
        #  multicast mappings of that size were not exercised)
        want = (multi and self.world > 1 and mode != '0' and (mode in ('force', '2') or (self.world > 4 and npad * 4 <= (64 << 20))))
        symm = self._symmetric_buffers(npad, dev, group) if want else None
        if symm is not None:
            self.flat_p, self.flat_g, self._symm = symm[0], symm[1], symm[2:]
            self.flat_p.zero_()
            self.flat_g.zero_()
        else:
            self.flat_p = torch.zeros(npad, dtype=torch.float32, device=dev)
            self.flat_g = torch.zeros(npad, dtype=torch.float32, device=dev)
        self.flat_m = torch.zeros(npad, dtype=torch.float32, device=dev)
        self.flat_v = torch.zeros(npad, dtype=torch.float32, device=dev)
        self.flags = torch.zeros(2 * 8, dtype=torch.int32, device=dev)
        self.words = torch.zeros(4, dtype=torch.int32, device=dev)          # call count, block counter, error word
        self.offsets, off = [], 0
        with torch.no_grad():
            for p in params:
                k = p.numel()
                self.flat_p[off:off + k].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[off:off + k].view(p.shape)
                st = self.state[p]
                st['step'] = torch.tensor(0.0)
                st['exp_avg'] = self.flat_m[off:off + k].view(p.shape)
                st['exp_avg_sq'] = self.flat_v[off:off + k].view(p.shape)
                self.offsets.append(off)
                off += k
        # this network's backward writes its gradients here (only while no p.grad is alive: functional._bucket_for)
        F.grad_buckets[self.flat_p.data_ptr()] = (self.flat_g, weakref.ref(self))
        if self.world > 1:
            dist.broadcast(self.flat_p, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            if self._symm is not None:
                hp, hg = self._symm
                self.peer_p, self.peer_g = [int(q) for q in hp.buffer_ptrs], [int(q) for q in hg.buffer_ptrs]
                self.mc_p, self.mc_g = int(hp.multicast_ptr), int(hg.multicast_ptr)
                if os.environ.get('BBB_PEER_NVLS', '1') == '2':      # (experiments) in-switch reduction only
                    self.mc_p = 0
            else:
                self.peer_p = open_peers(self.flat_p, group)
                self.peer_g = open_peers(self.flat_g, group)
            self.peer_f = open_peers(self.flags, group)
            dist.barrier(group)
        else:
            self.peer_p, self.peer_g, self.peer_f = ([self.flat_p.data_ptr()], [self.flat_g.data_ptr()],
                                                     [self.flags.data_ptr()])
        self.step_dev = None
        self.lr_scale_dev = None
        self._t = 0

    def use_device_step(self, counter):
        self.step_dev = counter

    @staticmethod
    def _symmetric_buffers(npad, dev, group):
        """(flat_p, flat_g, handle_p, handle_g) from torch's symmetric memory when every rank gets a multicast mapping
        for both, else None -- decided collectively, so that all ranks take the same path."""
        import torch.distributed as dist
        def agree(ok):
            flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            return int(flag) == 1
        sm = fp = fg = None
        try:
            import torch.distributed._symmetric_memory as sm
            fp = sm.empty(npad, dtype=torch.float32, device=dev)
            fg = sm.empty(npad, dtype=torch.float32, device=dev)
        except Exception:
            fp = fg = None
        if not agree(fp is not None and fg is not None):      # (nobody enters the rendezvous unless everybody allocated)
            return None
        out = None
        try:
            g = group if group is not None else dist.group.WORLD
            hp, hg = sm.rendezvous(fp, g), sm.rendezvous(fg, g)
            if (int(hp.multicast_ptr) and int(hg.multicast_ptr) and int(hp.buffer_ptrs[hp.rank]) == fp.data_ptr()
                    and int(hg.buffer_ptrs[hg.rank]) == fg.data_ptr()):
                out = (fp, fg, hp, hg)
        except Exception:
            out = None
        return out if agree(out is not None) else None

    def zero_grad(self, set_to_none=True):
        """Always drops the gradients: a p.grad kept alive would alias the shared bucket (functional._bucket_for)."""
        super().zero_grad(set_to_none=True)

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        steps = [float(st['step']) for st in self.state.values() if 'step' in st]
        self._t = int(max(steps)) if steps else 0

    def check_health(self):
        """Raise if a step's bounded wait for a peer rank expired (the kernel then finished without it).  Synchronises."""
        if int(self.words[2]) != 0:
            raise RuntimeError('PeerShardedAdam: a peer rank did not reach the gradient exchange within the kernel\'s '
                               'bounded wait; parameters are no longer consistent across ranks')

    def release(self):
        """Stop routing this network's gradients into the shared bucket (the mapped peer memory itself stays mapped
        for the life of the process: the other ranks may still hold it)."""
        from . import functional as F
        F.grad_buckets.pop(self.flat_p.data_ptr(), None)

    def _comm(self):
        c = L.PeerComm()
        c.world, c.rank = self.world, self.rank
        for k in range(self.world):
            c.grads[k], c.params[k], c.flags[k] = self.peer_g[k], self.peer_p[k], self.peer_f[k]
        c.epoch, c.done_blocks = self.words[0:1].data_ptr(), self.words[1:2].data_ptr()
        c.mc_grads, c.mc_params = (self.mc_g or None), (self.mc_p or None)
        return c

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        self._t += 1
        group = self.param_groups[0]
        # gradients that did not land in the bucket (layer-level API, foreign autograd paths) are copied into it
        for p, off in zip(group['params'], self.offsets):
            g = p.grad
            if g is None:
                self.flat_g[off:off + p.numel()].zero_()
            elif not (g.is_contiguous() and g.data_ptr() == self.flat_g.data_ptr() + 4 * off):
                self.flat_g[off:off + p.numel()].copy_(g.reshape(-1))
        b1, b2 = group['betas']
        comm = self._comm()
        L.check(L.lib().bbb_adam_step_peer(C.byref(comm), L.ptr(self.flat_m), L.ptr(self.flat_v), self.n,
                                           float(group['lr']), float(b1), float(b2), float(group['eps']), self._t,
                                           L.ptr(self.step_dev), L.ptr(self.lr_scale_dev), L.stream()),
                'bbb_adam_step_peer')
        for st in self.state.values():
            st['step'].fill_(float(self._t))
        return loss
