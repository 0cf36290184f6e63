"""Fused training step (train.py:182-196) and its data-parallel form.

``TrainStep`` chains, on one stream and without autograd bookkeeping,
    forward (activations kept) -> loss + dlogits kernel -> backward into the flat gradient
    buffer -> [NCCL all-reduce of the gradient-receiving prefix] -> one fused AdamW launch.
The only collective of the whole path is that all-reduce (SURVEY §8e) of the ``model.n_active``
gradient values, summed, with the 1/world mean folded into the AdamW kernel.  With more than one rank
it travels as two buckets: the head + Regulation-transformer gradients (78 % of the bytes, a contiguous
tail of the flat buffer) are final once the first part of the backward (``CHROMO_F_BWD_HEAD_REG``) has
run, so their all-reduce is issued there and overlaps the Pairwise / Embedding part
(``CHROMO_F_BWD_REST``); only the small second bucket is exposed.
"""
import ctypes

import torch
import torch.distributed as dist

from . import _lib
from .model import _BatchIO
from .parallel import allreduce_gradients
from .synthetic import FORWARD_KEYS


class TrainStep:
    """``use_graph``: after two eager steps with a given batch geometry the forward + loss + backward chain of that
    geometry (about 330 small launches at batch 64) is captured in a CUDA graph and replayed; every step then costs one
    graph launch, the copies of the new batch into the graph's input buffers, the (eager) all-reduce and one AdamW
    launch.  Other geometries (a short last batch) keep running eagerly."""

    GRAPH_AFTER = 2

    def __init__(self, model, lr=3e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, regression=False,
                 process_group=None, distributed=None, use_graph=True):
        self.model = model
        self.lr, self.betas, self.eps, self.wd = lr, betas, eps, weight_decay
        self.regression = regression
        self.group = process_group
        self.world = 1
        if distributed is None:
            distributed = dist.is_available() and dist.is_initialized()
        if distributed:
            self.world = dist.get_world_size(process_group)
        flat = model.flat_params
        self.grad = torch.zeros_like(flat)
        self.m = torch.zeros_like(flat)
        self.v = torch.zeros_like(flat)
        self.loss = torch.zeros(1, device=flat.device)
        self.step_count = 0
        self.flags = _lib.F_TRAINING | model._precision_flag()
        self._ws = None
        self.use_graph = use_graph
        self._seen = {}          # geometry -> eager steps so far
        self._graphs = {}        # geometry -> captured chain
        self._flat_ptr = flat.data_ptr()
        self.graph_replays = 0
        # first element of the head + Regulation bucket (parameter layout: embed x3 | pairwise x3 | regulation x3 | head)
        self.bucket_split = min(off for (name, _, off, _) in model._slots
                                if off < model.n_active and model._lib_name(name).startswith(("regulation.", "fc_head.")))
        # measured (B200, batch 64 per rank): 2 ranks 1.47 ms single bucket / 1.49 ms two buckets, 4 ranks 1.52 / 1.49: the
        # second graph launch and NCCL call cost what the overlap saves until the all-reduce takes ~0.1 ms
        self.overlap = self.world > 2

    # ---- forward + loss + backward into self.grad (everything a CUDA graph may hold) -------------------------
    def _chain(self, io, target, logits, dlogits, part=0):
        """part 0: the whole chain; 1: forward + loss + head / Regulation backward; 2: the rest of the backward."""
        lib = _lib.load()
        model = self.model
        flat = model.flat_params
        stream = torch.cuda.current_stream(flat.device).cuda_stream
        ws = self._ws
        cfg = ctypes.byref(io.cfg)
        n_out = int(io.cfg.n_out)
        if part in (0, 1):
            _lib.check(lib.chromo_forward(cfg, flat.data_ptr(), ctypes.byref(io.struct), logits.data_ptr(),
                                          ws.data_ptr(), ws.numel(), self.flags, stream), "chromo_forward")
            if self.regression:
                _lib.check(lib.chromo_mse_loss(logits.data_ptr(), target.data_ptr(), io.batch * n_out, 1.0,
                                               self.loss.data_ptr(), dlogits.data_ptr(), stream), "chromo_mse_loss")
            else:
                _lib.check(lib.chromo_ce_loss(logits.data_ptr(), target.data_ptr(), io.batch, n_out, 1.0,
                                              self.loss.data_ptr(), dlogits.data_ptr(), stream), "chromo_ce_loss")
            self.grad[:model.n_active].zero_()
        flags = self.flags | {0: 0, 1: _lib.F_BWD_HEAD_REG, 2: _lib.F_BWD_REST}[part]
        _lib.check(lib.chromo_backward(cfg, flat.data_ptr(), ctypes.byref(io.struct), dlogits.data_ptr(),
                                       self.grad.data_ptr(), ws.data_ptr(), ws.numel(), flags, stream),
                   "chromo_backward")

    def _reduce(self, lo, hi):
        """Asynchronous SUM all-reduce of grad[lo:hi] (ordered behind the work enqueued so far on the current stream)."""
        return dist.all_reduce(self.grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    def _io(self, batch):
        model = self.model
        return _BatchIO(model, *[[batch[k][b] for b in model.binsizes] if isinstance(batch[k], dict) else batch[k]
                                 for k in FORWARD_KEYS])

    def _target(self, target):
        return target.to(torch.float32 if self.regression else torch.int64).contiguous()

    @staticmethod
    def _geometry(batch, target):
        key = [tuple(target.shape)]
        for k in FORWARD_KEYS:
            v = batch[k]
            key += [(b, tuple(t.shape), t.dtype) for b, t in v.items()] if isinstance(v, dict) else [(tuple(v.shape), v.dtype)]
        return tuple(key)

    def _capture(self, key, batch, target):
        """Static copies of the batch, one eager run on them, then the same chain under graph capture."""
        dev = self.model.flat_params.device
        static = {k: ({b: t.detach().clone().contiguous() for b, t in batch[k].items()} if isinstance(batch[k], dict)
                      else batch[k].detach().clone().contiguous()) for k in FORWARD_KEYS}
        tgt = self._target(target).clone()
        io = self._io(static)
        logits = torch.empty(io.batch, int(io.cfg.n_out), dtype=torch.float32, device=dev)
        dlogits = torch.empty_like(logits)
        graphs = [torch.cuda.CUDAGraph() for _ in range(2 if self.overlap else 1)]
        try:
            torch.cuda.synchronize(dev)
            for part, graph in enumerate(graphs, 1 if self.overlap else 0):
                with torch.cuda.graph(graph):
                    self._chain(io, tgt, logits, dlogits, part)
        except Exception:                      # a driver / toolkit that cannot capture this chain: stay eager
            self.use_graph = False
            torch.cuda.synchronize(dev)
            return None
        self._flat_ptr = self.model.flat_params.data_ptr()
        ent = {"graphs": graphs, "static": static, "target": tgt, "io": io, "logits": logits, "dlogits": dlogits}
        self._graphs[key] = ent
        return ent

    def __call__(self, batch, target):
        """batch: dict with the six forward arguments on the model's device; target: labels.
        Returns the (device) loss tensor of this rank's micro-batch; no host sync."""
        lib = _lib.load()
        model = self.model
        flat = model.flat_params
        dev = flat.device
        key = self._geometry(batch, target) if self.use_graph else None
        if self._graphs and self._flat_ptr != flat.data_ptr():      # the model's buffer moved: captured chains are stale
            self._graphs.clear()
            self._seen.clear()
        ent = self._graphs.get(key) if self.use_graph else None
        if ent is None:
            io = self._io(batch)
            need = _lib.check(lib.chromo_workspace_floats(ctypes.byref(io.cfg), io.batch, self.flags), "workspace")
            if self._ws is None or self._ws.numel() < need:
                if self._graphs:               # captured chains point into the old workspace
                    self._graphs.clear()
                    self._seen.clear()
                self._ws = torch.empty(need, dtype=torch.float32, device=dev)
            seen = self._seen.get(key, 0) if self.use_graph else 0
            if self.use_graph and seen >= self.GRAPH_AFTER:
                ent = self._capture(key, batch, target)
        if ent is not None:
            # the captured chain reads its own input buffers; a caller that already wrote the batch into them
            # (`input_buffers`, e.g. as the destination of its host->device copies) pays no copy here
            for k in FORWARD_KEYS:
                if isinstance(batch[k], dict):
                    for b, t in batch[k].items():
                        if t.data_ptr() != ent["static"][k][b].data_ptr():
                            ent["static"][k][b].copy_(t, non_blocking=True)
                elif batch[k].data_ptr() != ent["static"][k].data_ptr():
                    ent["static"][k].copy_(batch[k], non_blocking=True)
            if target.data_ptr() != ent["target"].data_ptr():
                ent["target"].copy_(target, non_blocking=True)
            pending = []
            for i, graph in enumerate(ent["graphs"]):
                graph.replay()
                if self.overlap:               # bucket 1 travels under the second graph, bucket 2 behind it
                    pending.append(self._reduce(self.bucket_split, model.n_active) if i == 0 else self._reduce(0, self.bucket_split))
            self.graph_replays += 1
            logits = ent["logits"]
        else:
            if self.use_graph:
                self._seen[key] = self._seen.get(key, 0) + 1
            logits = torch.empty(io.batch, int(io.cfg.n_out), dtype=torch.float32, device=dev)
            dlogits = torch.empty_like(logits)
            tgt = self._target(target)
            pending = []
            if self.overlap:
                self._chain(io, tgt, logits, dlogits, 1)
                pending.append(self._reduce(self.bucket_split, model.n_active))
                self._chain(io, tgt, logits, dlogits, 2)
                pending.append(self._reduce(0, self.bucket_split))
            else:
                self._chain(io, tgt, logits, dlogits)
        stream = torch.cuda.current_stream(dev).cuda_stream
        if self.overlap:
            for h in pending:
                h.wait()                       # (stream-side wait: the host does not block)
            scale = 1.0 / self.world
        else:
            scale = allreduce_gradients(self.grad, model.n_active, self.group) if self.world > 1 else 1.0
        self.step_count += 1
        _lib.check(lib.chromo_adamw(flat.data_ptr(), self.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                    model.n_active, self.lr, self.betas[0], self.betas[1], self.eps, self.wd,
                                    self.step_count, scale, stream), "chromo_adamw")
        model.mark_parameters_changed()
        self.logits = logits
        return self.loss

    def input_buffers(self, batch, target):
        """The device buffers the captured chain of this batch geometry reads: (batch dict, target), or None while the
        geometry still runs eagerly.  Filling them directly (they are the natural destination of the host->device copies of
        the next batch) and passing them to `__call__` removes the per-step device-to-device copies."""
        ent = self._graphs.get(self._geometry(batch, target)) if self.use_graph else None
        if ent is None:
            return None
        tgt = ent["target"]
        return dict(ent["static"]), tgt.view(target.shape) if tgt.numel() == target.numel() else tgt

    def set_lr(self, lr):
        """StepLR hook (train.py:158,344)."""
        self.lr = float(lr)
