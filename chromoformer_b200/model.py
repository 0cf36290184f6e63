"""Chromoformer modules on top of ``libchromo_b200.so``.

Mirrors the reference's public surface — ``chromoformer/net.py`` classes
``Chromoformer`` (flat API, net.py:156-270), ``ChromoformerBase`` /
``ChromoformerClassifier`` (dict API, net.py:273-383) and
``ChromoformerRegressor`` (net.py:386-428): same constructor arguments, same
``forward`` signatures, same ``state_dict`` keys/shapes and, because parameters
are created by the same sequence of ``nn.Linear`` / ``nn.LayerNorm`` constructor
calls after ``torch.manual_seed(seed)`` (SURVEY A.5), the same initial weights.

What differs is everything behind ``forward``: the sub-modules only OWN
parameters (all of them views into one flat FP32 buffer whose layout the C
library dictates); the math runs in hand-written sm_100a kernels reached through
the C ABI, forward and backward.  There is no PyTorch fallback.
"""
import ctypes
import math
import os
import re

import numpy as np
import torch
import torch.nn as nn

from . import _lib

__all__ = ["Chromoformer", "ChromoformerBase", "ChromoformerClassifier", "ChromoformerRegressor",
           "EmbeddingTransformer", "PairwiseInteractionTransformer", "RegulationTransformer",
           "sinusoid_table"]


def sinusoid_table(n_pos, dim):
    """Sinusoidal position table of net.py:23-29, evaluated on the host with the same
    FP32 operation sequence so that the values are bit-identical to the reference's."""
    rate = torch.exp(-np.log(10000) * torch.arange(0, dim, 2) / dim)
    phase = torch.arange(0, n_pos, 1).unsqueeze(1) * rate
    table = torch.zeros(n_pos, dim)
    table[:, 0::2] = torch.sin(phase)
    table[:, 1::2] = torch.cos(phase)
    return table


# --------------------------------------------------------------------------------------
# Parameter containers.  Attribute names ARE the checkpoint schema (SURVEY A.3); the
# construction order IS the initialisation contract (SURVEY A.5).
# --------------------------------------------------------------------------------------
class _SelfAttention(nn.Module):
    """Parameters of modules.py:8-26 (``gate`` widens the fused projection to q|k|v|gate)."""

    def __init__(self, d_emb, n_heads, d_model, gate):
        super().__init__()
        width = (d_model // n_heads) * n_heads
        self.gamma_f = nn.Parameter(torch.ones([n_heads]))
        self.w_bias = nn.Linear(2, n_heads, bias=False)      # never used by the reference; consumes RNG
        self.att = nn.Linear(d_emb, (4 if gate else 3) * width, bias=False)
        self.ff = nn.Linear(width, d_emb)
        self.ln = nn.LayerNorm(d_emb)


class _CrossAttention(nn.Module):
    """Parameters of modules.py:127-148 (promoter queries, pCRE keys/values)."""

    def __init__(self, d_emb, n_heads, d_model):
        super().__init__()
        width = (d_model // n_heads) * n_heads
        self.gamma_f = nn.Parameter(torch.ones([n_heads]))
        self.p_att = nn.Linear(d_emb, width, bias=False)
        self.c_att = nn.Linear(d_emb, 2 * width, bias=False)
        self.ff = nn.Linear(width, d_emb)
        self.ln = nn.LayerNorm(d_emb)


class _FeedForward(nn.Module):
    """Parameters of modules.py:91-97."""

    def __init__(self, d_emb, d_ff):
        super().__init__()
        self.l1 = nn.Linear(d_emb, d_ff)
        self.l2 = nn.Linear(d_ff, d_emb)
        self.ln = nn.LayerNorm(d_emb)


class _Layer(nn.Module):
    def __init__(self, att, d_emb, d_ff):
        super().__init__()
        self.self_att = att
        self.ff = _FeedForward(d_emb, d_ff)


class _Stack(nn.Module):
    def __init__(self, layers):
        super().__init__()
        self.layers = nn.ModuleList(layers)


def _default_precision():
    p = os.environ.get("CHROMO_PRECISION", "fp32").strip().lower()
    if p not in ("fp32", "bf16"):
        raise ValueError(f"CHROMO_PRECISION must be 'fp32' or 'bf16', got {p!r}")
    return p


# Legacy checkpoint key generations (misc/convert_weight.py:19-88), oldest first.  Each rule rewrites one
# generation's spelling into the dict layout of net.py:273-330; `canonical_key` applies them in that order.
_LEGACY_RULES = (
    (re.compile(r"lin_proj_c(?=\.)"), "lin_proj_pcre"),
    (re.compile(r"^transformer(\d+)\."), r"regulation.\1.transformer."),
    (re.compile(r"^embed(\d+)_a\."), r"embed.\1."),
    (re.compile(r"^embed(\d+)_b\."), r"pairwise_interaction.\1."),
    (re.compile(r"^embed(\d+)\."), r"embed.\1."),
    (re.compile(r"^pw_int(\d+)\."), r"pairwise_interaction.\1."),
    (re.compile(r"^reg(\d+)\."), r"regulation.\1."),
)


def canonical_key(key):
    """Any generation of checkpoint key -> the dict-layout key (`embed.2000.…`, `pairwise_interaction.2000.…`,
    `regulation.2000.…`); keys already in that layout come back unchanged."""
    for pat, rep in _LEGACY_RULES:
        key = pat.sub(rep, key)
    return key


def _standalone_error(name):
    raise NotImplementedError(
        f"{name} is a parameter container here: the sm_100a kernels evaluate the whole "
        "Chromoformer forward (centre-query pruned) through the parent model; calling the "
        "sub-module on its own is not part of the accelerated path.")


class EmbeddingTransformer(nn.Module):
    """net.py:9-59."""

    def __init__(self, n_feats, n_layers, n_heads, d_model, d_ff, **_unused):
        super().__init__()
        self.d_model = d_model
        self.lin_proj = nn.Linear(n_feats, d_model, bias=False)
        self.transformer = _Stack([
            _Layer(_SelfAttention(d_model, n_heads, d_model, gate=False), d_model, d_ff) for _ in range(n_layers)])

    def forward(self, *a, **k):
        _standalone_error("EmbeddingTransformer")


class PairwiseInteractionTransformer(nn.Module):
    """net.py:62-139."""

    def __init__(self, n_feats_p, n_feats_pcre, n_layers, n_heads, d_model, d_ff, **_unused):
        super().__init__()
        self.d_model = d_model
        self.ln = nn.LayerNorm(d_model)                     # constructed, never applied (net.py:80)
        self.lin_proj_p = nn.Linear(n_feats_p, d_model, bias=False)
        self.lin_proj_pcre = nn.Linear(n_feats_pcre, d_model, bias=False)
        self.transformer = _Stack([
            _Layer(_CrossAttention(d_model, n_heads, d_model), d_model, d_ff) for _ in range(n_layers)])

    def forward(self, *a, **k):
        _standalone_error("PairwiseInteractionTransformer")


class RegulationTransformer(nn.Module):
    """net.py:142-153."""

    def __init__(self, n_layers, n_heads, d_emb, d_model, d_ff, **_unused):
        super().__init__()
        self.transformer = _Stack([
            _Layer(_SelfAttention(d_emb, n_heads, d_model, gate=True), d_emb, d_ff) for _ in range(n_layers)])

    def forward(self, *a, **k):
        _standalone_error("RegulationTransformer")


# --------------------------------------------------------------------------------------
# autograd bridge
# --------------------------------------------------------------------------------------
class _ChromoFunction(torch.autograd.Function):
    """loss.backward() support for the unchanged training loop (train.py:182-196), and gradients with respect to the
    inputs: the histone-mark features (``promoter_feats`` / ``pcre_feats``) and ``interaction_freq``, passed as
    ``inputs``: every x_p, then every x_pcre, then interaction_freq.

    Limits (by design: the backward kernels write straight into the flat gradient buffer): parameter gradients
    arrive as a side effect on ``p.grad`` (``torch.autograd.grad(loss, params)`` sees only the zero anchor), the
    masks and position tables get no gradient, and a forward's activations are released by its first backward
    (no ``retain_graph``)."""

    @staticmethod
    def forward(ctx, anchor, model, io, *inputs):
        logits, ws = model._launch_forward(io, _lib.F_TRAINING | model._precision_flag())
        ctx.model, ctx.io, ctx.ws = model, io, ws
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        model, io, ws = ctx.model, ctx.io, ctx.ws
        if ws is None:
            raise RuntimeError("chromoformer_b200: this forward's activations were released by its first backward "
                               "(retain_graph is not supported: run the forward again)")
        want = ctx.needs_input_grad[3:]
        dx = model._launch_backward(io, ws, dlogits.contiguous(), want if any(want) else None)
        ctx.ws = None
        return (None, None, None) + tuple(dx if dx is not None else [None] * len(want))


class _BatchIO:
    """Validated, contiguous device tensors of one batch + the C struct pointing at them."""

    def __init__(self, model, x_p, mask_p, x_pcre, mask_pcre, imask, freq):
        # i_max and the bins per resolution are properties of the batch, as in the reference
        # (net.py:36,110 read them off the tensors), not of the parameters.
        cfg = _lib.Config.from_buffer_copy(model._cfg)
        cfg.i_max = int(x_pcre[0].size(1))
        for r in range(cfg.n_res):
            cfg.n_bins[r] = int(x_p[r].size(-2))
        self.cfg = cfg
        dev = model._flat.device
        if dev.type != "cuda":
            raise _lib.ChromoLibError("Chromoformer parameters are on %s; the sm_100a kernels need "
                                      "model.cuda() (there is no CPU fallback)" % dev)
        self.keep = []
        self.x_p, self.x_pcre = [], []            # the FP32 contiguous features (their gradients take these shapes)
        st = _lib.Batch()
        B = int(mask_p[0].size(0))
        S = cfg.i_max + 1
        st.batch = B
        self.batch = B

        def dev_tensor(t, dtype, what):
            if t.device != dev:
                raise ValueError(f"{what} is on {t.device}, model on {dev}")
            t = t.detach()        # (a feature that requires grad reaches the kernels through _ChromoFunction)
            if t.dtype != dtype:
                t = t.to(dtype)
            t = t.contiguous()
            self.keep.append(t)
            return t

        for r in range(cfg.n_res):
            n = int(cfg.n_bins[r])
            xp = dev_tensor(x_p[r], torch.float32, "promoter_feats")
            xc = dev_tensor(x_pcre[r], torch.float32, "pcre_feats")
            if xp.numel() != B * n * cfg.n_feats:
                raise ValueError(f"promoter_feats[{r}] has shape {tuple(xp.shape)}, expected [{B},1,{n},{cfg.n_feats}]")
            if xc.numel() != B * cfg.i_max * n * cfg.n_feats:
                raise ValueError(f"pcre_feats[{r}] has shape {tuple(xc.shape)}, expected "
                                 f"[{B},{cfg.i_max},{n},{cfg.n_feats}]")
            st.x_p[r] = xp.data_ptr()
            st.x_pcre[r] = xc.data_ptr()
            self.x_p.append(xp)
            self.x_pcre.append(xc)
            for name, m, regions in (("p", mask_p[r], 1), ("pcre", mask_pcre[r], cfg.i_max)):
                m = dev_tensor(m, torch.bool, "pad mask")
                if m.numel() == B * regions * n * n:          # [B,regions,1,n,n] as in data.py:156-198
                    stride, off = n * n, (n // 2) * n
                elif m.numel() == B * regions * n:            # centre rows only
                    stride, off = n, 0
                else:
                    raise ValueError(f"pad mask has shape {tuple(m.shape)}; expected [{B},{regions},1,{n},{n}]")
                setattr_arr = getattr(st, "mask_" + name)
                setattr_arr[r] = m.data_ptr()
                getattr(st, "mask_" + name + "_stride")[r] = stride
                getattr(st, "mask_" + name + "_row_offset")[r] = off
            im = dev_tensor(imask[r], torch.bool, "interaction_mask")
            if im.numel() != B * S * S:
                raise ValueError(f"interaction_mask has shape {tuple(im.shape)}, expected [{B},1,{S},{S}]")
            st.imask[r] = im.data_ptr()
            st.pos_enc[r] = model._pos_table(n, dev).data_ptr()
        fq = dev_tensor(freq, torch.float32, "interaction_freq")
        if fq.numel() != B * S * S:
            raise ValueError(f"interaction_freq has shape {tuple(fq.shape)}, expected [{B},{S},{S}]")
        st.freq = fq.data_ptr()
        self.freq = fq                            # (and its gradient this shape)
        self.struct = st


class _ChromoformerCore(nn.Module):
    """Shared machinery: flat parameter buffer, C config, launchers."""

    #: "fp32" = strict FP32 on the CUDA cores, "bf16" = tcgen05 BF16 operands / FP32 accumulate.  The class default
    #: comes from the environment (CHROMO_PRECISION=bf16) so that callers that cannot be edited - the reference's
    #: demo/run_demo.py, `python -m chromoformer.train` - reach the tensor path without a code change.
    precision = _default_precision()

    # ---- construction ----------------------------------------------------------------
    def _finalise(self, n_feats, d_emb, d_head, n_out, embed_kws, pw_kws, reg_kws, binsizes, i_max, w_max):
        cfg = _lib.Config()
        cfg.n_feats, cfg.d_emb, cfg.d_head, cfg.n_out = n_feats, d_emb, d_head, n_out
        cfg.n_res, cfg.i_max = len(binsizes), i_max
        cfg.embed_layers, cfg.embed_heads = embed_kws["n_layers"], embed_kws["n_heads"]
        cfg.embed_d_model, cfg.embed_d_ff = embed_kws["d_model"], embed_kws["d_ff"]
        cfg.pw_layers, cfg.pw_heads = pw_kws["n_layers"], pw_kws["n_heads"]
        cfg.pw_d_model, cfg.pw_d_ff = pw_kws["d_model"], pw_kws["d_ff"]
        cfg.reg_layers, cfg.reg_heads = reg_kws["n_layers"], reg_kws["n_heads"]
        cfg.reg_d_model, cfg.reg_d_ff = reg_kws["d_model"], reg_kws["d_ff"]
        for r, b in enumerate(binsizes):
            cfg.n_bins[r] = w_max // int(b)
        object.__setattr__(self, "_cfg", cfg)
        object.__setattr__(self, "_pe_cache", {})
        object.__setattr__(self, "_ws_cache", {})
        object.__setattr__(self, "_flat", None)
        object.__setattr__(self, "_flat_grad", None)
        object.__setattr__(self, "_anchor", None)
        object.__setattr__(self, "_table", None)
        object.__setattr__(self, "_packed_key", None)
        object.__setattr__(self, "_deletion_packed_key", None)
        object.__setattr__(self, "_param_epoch", 0)
        self._rebuild_flat()

    def _lib_name(self, name):
        """state_dict key -> library tensor name (resolution index instead of bin size)."""
        raise NotImplementedError

    def _rebuild_flat(self):
        """(Re)create the flat buffer on the parameters' current device and re-point every
        parameter at its slice.  Called after construction and after .cuda()/.to()."""
        lib = _lib.load()
        cfg = self._cfg
        table = _lib.param_table(cfg)
        total = _lib.check(lib.chromo_param_total(ctypes.byref(cfg)), "chromo_param_total")
        params = list(self.named_parameters())
        dev = params[0][1].device
        flat = torch.zeros(total, dtype=torch.float32, device=dev)
        seen = set()
        slots = []
        with torch.no_grad():
            for name, p in params:
                key = self._lib_name(name)
                if key not in table:
                    raise _lib.ChromoLibError(f"parameter {name} ({key}) unknown to libchromo_b200")
                off, numel = table[key]
                if numel != p.numel():
                    raise _lib.ChromoLibError(f"parameter {name}: {p.numel()} elements, library expects {numel}")
                view = flat[off:off + numel].view(p.shape)
                view.copy_(p.detach().to(torch.float32))
                p.data = view
                seen.add(key)
                slots.append((name, p, off, numel))
        missing = set(table) - seen
        if missing:
            raise _lib.ChromoLibError(f"library tensors without a parameter: {sorted(missing)[:4]}...")
        active = _lib.check(lib.chromo_param_active(ctypes.byref(cfg)), "chromo_param_active")
        object.__setattr__(self, "_flat", flat)
        object.__setattr__(self, "_flat_grad", None)
        object.__setattr__(self, "_slots", slots)
        object.__setattr__(self, "_n_active", int(active))
        object.__setattr__(self, "_active", [p for (_, p, off, _) in slots if off < active])
        object.__setattr__(self, "_anchor", torch.zeros(1, device=dev, requires_grad=True))
        self._ws_cache.clear()
        self.mark_parameters_changed()

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        if getattr(self, "_flat", None) is not None:
            self._rebuild_flat()
        return out

    def mark_parameters_changed(self):
        """Call after updating parameters through raw pointers (the fused optimiser does): cached
        BF16 weight packs are rebuilt on the next forward.  In-place torch ops are tracked automatically."""
        object.__setattr__(self, "_param_epoch", self._param_epoch + 1)
        object.__setattr__(self, "_packed_key", None)
        object.__setattr__(self, "_deletion_packed_key", None)

    def _flat_is_current(self):
        base = self._flat.data_ptr()
        return all(p.data_ptr() == base + 4 * off for (_, p, off, _) in self._slots)

    # ---- flat views used by the optimiser / data-parallel wrapper ----------------------
    @property
    def flat_params(self):
        """The single FP32 buffer all parameters live in (gradient-receiving tensors first)."""
        return self._flat

    @property
    def flat_grads(self):
        return self._flat_grad

    @property
    def n_active(self):
        """Length of the gradient-receiving prefix of the flat buffers (SURVEY A.4)."""
        return self._n_active

    def active_parameters(self):
        return self._active

    # ---- launchers ---------------------------------------------------------------------
    def _precision_flag(self):
        if self.precision == "fp32":
            return 0
        if self.precision == "bf16":
            return _lib.F_BF16
        raise ValueError("precision must be 'fp32' or 'bf16'")

    def _pos_table(self, n, dev):
        key = (n, str(dev))
        t = self._pe_cache.get(key)
        if t is None:
            t = sinusoid_table(n, int(self._cfg.d_emb)).to(dev).contiguous()
            self._pe_cache[key] = t
        return t

    def _workspace(self, cfg, batch, flags, cached, entry="chromo_workspace_floats"):
        lib = _lib.load()
        n = _lib.check(getattr(lib, entry)(ctypes.byref(cfg), batch, flags), entry)
        if not cached:
            return torch.empty(n, dtype=torch.float32, device=self._flat.device)
        key = (str(self._flat.device), flags & ~_lib.F_DENSE)      # (the hint does not change the layout)
        if entry != "chromo_workspace_floats":
            key = (entry,) + key
        ws = self._ws_cache.get(key)
        if ws is None or ws.numel() < n:
            ws = torch.empty(n, dtype=torch.float32, device=self._flat.device)
            self._ws_cache[key] = ws
        return ws

    def _launch_forward(self, io, flags):
        lib = _lib.load()
        if not self._flat_is_current():
            self._rebuild_flat()
        training = bool(flags & _lib.F_TRAINING)
        ws = self._workspace(io.cfg, io.batch, flags, cached=not training)
        packed_key = self._packed_key_of(ws, io, flags) if not training else None
        if packed_key is not None and packed_key == self._packed_key:
            flags |= _lib.F_PACKED
        logits = torch.empty(io.batch, int(self._cfg.n_out), dtype=torch.float32, device=self._flat.device)
        stream = torch.cuda.current_stream(self._flat.device).cuda_stream
        _lib.check(lib.chromo_forward(ctypes.byref(io.cfg), self._flat.data_ptr(), ctypes.byref(io.struct),
                                      logits.data_ptr(), ws.data_ptr(), ws.numel(), flags, stream),
                   "chromo_forward")
        if packed_key is not None:
            object.__setattr__(self, "_packed_key", packed_key)
        return logits, ws

    def _packed_key_of(self, ws, io, flags):
        """The packed BF16 weights live at the (batch-independent) front of a cached inference workspace: they can be
        reused while neither the buffer nor the parameters changed (p.data = view keeps each parameter's own version
        counter, so sum them).  None: nothing is packed (FP32)."""
        if not flags & _lib.F_BF16:
            return None
        return (ws.data_ptr(), sum(p._version for (_, p, _, _) in self._slots), self._param_epoch,
                int(io.cfg.i_max), tuple(io.cfg.n_bins[r] for r in range(io.cfg.n_res)))

    def _launch_deletion(self, io, flags):
        """chromo_pcre_deletion: (logits [B, n_out], without [B, I, n_out], promoter_only [B, n_out]).  Its workspace
        and packed BF16 weights are cached apart from the forward's, so the two never invalidate each other."""
        lib = _lib.load()
        if not self._flat_is_current():
            self._rebuild_flat()
        ws = self._workspace(io.cfg, io.batch, flags, cached=True, entry="chromo_pcre_deletion_workspace_floats")
        packed_key = self._packed_key_of(ws, io, flags)
        if packed_key is not None and packed_key == self._deletion_packed_key:
            flags |= _lib.F_PACKED
        dev, n_out, I = self._flat.device, int(self._cfg.n_out), int(io.cfg.i_max)
        logits = torch.empty(io.batch, n_out, dtype=torch.float32, device=dev)
        without = torch.empty(io.batch, I, n_out, dtype=torch.float32, device=dev)
        promoter_only = torch.empty(io.batch, n_out, dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.chromo_pcre_deletion(ctypes.byref(io.cfg), self._flat.data_ptr(), ctypes.byref(io.struct),
                                            logits.data_ptr(), without.data_ptr(), promoter_only.data_ptr(),
                                            ws.data_ptr(), ws.numel(), flags, stream), "chromo_pcre_deletion")
        if packed_key is not None:
            object.__setattr__(self, "_deletion_packed_key", packed_key)
        return logits, without, promoter_only

    def _launch_backward(self, io, ws, dlogits, want_dx=None):
        """Parameter gradients into ``p.grad`` (chromo_backward).  ``want_dx``: one flag per input tensor (every x_p,
        then every x_pcre, then interaction_freq); the pass then also returns those inputs' gradients
        (chromo_backward_inputs), and leaves the parameter gradients out entirely when no active parameter requires
        grad."""
        lib = _lib.load()
        flat = self._flat
        active = self.active_parameters()
        stream = torch.cuda.current_stream(flat.device).cuda_stream
        flags = _lib.F_TRAINING | self._precision_flag()
        dx, dx_struct = None, None
        if want_dx is not None:
            nr = len(io.x_p)
            dx = [torch.empty_like(t) if w else None for t, w in zip(io.x_p + io.x_pcre + [io.freq], want_dx)]
            dx_struct = _lib.InputGrads()
            for r in range(nr):
                dx_struct.x_p[r] = dx[r].data_ptr() if dx[r] is not None else None
                dx_struct.x_pcre[r] = dx[nr + r].data_ptr() if dx[nr + r] is not None else None
            if dx[-1] is not None:
                dx_struct.freq = dx[-1].data_ptr()
                flags |= _lib.F_FREQ_GRAD
            if not any(p.requires_grad for p in active):
                _lib.check(lib.chromo_backward_inputs(ctypes.byref(io.cfg), flat.data_ptr(), ctypes.byref(io.struct),
                                                      dlogits.data_ptr(), None, ctypes.byref(dx_struct), ws.data_ptr(),
                                                      ws.numel(), flags, stream), "chromo_backward_inputs")
                return dx
        fresh = all(p.grad is None for p in active)
        ours = self._flat_grad is not None and not fresh and all(
            p.grad is not None and p.grad.data_ptr() == self._flat_grad.data_ptr() + 4 * off
            for (_, p, off, _) in self._slots if off < self._n_active)
        if self._flat_grad is None or self._flat_grad.device != flat.device:
            object.__setattr__(self, "_flat_grad", torch.zeros_like(flat))
            ours = False
        if fresh:
            target = self._flat_grad
            target.zero_()
        elif ours:
            target = self._flat_grad
        else:
            target = torch.zeros_like(flat)
        if dx_struct is None:
            _lib.check(lib.chromo_backward(ctypes.byref(io.cfg), flat.data_ptr(), ctypes.byref(io.struct),
                                           dlogits.data_ptr(), target.data_ptr(), ws.data_ptr(), ws.numel(),
                                           flags, stream), "chromo_backward")
        else:
            _lib.check(lib.chromo_backward_inputs(ctypes.byref(io.cfg), flat.data_ptr(), ctypes.byref(io.struct),
                                                  dlogits.data_ptr(), target.data_ptr(), ctypes.byref(dx_struct),
                                                  ws.data_ptr(), ws.numel(), flags, stream), "chromo_backward_inputs")
        if fresh:
            for (_, p, off, numel) in self._slots:
                if off < self._n_active and p.requires_grad:
                    p.grad = target[off:off + numel].view(p.shape)
        elif not ours:
            for (_, p, off, numel) in self._slots:
                if off < self._n_active and p.requires_grad:
                    g = target[off:off + numel].view(p.shape)
                    p.grad = g.clone() if p.grad is None else p.grad + g
        return dx

    # ---- checkpoints: every key generation of the reference loads into every class (misc/convert_weight.py) ----
    def _own_key(self, canon):
        """dict-layout key -> this class's own state_dict key."""
        return canon

    def load_state_dict(self, state_dict, strict=True, assign=False):
        mapped = {self._own_key(canonical_key(k)): v for k, v in state_dict.items()}
        out = super().load_state_dict(mapped, strict=strict, assign=assign)
        if not self._flat_is_current():          # assign=True rebinds the parameters: re-home them in the flat buffer
            self._rebuild_flat()
        else:
            self.mark_parameters_changed()
        return out

    def forward_batch(self, batch, dense=False):
        """Forward from a dict of the six arguments keyed like the reference's collated items (dicts by int bin size):
        the one calling convention `InferenceEngine` / `EnsembleSweep` use for the flat and the dict API alike.
        `dense`: hint that the batch carries no padding (CHROMO_F_DENSE: the ragged plan is not built; same results)."""
        def pick(d, b):
            return d[b] if b in d else d[str(b)]
        bs = self.binsizes
        return self._run([pick(batch["promoter_feats"], b) for b in bs], [pick(batch["promoter_pad_masks"], b) for b in bs],
                         [pick(batch["pcre_feats"], b) for b in bs], [pick(batch["pcre_pad_masks"], b) for b in bs],
                         [pick(batch["interaction_masks"], b) for b in bs], batch["interaction_freq"], dense=dense)

    def _run(self, x_p, mask_p, x_pcre, mask_pcre, imask, freq, dense=False):
        io = _BatchIO(self, x_p, mask_p, x_pcre, mask_pcre, imask, freq)
        inputs = list(x_p) + list(x_pcre) + [freq]
        if torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters()) or
                                        any(t.requires_grad for t in inputs)):
            return _ChromoFunction.apply(self._anchor, self, io, *inputs)
        logits, _ = self._launch_forward(io, self._precision_flag() | (_lib.F_DENSE if dense else 0))
        return logits


_DEFAULT_EMBED = {"n_layers": 1, "n_heads": 2, "d_model": 128, "d_ff": 128}
_DEFAULT_PAIRWISE = {"n_layers": 2, "n_heads": 2, "d_model": 128, "d_ff": 256}
_DEFAULT_REGULATION = {"n_layers": 6, "n_heads": 8, "d_model": 256, "d_ff": 256}


class ChromoformerBase(_ChromoformerCore):
    """Dict-keyed API of net.py:273-380 (``ChromoformerClassifier`` is an alias)."""

    n_out = 2

    def __init__(self, n_feats=7, d_emb=128, d_head=128, embed_kws=None, pairwise_interaction_kws=None,
                 regulation_kws=None, binsizes=(2000, 500, 100), seed=42, i_max=8, w_max=40000):
        super().__init__()
        torch.manual_seed(seed)
        embed_kws = dict(_DEFAULT_EMBED if embed_kws is None else embed_kws)
        pw_kws = dict(_DEFAULT_PAIRWISE if pairwise_interaction_kws is None else pairwise_interaction_kws)
        reg_kws = dict(_DEFAULT_REGULATION if regulation_kws is None else regulation_kws)
        # same argument plumbing as net.py:304-308
        embed_kws["n_feats"], embed_kws["d_model"] = n_feats, d_emb
        pw_kws["n_feats_p"], pw_kws["n_feats_pcre"] = embed_kws["d_model"], n_feats
        reg_kws["d_emb"] = d_emb
        self.binsizes = [int(b) for b in binsizes]     # CLI may hand strings (train.py:33)
        self.embed = nn.ModuleDict({str(b): EmbeddingTransformer(**embed_kws) for b in self.binsizes})
        self.pairwise_interaction = nn.ModuleDict(
            {str(b): PairwiseInteractionTransformer(**pw_kws) for b in self.binsizes})
        self.regulation = nn.ModuleDict({str(b): RegulationTransformer(**reg_kws) for b in self.binsizes})
        self.fc_head = nn.Sequential(nn.Linear(d_emb * 3, d_head), nn.ReLU(), nn.Linear(d_head, 2))
        self._head_hook(d_emb, d_head)
        self._finalise(n_feats, d_emb, d_head, self.n_out, embed_kws, pw_kws, reg_kws, self.binsizes, i_max, w_max)

    def _head_hook(self, d_emb, d_head):
        pass

    def _lib_name(self, name):
        parts = name.split(".")
        if parts[0] in ("embed", "pairwise_interaction", "regulation"):
            parts[1] = str(self.binsizes.index(int(parts[1])))
        return ".".join(parts)

    def forward(self, promoter_feats, promoter_pad_masks, pcre_feats, pcre_pad_masks, interaction_masks,
                interaction_freq):
        def pick(d, b):
            # DataLoader collation keys by int; tolerate str keys as well
            return d[b] if b in d else d[str(b)]
        bs = self.binsizes
        return self._run([pick(promoter_feats, b) for b in bs], [pick(promoter_pad_masks, b) for b in bs],
                         [pick(pcre_feats, b) for b in bs], [pick(pcre_pad_masks, b) for b in bs],
                         [pick(interaction_masks, b) for b in bs], interaction_freq)


ChromoformerClassifier = ChromoformerBase


class ChromoformerRegressor(ChromoformerBase):
    """net.py:386-428: the 2-logit head is built first (consuming RNG) and then replaced."""

    n_out = 1

    def _head_hook(self, d_emb, d_head):
        self.fc_head = nn.Sequential(nn.Linear(d_emb * 3, d_head), nn.ReLU(), nn.Linear(d_head, 1))


class Chromoformer(_ChromoformerCore):
    """Legacy flat API of net.py:156-270 (state_dict prefixes embed2000 / pw_int2000 / reg2000)."""

    _BINS = (2000, 500, 100)

    def __init__(self, n_feats=7, embed_n_layers=1, embed_n_heads=2, embed_d_model=128, embed_d_ff=128,
                 pw_int_n_layers=2, pw_int_n_heads=2, pw_int_d_model=128, pw_int_d_ff=256, reg_n_layers=6,
                 reg_n_heads=8, reg_d_model=256, reg_d_ff=256, head_n_feats=128, seed=42, i_max=8,
                 w_max=40000):
        super().__init__()
        torch.manual_seed(seed)
        self.binsizes = list(self._BINS)
        for b in self._BINS:
            setattr(self, f"embed{b}", EmbeddingTransformer(n_feats, embed_n_layers, embed_n_heads,
                                                            embed_d_model, embed_d_ff))
        for b in self._BINS:
            setattr(self, f"pw_int{b}", PairwiseInteractionTransformer(
                embed_d_model, n_feats, pw_int_n_layers, pw_int_n_heads, pw_int_d_model, pw_int_d_ff))
        for b in self._BINS:
            setattr(self, f"reg{b}", RegulationTransformer(reg_n_layers, reg_n_heads, embed_d_model,
                                                           reg_d_model, reg_d_ff))
        self.fc_head = nn.Sequential(nn.Linear(embed_d_model * 3, head_n_feats), nn.ReLU(),
                                     nn.Linear(head_n_feats, 2))
        self._finalise(
            n_feats, embed_d_model, head_n_feats, 2,
            {"n_layers": embed_n_layers, "n_heads": embed_n_heads, "d_model": embed_d_model, "d_ff": embed_d_ff},
            {"n_layers": pw_int_n_layers, "n_heads": pw_int_n_heads, "d_model": pw_int_d_model, "d_ff": pw_int_d_ff},
            {"n_layers": reg_n_layers, "n_heads": reg_n_heads, "d_model": reg_d_model, "d_ff": reg_d_ff},
            list(self._BINS), i_max, w_max)

    _PREFIX = {"embed": "embed", "pw_int": "pairwise_interaction", "reg": "regulation"}

    def _own_key(self, canon):
        for short, full in self._PREFIX.items():
            if canon.startswith(full + "."):
                res, rest = canon[len(full) + 1:].split(".", 1)
                return f"{short}{res}.{rest}"
        return canon

    def _lib_name(self, name):
        head, rest = name.split(".", 1)
        for short, full in self._PREFIX.items():
            if head.startswith(short) and head[len(short):].isdigit():
                return f"{full}.{self._BINS.index(int(head[len(short):]))}.{rest}"
        return name

    def forward(self, x_p_2000, pad_mask_p_2000, x_pcre_2000, pad_mask_pcre_2000, interaction_mask_2000,
                x_p_500, pad_mask_p_500, x_pcre_500, pad_mask_pcre_500, interaction_mask_500,
                x_p_100, pad_mask_p_100, x_pcre_100, pad_mask_pcre_100, interaction_mask_100,
                interaction_freq):
        return self._run([x_p_2000, x_p_500, x_p_100], [pad_mask_p_2000, pad_mask_p_500, pad_mask_p_100],
                         [x_pcre_2000, x_pcre_500, x_pcre_100],
                         [pad_mask_pcre_2000, pad_mask_pcre_500, pad_mask_pcre_100],
                         [interaction_mask_2000, interaction_mask_500, interaction_mask_100], interaction_freq)
