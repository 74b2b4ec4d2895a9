"""Drop-in for the reference's ``roko/rnn_model.py``: same public names, same constructor,
same 31 parameter names/shapes (so ``.pth`` files interchange), but ``forward`` runs the
hand-written sm_100a kernels of ``libroko_b200.so`` through its C ABI instead of torch ops.

Reference interface mirrored here (file:line in /root/reference):
  * constants ``IN_SIZE, HIDDEN_SIZE, NUM_LAYERS``                     roko/rnn_model.py:10-12
  * ``gru_init``  (orthogonal matrices, N(0,1) biases)                 roko/rnn_model.py:15-21
  * ``RNN(in_size, hidden_size, num_layers, dropout=0.2)``             roko/rnn_model.py:24-44
  * ``RNN.forward(x) -> (B, 90, 5)`` fp32 logits                        roko/rnn_model.py:46-59
  * callers do ``from rnn_model import *`` and use ``nn`` / ``F``       roko/inference.py:9, train.py:10

``forward`` is differentiable: in train mode (dropout active) or whenever autograd needs parameter
gradients it runs the training kernels with a hand-written backward (roko/train.py:46-53).

Additions (not in the reference): ``predict`` (fused argmax, uint8 labels), ``predict_host``
(pipelined host-buffer loop), ``forward_taps`` (stage outputs for parity tests),
``dropout_masks`` (the training kernels' keep-masks, for tests).

There is no CPU path: a CPU tensor, a missing library or a non-sm_100 device raise.
"""
import ctypes
import math  # noqa: F401  (re-exported: the reference's callers star-import this module)

import numpy as np  # noqa: F401
import torch
import torch.nn as nn
import torch.nn.functional as F  # noqa: F401
import torch.nn.init as init

from . import _cabi

IN_SIZE = 500
HIDDEN_SIZE = 128
NUM_LAYERS = 3

READS, COLS, CLASSES = 200, 90, 5
MAX_CHUNK = 2368          # windows per internal chunk = 148 SMs x 16 (bounds scratch: 0.66 MB / window)
MAX_TRAIN_BATCH = 1024    # windows per training forward/backward (4.7 MB of saved activations each)


def gru_init(gru):
    """Initialisation the reference applies to its GRU (roko/rnn_model.py:15-21).

    Written through the parameter itself under ``no_grad`` (not ``p.data``) so the in-place update bumps
    the tensor version the packed-weight cache watches."""
    with torch.no_grad():
        for p in gru.parameters():
            if p.dim() >= 2:
                init.orthogonal_(p)
            else:
                init.normal_(p)


def state_keys():
    keys = ["embedding.weight", "fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias"]
    for layer in range(NUM_LAYERS):
        for sfx in ("", "_reverse"):
            keys += [f"gru.{kind}_l{layer}{sfx}" for kind in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    return keys + ["fc4.weight", "fc4.bias"]


class _Handle:
    """Owns one roko_b200_model (packed weights on one device)."""

    def __init__(self, device_index):
        self.lib = _cabi.lib()
        self.ptr = _cabi.c_model_p()
        _cabi.check(self.lib.roko_b200_model_create(ctypes.byref(self.ptr), device_index))
        self.device_index = device_index
        self.version = None          # (weights epoch, sum of tensor versions, first data_ptr) the packed copy was made from
        self.workspaces = {}

    def __del__(self):
        try:
            if self.ptr:
                self.lib.roko_b200_model_destroy(self.ptr)
                self.ptr = None
        except Exception:
            pass


DROPOUT_SITES = {"emb": (READS, COLS, 50), "fc1": (COLS, 50, 100), "fc2": (COLS, 50, 10),
                 "gru0": (COLS, 2 * HIDDEN_SIZE), "gru1": (COLS, 2 * HIDDEN_SIZE)}


def dropout_masks(p_drop, seed, batch, device):
    """Keep-masks (uint8, 1 = kept) the training kernels derive from ``seed`` for a batch, one per
    dropout site, shaped like the reference tensor each site masks (roko/rnn_model.py:47,51,54,57)."""
    lib = _cabi.lib()
    dev = torch.device(device)
    stream = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    with torch.cuda.device(dev):
        for site, (name, shape) in enumerate(DROPOUT_SITES.items()):
            m = torch.empty((batch,) + shape, dtype=torch.uint8, device=dev)
            _cabi.check(lib.roko_b200_dropout_mask(float(p_drop), int(seed), site, m.numel(), m.data_ptr(), stream))
            out[name] = m
    return out


class _TrainFn(torch.autograd.Function):
    """Train-mode forward / backward of the whole network as two C-ABI calls.

    The parameters are inputs of the Function, so autograd routes the gradients the library
    writes (one flat fp32 buffer in state_dict order) to ``param.grad`` like any other op --
    optimisers, ``zero_grad`` and DDP's gradient hooks work unchanged.
    """

    @staticmethod
    def forward(ctx, module, x8, p_drop, seed, *params):
        h = module._handle(x8.device, force=module.training)     # train mode: always re-pack (``.data`` writes are invisible)
        n, idx = x8.shape[0], h.device_index
        stream = torch.cuda.current_stream(idx).cuda_stream
        tws = torch.empty(h.lib.roko_b200_train_workspace_bytes(n), dtype=torch.uint8, device=x8.device)
        logits = torch.empty((n, COLS, CLASSES), dtype=torch.float32, device=x8.device)
        _cabi.check(h.lib.roko_b200_train_forward(h.ptr, x8.data_ptr(), n, p_drop, seed, logits.data_ptr(),
                                                  tws.data_ptr(), tws.numel(), stream))
        ctx.h, ctx.x8, ctx.p_drop, ctx.seed, ctx.tws, ctx.version = h, x8, p_drop, seed, tws, h.version
        ctx.shapes = [tuple(q.shape) for q in params]
        return logits

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dlogits):
        h = ctx.h
        if ctx.tws is None:
            raise RuntimeError("roko_b200: backward through the same forward twice (the saved activations "
                               "are consumed by the first backward)")
        if h.version != ctx.version:
            raise RuntimeError("roko_b200: parameters changed between forward and backward")
        n, idx = ctx.x8.shape[0], h.device_index
        dlogits = dlogits.to(torch.float32).contiguous()
        stream = torch.cuda.current_stream(idx).cuda_stream
        grad_raw = torch.empty(h.lib.roko_b200_raw_weight_count(), dtype=torch.float32, device=dlogits.device)
        _cabi.check(h.lib.roko_b200_train_backward(h.ptr, ctx.x8.data_ptr(), n, ctx.p_drop, ctx.seed,
                                                   dlogits.data_ptr(), grad_raw.data_ptr(), ctx.tws.data_ptr(),
                                                   ctx.tws.numel(), stream))
        ctx.tws = None
        grads, off = [], 0
        for shape in ctx.shapes:
            k = math.prod(shape)
            grads.append(grad_raw[off:off + k].view(shape))
            off += k
        return (None, None, None, None, *grads)


class RNN(nn.Module):
    def __init__(self, in_size, hidden_size, num_layers, dropout=0.2):
        super().__init__()
        if (in_size, hidden_size, num_layers) != (IN_SIZE, HIDDEN_SIZE, NUM_LAYERS):
            raise ValueError("roko_b200 kernels are specialised for RNN(500, 128, 3) "
                             f"(roko/rnn_model.py:10-12); got {(in_size, hidden_size, num_layers)}")
        # construction order matches the reference so a given torch seed yields the same weights
        self.embedding = nn.Embedding(12, 50)
        self.do = nn.Dropout(dropout)
        self.fc1 = nn.Linear(READS, 100)
        self.do1 = nn.Dropout(dropout)
        self.fc2 = nn.Linear(100, 10)
        self.do2 = nn.Dropout(dropout)
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.gru = nn.GRU(in_size, hidden_size, num_layers=num_layers, batch_first=True,
                          bidirectional=True, dropout=dropout)
        gru_init(self.gru)
        self.fc4 = nn.Linear(2 * hidden_size, CLASSES)
        self._handles = {}

    # the C handles (device pointers) are a derived cache: never copied or pickled with the module
    def __getstate__(self):
        state = self.__dict__.copy()
        state["_handles"] = {}
        state.pop("_param_list", None)
        return state

    # ---- packed-weight cache ------------------------------------------------------------------
    # The kernels read a packed copy of the 31 tensors.  It is rebuilt when (a) any parameter's autograd
    # version counter moved (optimizer steps, ``copy_``, ``load_state_dict``, in-place init under no_grad),
    # (b) the module was moved/cast (``_apply``) or (c) ``invalidate()`` was called.  The one thing torch
    # does not count is a write through ``param.data`` (``p.data.add_(..)``, ``init.*_(p.data)``): code that
    # edits weights that way must call ``model.invalidate()`` before the next forward.  In train mode the
    # copy is refreshed on every forward regardless, so optimisers that write through ``.data`` are safe.
    def _ordered_params(self):
        ps = self.__dict__.get("_param_list")
        if ps is None:
            sd = dict(self.named_parameters())
            ps = [sd[k] for k in state_keys()]
            self.__dict__["_param_list"] = ps
        return ps

    def invalidate(self):
        """Force the next forward to re-pack the weights (needed after writes through ``param.data``)."""
        self.__dict__["_weights_epoch"] = self.__dict__.get("_weights_epoch", 0) + 1
        self.__dict__.pop("_param_list", None)

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.invalidate()
        return out

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate()
        return out

    def _handle(self, device, force=False):
        if device.type != "cuda":
            raise RuntimeError("roko_b200.RNN runs on CUDA (sm_100a) only; there is no CPU fallback. "
                               "Move the module and the input to a B200: model.to('cuda')")
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            h = self._handles[idx] = _Handle(idx)
        params = self._ordered_params()
        version = (self.__dict__.get("_weights_epoch", 0), sum([p._version for p in params]), params[0].data_ptr())
        if force or h.version != version:
            for p in params:
                if p.device.type != "cuda" or (p.device.index or 0) != idx:
                    raise RuntimeError(f"parameter on {p.device}, input on cuda:{idx}")
            with torch.no_grad():
                raw = torch.cat([p.detach().reshape(-1).to(torch.float32) for p in params]).contiguous()
            assert raw.numel() == h.lib.roko_b200_raw_weight_count()
            stream = torch.cuda.current_stream(idx).cuda_stream
            # inference loads synchronise (forwards may follow on other streams); the per-step reload of the
            # training path stays asynchronous on the training stream (flag bit 1)
            _cabi.check(h.lib.roko_b200_model_load(h.ptr, raw.data_ptr(), 3 if force else 1, stream))
            h.version = version
        return h

    @staticmethod
    def _workspace(h, n, idx, stream):
        need = h.lib.roko_b200_workspace_bytes(min(n, MAX_CHUNK))
        ws = h.workspaces.get(stream)
        if ws is None or ws.numel() < need:
            ws = h.workspaces[stream] = torch.empty(need, dtype=torch.uint8, device=f"cuda:{idx}")
        return ws

    @staticmethod
    def _check_input(x):
        if x.dim() != 3 or x.shape[1] != READS or x.shape[2] != COLS:
            raise RuntimeError(f"expected input of shape (B, {READS}, {COLS}), got {tuple(x.shape)}")
        if x.dtype not in (torch.uint8, torch.int64):
            raise RuntimeError(f"expected uint8 or int64 codes, got {x.dtype}")
        return x.contiguous()

    def _run(self, x, want_logits, want_labels, labels_out=None):
        x = self._check_input(x)
        h = self._handle(x.device)
        idx = h.device_index
        n = x.shape[0]
        logits = torch.empty((n, COLS, CLASSES), dtype=torch.float32, device=x.device) if want_logits else None
        labels = None
        if want_labels:
            labels = labels_out if labels_out is not None else \
                torch.empty((n, COLS), dtype=torch.uint8, device=x.device)
            if (labels.dtype != torch.uint8 or tuple(labels.shape) != (n, COLS) or not labels.is_contiguous()
                    or labels.device != x.device):
                raise RuntimeError("labels_out must be a contiguous uint8 (B, 90) tensor on the input's device")
        if n == 0:
            return logits, labels
        stream = torch.cuda.current_stream(idx).cuda_stream
        ws = self._workspace(h, n, idx, stream)
        fn = h.lib.roko_b200_forward_u8 if x.dtype == torch.uint8 else h.lib.roko_b200_forward_i64
        _cabi.check(fn(h.ptr, x.data_ptr(), n, logits.data_ptr() if want_logits else None,
                       labels.data_ptr() if want_labels else None, ws.data_ptr(), ws.numel(), stream))
        return logits, labels

    # ---- reference interface ------------------------------------------------------------------
    def forward(self, x):
        """``(B,200,90)`` uint8|int64 codes 0..11 on a CUDA device -> ``(B,90,5)`` fp32 logits.

        Inference (eval mode, nothing to differentiate) runs the fused inference kernels.  In train mode,
        or whenever autograd is recording and a parameter requires grad, it runs the training kernels:
        the same network with the four dropout sites of roko/rnn_model.py:29,32,35,41 active (train mode)
        and a hand-written backward behind ``torch.autograd`` (roko/train.py:46-53).
        """
        differentiate = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        if not self.training and not differentiate:
            return self._run(x, True, False)[0]
        return self._train_forward(x)

    def _dropout_p(self):
        ps = {float(self.do.p), float(self.do1.p), float(self.do2.p), float(self.gru.dropout)}
        if len(ps) != 1:
            raise RuntimeError("roko_b200 kernels use one dropout probability for all four sites "
                               f"(roko/rnn_model.py:25 passes a single `dropout`); got {sorted(ps)}")
        return ps.pop() if self.training else 0.0

    def _train_forward(self, x, seed=None):
        x = self._check_input(x)
        if x.dtype != torch.uint8:
            if x.numel() and (int(x.min()) < 0 or int(x.max()) > 11):      # a wrapping cast would hide e.g. 256 -> 0
                raise IndexError("index out of range in embedding: pileup codes must be 0..11")
            x = x.to(torch.uint8)
        if x.shape[0] == 0:
            return torch.zeros((0, COLS, CLASSES), dtype=torch.float32, device=x.device)
        if x.shape[0] > MAX_TRAIN_BATCH:
            raise RuntimeError(f"training batches hold at most {MAX_TRAIN_BATCH} windows (got {x.shape[0]})")
        if seed is None:                      # drawn from torch's CPU generator: torch.manual_seed reproduces a run
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        return _TrainFn.apply(self, x, self._dropout_p(), int(seed), *self._ordered_params())

    # ---- additions ----------------------------------------------------------------------------
    @torch.no_grad()
    def predict(self, x, return_logits=False, out=None):
        """Fused ``argmax(model(x), 2)`` (roko/inference.py:115-116): uint8 labels ``(B,90)``."""
        logits, labels = self._run(x, return_logits, True, out)
        return (labels, logits) if return_logits else labels

    @torch.no_grad()
    def predict_host(self, x_host, batch=128, out=None, logits_out=None, device=None):
        """The loop body of roko/inference.py:111-117 over HOST windows.

        ``x_host``: CPU uint8 tensor ``(N,200,90)`` (pinned memory makes the copies async).
        Returns CPU uint8 labels ``(N,90)``; copies in/out are inside the call.
        """
        if x_host.device.type != "cpu" or x_host.dtype != torch.uint8:
            raise RuntimeError("predict_host expects a CPU uint8 tensor")
        x_host = self._check_input(x_host)
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        h = self._handle(dev)
        n = x_host.shape[0]
        if out is None:
            out = torch.empty((n, COLS), dtype=torch.uint8, pin_memory=True)
        _cabi.check(h.lib.roko_b200_infer_host(h.ptr, x_host.data_ptr(), n, int(batch), out.data_ptr(),
                                               logits_out.data_ptr() if logits_out is not None else None))
        return out

    @torch.no_grad()
    def forward_taps(self, x):
        """Stage outputs for parity tests: dict(front, gru_l0..2, logits, labels)."""
        x = self._check_input(x)
        if x.dtype != torch.uint8:
            x = x.to(torch.uint8)
        h = self._handle(x.device)
        idx, n = h.device_index, x.shape[0]
        f32 = dict(dtype=torch.float32, device=x.device)
        t = {"front": torch.empty((n, COLS, IN_SIZE), **f32), "logits": torch.empty((n, COLS, CLASSES), **f32),
             "labels": torch.empty((n, COLS), dtype=torch.uint8, device=x.device)}
        for layer in range(NUM_LAYERS):
            t[f"gru_l{layer}"] = torch.empty((n, COLS, 2 * HIDDEN_SIZE), **f32)
        stream = torch.cuda.current_stream(idx).cuda_stream
        need = h.lib.roko_b200_workspace_bytes(n)
        ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        _cabi.check(h.lib.roko_b200_forward_taps(
            h.ptr, x.data_ptr(), n, t["front"].data_ptr(), t["gru_l0"].data_ptr(), t["gru_l1"].data_ptr(),
            t["gru_l2"].data_ptr(), t["logits"].data_ptr(), t["labels"].data_ptr(), ws.data_ptr(), ws.numel(), stream))
        torch.cuda.current_stream(idx).synchronize()
        return t

    def set_option(self, name, value, device=None):
        """Scheduling / kernel-selection knobs of the C library (see include/roko_b200.h): rec_tc_min, superbatch,
        proj (0 ffma, 3 tf32, 4 fp16), rec (1 tf32, 2 fp16), front (0 mma.sync, 1 tcgen05), graphs (0/1), geometry (0 full-chip,
        1 work-sized grids) and its minima geo_front / geo_proj / geo_head."""
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        h = self._handle(dev)
        _cabi.check(h.lib.roko_b200_model_set_option(h.ptr, name.encode(), int(value)))

    def check_codes(self):
        """Synchronise and raise IndexError if an earlier forward saw a code outside 0..11 (RokoB200Error if a
        weight or activation left the range of the fp16-split kernels)."""
        for h in self._handles.values():
            _cabi.check(h.lib.roko_b200_model_check(h.ptr))
