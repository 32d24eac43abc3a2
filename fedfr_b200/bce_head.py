"""``BCE_module`` -- the cosine head of FedFR's personalised branch (client.py:25-60) on two fused sm_100a launches.

Same constructor, parameters (``converter.0.weight/bias``, ``weight``, ``bias`` -- so ``bce_module.pth``, client.py:485,
loads either way), ``forward(x, labels) -> (logits, gt)`` and ``initialize(fc)`` as the reference class.  The converter
(an identity-initialised ``nn.Linear``, client.py:30-34) stays a torch module; everything after it -- both
normalisations, the cosine matmul, ``g_func``, the +/- margin, ``r`` and the bias, and the matching backward -- is
``pfc_bce_head_fwd`` / ``pfc_bce_head_bwd`` (``csrc/bce_head.cu``).  The returned logits are an ordinary autograd tensor:
``losses.BCE_loss`` (losses.py:4-15), which edits them in place, works on them unchanged.  ``loss(x, labels)`` is that
loss fused into the head (``pfc_bce_loss_fwd`` / ``pfc_bce_loss_bwd``): the same value and gradients without the logits
and without a host synchronisation.  No CPU fallback.
"""
import torch
from torch import nn

from . import _native as N


class _CudaBceOps:
    def fwd(self, feat, weight, bias, labels, m, r, t):
        B, C, E = feat.shape[0], weight.shape[0], feat.shape[1]
        dev = feat.device
        logits = torch.empty((B, C), dtype=torch.float32, device=dev)
        gt = torch.empty((B, C), dtype=torch.uint8, device=dev)
        cosine = torch.empty((B, C), dtype=torch.float32, device=dev)
        inv_nf = torch.empty((B,), dtype=torch.float32, device=dev)
        inv_nw = torch.empty((C,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.pfc_bce_head_fwd(N.ptr(feat), N.ptr(weight), N.ptr(bias), N.ptr(labels), B, C, E, m, r, t,
                                           N.ptr(logits), N.ptr(gt), N.ptr(cosine), N.ptr(inv_nf), N.ptr(inv_nw),
                                           torch.cuda.current_stream(dev).cuda_stream), "pfc_bce_head_fwd")
        return logits, gt.bool(), cosine, inv_nf, inv_nw

    def bwd(self, feat, weight, cosine, inv_nf, inv_nw, dlogits, r, t, need_dfeat, need_dbias):
        B, C, E = feat.shape[0], weight.shape[0], feat.shape[1]
        dev = feat.device
        dfeat = torch.empty_like(feat) if need_dfeat else None
        dweight = torch.empty_like(weight)
        dbias = torch.empty((C,), dtype=torch.float32, device=dev) if need_dbias else None
        with torch.cuda.device(dev):
            N.check(N.lib.pfc_bce_head_bwd(N.ptr(feat), N.ptr(weight), N.ptr(cosine), N.ptr(inv_nf), N.ptr(inv_nw),
                                           N.ptr(dlogits), B, C, E, r, t, N.ptr(dfeat), N.ptr(dweight), N.ptr(dbias),
                                           torch.cuda.current_stream(dev).cuda_stream), "pfc_bce_head_bwd")
        return dfeat, dweight, dbias

    def loss_fwd(self, feat, weight, bias, labels, m, r, t, pos_coef, neg_coef):
        B, C, E = feat.shape[0], weight.shape[0], feat.shape[1]
        dev = feat.device
        loss = torch.empty((), dtype=torch.float32, device=dev)
        row_loss = torch.empty((B,), dtype=torch.float32, device=dev)
        cosine = torch.empty((B, C), dtype=torch.float32, device=dev)
        inv_nf = torch.empty((B,), dtype=torch.float32, device=dev)
        inv_nw = torch.empty((C,), dtype=torch.float32, device=dev)
        # a ticket of this call's own (one 4-byte memset on the stream, no host wait): a counter shared between calls
        # would be wrong for calls that overlap, such as a captured CUDA graph replayed beside eager calls
        ticket = torch.zeros((1,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.pfc_bce_loss_fwd(N.ptr(feat), N.ptr(weight), N.ptr(bias), N.ptr(labels), B, C, E, m, r, t, pos_coef,
                                           neg_coef, N.ptr(loss), N.ptr(row_loss), N.ptr(ticket), N.ptr(cosine), N.ptr(inv_nf),
                                           N.ptr(inv_nw), torch.cuda.current_stream(dev).cuda_stream), "pfc_bce_loss_fwd")
        return loss, cosine, inv_nf, inv_nw

    def loss_bwd(self, feat, weight, bias, labels, cosine, inv_nf, inv_nw, grad_out, m, r, t, pos_coef, neg_coef, need_dfeat,
                 need_dbias):
        B, C, E = feat.shape[0], weight.shape[0], feat.shape[1]
        dev = feat.device
        dfeat = torch.empty_like(feat) if need_dfeat else None
        dweight = torch.empty_like(weight)
        dbias = torch.empty((C,), dtype=torch.float32, device=dev) if need_dbias else None
        with torch.cuda.device(dev):
            N.check(N.lib.pfc_bce_loss_bwd(N.ptr(feat), N.ptr(weight), N.ptr(bias), N.ptr(labels), N.ptr(cosine), N.ptr(inv_nf),
                                           N.ptr(inv_nw), N.ptr(grad_out), B, C, E, m, r, t, pos_coef, neg_coef, N.ptr(dfeat),
                                           N.ptr(dweight), N.ptr(dbias), torch.cuda.current_stream(dev).cuda_stream),
                    "pfc_bce_loss_bwd")
        return dfeat, dweight, dbias


class _BceCosineHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, weight, bias, labels, m, r, t, ops):
        ops = _cuda_ops(ops, feat, weight, "BCE_module")
        f = feat.detach().to(torch.float32).contiguous()
        w = weight.detach().to(torch.float32).contiguous()
        b = None if bias is None else bias.detach().to(torch.float32).contiguous()
        y = labels.to(device=f.device, dtype=torch.long).contiguous()
        logits, gt, cosine, inv_nf, inv_nw = ops.fwd(f, w, b, y, float(m), float(r), float(t))
        ctx.save_for_backward(f, w, cosine, inv_nf, inv_nw)
        ctx.ops, ctx.r, ctx.t, ctx.has_bias = ops, float(r), float(t), bias is not None
        ctx.in_dtypes = (feat.dtype, weight.dtype, None if bias is None else bias.dtype)
        ctx.mark_non_differentiable(gt)
        return logits, gt

    @staticmethod
    def backward(ctx, dlogits, _dgt):
        f, w, cosine, inv_nf, inv_nw = ctx.saved_tensors
        need_f, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        dfeat, dweight, dbias = ctx.ops.bwd(f, w, cosine, inv_nf, inv_nw, dlogits.to(torch.float32).contiguous(), ctx.r, ctx.t,
                                            need_f, need_b)
        df = dfeat.to(ctx.in_dtypes[0]) if need_f else None
        dw = dweight.to(ctx.in_dtypes[1]) if need_w else None
        db = dbias.to(ctx.in_dtypes[2]) if need_b else None
        return df, dw, db, None, None, None, None, None


def _cuda_ops(ops, feat, weight, who):
    if ops is not None:
        return ops
    if not (feat.is_cuda and weight.is_cuda):
        raise RuntimeError("fedfr_b200.%s needs CUDA tensors on an sm_100 device (no CPU fallback)" % who)
    return _CudaBceOps()


class _BceLoss(torch.autograd.Function):
    """losses.BCE_loss()(*BCE_module.forward(feat, labels)) as one forward and one backward launch, without the logits."""

    @staticmethod
    def forward(ctx, feat, weight, bias, labels, m, r, t, pos_coef, neg_coef, ops):
        ops = _cuda_ops(ops, feat, weight, "BCE_module.loss")
        f = feat.detach().to(torch.float32).contiguous()
        w = weight.detach().to(torch.float32).contiguous()
        b = None if bias is None else bias.detach().to(torch.float32).contiguous()
        y = labels.to(device=f.device, dtype=torch.long).contiguous()
        loss, cosine, inv_nf, inv_nw = ops.loss_fwd(f, w, b, y, m, r, t, pos_coef, neg_coef)
        ctx.save_for_backward(f, w, b, y, cosine, inv_nf, inv_nw)
        ctx.ops, ctx.consts = ops, (m, r, t, pos_coef, neg_coef)
        ctx.in_dtypes = (feat.dtype, weight.dtype, None if bias is None else bias.dtype)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        f, w, b, y, cosine, inv_nf, inv_nw = ctx.saved_tensors
        need_f, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], b is not None and ctx.needs_input_grad[2]
        dfeat, dweight, dbias = ctx.ops.loss_bwd(f, w, b, y, cosine, inv_nf, inv_nw, dloss.to(torch.float32).contiguous(),
                                                 *ctx.consts, need_f, need_b)
        df = dfeat.to(ctx.in_dtypes[0]) if need_f else None
        dw = dweight.to(ctx.in_dtypes[1]) if need_w else None
        db = dbias.to(ctx.in_dtypes[2]) if need_b else None
        return df, dw, db, None, None, None, None, None, None, None


class BCE_module(nn.Module):
    def __init__(self, hidden, n_class, converter_layer=1, m=0.4, r=30.0, t=3, converter=None, _ops=None):
        super(BCE_module, self).__init__()
        if converter is not None:
            self.converter = converter
        elif converter_layer == 1:          # client.py:30-35
            layer = nn.Linear(hidden, hidden)
            nn.init.eye_(layer.weight)
            nn.init.constant_(layer.bias, 0.0)
            self.converter = nn.Sequential(layer)
        else:                               # client.py:36-37 uses backbones.BottleBlock(hidden, 4): pass it as `converter`
            raise NotImplementedError("converter_layer != 1: pass the reference's BottleBlock as converter=")
        self.weight = nn.Parameter(torch.normal(0, 0.01, (n_class, hidden)))
        self.bias = nn.Parameter(torch.zeros(n_class))
        self.g_func = lambda x: (2 * (((x + 1) / 2).pow(t)) - 1)       # kept for callers that read it (client.py:40)
        self.n_class = n_class
        self.hidden = hidden
        self.m = m
        self.r = r
        self.t = t
        self._ops = _ops

    def forward(self, x, labels):
        feat = self.converter(x)
        return _BceCosineHead.apply(feat, self.weight, self.bias, labels, self.m, self.r, self.t, self._ops)

    def loss(self, x, labels, lam=0.7, r_loss=30.0):
        """``losses.BCE_loss(lam, r_loss)(*self(x, labels))`` (losses.py:4-15) as a 0-d fp32 tensor, fused into the head:
        no [B, C] logits, and neither the forward nor the backward waits for the device.  ``r_loss`` is the loss's own
        scale, not the head's ``r``.  client.py:382,393 become ``10 * bce_module.loss(feat, labels)``."""
        feat = self.converter(x)
        return _BceLoss.apply(feat, self.weight, self.bias, labels, float(self.m), float(self.r), float(self.t),
                              lam / r_loss, (1 - lam) / r_loss, self._ops)

    def initialize(self, fc):
        self.weight.data = fc.clone()
