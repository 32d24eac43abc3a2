"""Closed-form fp64 restatement of the fused BCE loss (include/fedfr_b200.h ``pfc_bce_loss_fwd`` / ``pfc_bce_loss_bwd``):
``losses.BCE_loss`` (losses.py:4-15) on the logits of ``client.BCE_module`` and its derivative, without autograd.  The
head itself (cosine, logits, gt, the backward from d logit) is ``oracle/bce_head_oracle.py``; this file adds the loss on
top and a CPU stand-in for the module's fused ops (host-logic tests only)."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import bce_head_oracle as O  # noqa: E402
from oracle.bce_head_oracle import OracleBceOps  # noqa: E402

FLT_MAX = float(np.finfo(np.float32).max)


def coefs(lam=0.7, r_loss=30.0):
    """(pos_coef, neg_coef): the Python doubles lam / r_loss and (1 - lam) / r_loss, rounded once to fp32 as torch rounds
    a scalar factor of an fp32 tensor."""
    return float(np.float32(lam / r_loss)), float(np.float32((1 - lam) / r_loss))


def reference_bce_loss(logits, gts, lam=0.7, r=30.0):
    """losses.py:4-15 as written: in-place edits through the boolean masks, each mask evaluating only its own branch
    (a ``torch.where`` of both branches would leak the other branch's overflow into the gradient as NaN)."""
    logits = logits.clone()
    logits[gts] = (lam / r) * torch.log(1 + torch.exp(-1 * logits[gts]) + 1e-8)
    logits[~gts] = ((1 - lam) / r) * torch.log(1 + torch.exp(1 * logits[~gts]) + 1e-8)
    return torch.mean(torch.sum(logits, dim=1))


def _exp32(x):
    """exp in fp64, except that a value beyond fp32's range is inf: the reference's fp32 exp overflows at |x| ~ 88.7."""
    e = torch.exp(x)
    return torch.where(e > FLT_MAX, torch.full_like(e, float("inf")), e)


def loss_from_logits(z, gt, pos_coef, neg_coef, grad_out=1.0):
    """-> (loss, row_loss [B], d loss / d z [B, C] scaled by grad_out).
    term = gt ? pc log((1 + exp(-z)) + 1e-8) : nc log((1 + exp(z)) + 1e-8);  loss = mean_b sum_c term;
    d term / d z = gt ? -pc exp(-z) / ((1 + exp(-z)) + 1e-8) : nc exp(z) / ((1 + exp(z)) + 1e-8)."""
    pc, nc = (float(np.float32(c)) for c in (pos_coef, neg_coef))
    z = z.double()
    e = _exp32(torch.where(gt, -z, z))
    x = (1 + e) + 1e-8
    term = torch.where(gt, pc, nc).double() * torch.log(x)          # fp32 coefficients, exact in either dtype
    dterm = torch.where(gt, -pc, nc).double() * e / x
    row = term.sum(dim=1)
    B = z.shape[0]
    loss = row.sum() / B if B else torch.tensor(float("nan"), dtype=torch.float64)
    dz = (torch.as_tensor(grad_out, dtype=torch.float64) / max(B, 1)) * dterm
    return loss, row, dz


def restate(feat, weight, bias, labels, m, r, t, pos_coef, neg_coef, grad_out=1.0):
    """The whole fused loss from the head's inputs, in the inputs' dtype (pass fp64):
    {loss, row_loss, dz, logits, gt, cosine, inv_nf, inv_nw, dfeat, dweight, dbias}."""
    logits, gt, cosine, nf, nw = O.forward(feat, weight, bias, labels, m, r, t)
    loss, row, dz = loss_from_logits(logits, gt, pos_coef, neg_coef, grad_out)
    dfeat, dweight, dbias = O.backward(feat, weight, cosine, nf, nw, dz, r, t)
    return {"loss": loss, "row_loss": row, "dz": dz, "logits": logits, "gt": gt, "cosine": cosine, "inv_nf": 1.0 / nf,
            "inv_nw": 1.0 / nw, "dfeat": dfeat, "dweight": dweight, "dbias": dbias}


class OracleBceLossOps(OracleBceOps):
    """CPU stand-in for fedfr_b200.bce_head._CudaBceOps, the fused loss included.  ``calls`` records the backward's
    need_dfeat / need_dbias flags."""

    def __init__(self):
        self.calls = []

    def loss_fwd(self, feat, weight, bias, labels, m, r, t, pos_coef, neg_coef):
        logits, gt, cosine, nf, nw = O.forward(feat, weight, bias, labels, m, r, t)
        loss, _, _ = loss_from_logits(logits, gt, pos_coef, neg_coef)
        return loss.to(feat.dtype), cosine, 1.0 / nf, 1.0 / nw

    def loss_bwd(self, feat, weight, bias, labels, cosine, inv_nf, inv_nw, grad_out, m, r, t, pos_coef, neg_coef, need_dfeat,
                 need_dbias):
        self.calls.append((need_dfeat, need_dbias))
        logits, gt, _, _, _ = O.forward(feat, weight, bias, labels, m, r, t)
        _, _, dz = loss_from_logits(logits, gt, pos_coef, neg_coef, grad_out)
        dfeat, dweight, dbias = O.backward(feat, weight, cosine, 1.0 / inv_nf, 1.0 / inv_nw, dz.to(feat.dtype), r, t)
        return (dfeat if need_dfeat else None), dweight, (dbias if need_dbias else None)
