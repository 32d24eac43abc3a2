"""CPU oracle for the cosine head of FedFR's personalised branch  --  TEST INFRASTRUCTURE ONLY (see partial_fc_oracle.py).

Closed-form restatement (no autograd) of ``client.BCE_module.forward`` after its converter (client.py:47-58) and of the
gradient autograd derives for it.  Pinned by ``tests/golden/bce_head.npz``: the unmodified reference classes
(``client.BCE_module`` + ``losses.BCE_loss``, losses.py:4-15) run on CPU with ``loss.backward()``
(``tests/golden/make_golden.py bce``).
"""
import torch

EPS = 1e-12     # F.normalize default, client.py:47


def target_col(labels, n_class):
    """Column picked by ``gt[arange, tmp_labels]`` on the [B, n_class + 1] matrix whose last column is dropped
    (client.py:48-52): labels >= n_class and -1 pick nothing; other negatives index from the end."""
    col = labels.clone()
    col[col >= n_class] = n_class
    col = torch.where(col < 0, col + n_class + 1, col)
    col[(col < 0) | (col >= n_class)] = -1
    return col


def forward(feat, weight, bias, labels, m, r, t):
    """-> logits [B, C], gt bool [B, C], cosine [B, C], |feat| [B], |weight| [C]  (computed in feat's dtype)."""
    nf = feat.norm(dim=1).clamp_min(EPS)
    nw = weight.norm(dim=1).clamp_min(EPS)
    cosine = (feat / nf[:, None]) @ (weight / nw[:, None]).t()          # client.py:47
    col = target_col(labels, weight.shape[0])
    gt = torch.zeros_like(cosine, dtype=torch.bool)
    rows = torch.nonzero(col >= 0, as_tuple=True)[0]
    gt[rows, col[rows]] = True                                           # client.py:48-52
    g = 2 * ((cosine + 1) / 2).clamp_min(0).pow(t) - 1                   # client.py:40 (an antipodal pair may round below -1)
    logits = torch.where(gt, r * (g - m), r * (g + m))                   # client.py:54,56
    if bias is not None:
        logits = logits + bias[None, :]                                  # client.py:57
    return logits, gt, cosine, nf, nw


def backward(feat, weight, cosine, nf, nw, dlogits, r, t):
    """d loss / d (feat, weight, bias) given d loss / d logits."""
    dcos = dlogits * (r * t) * ((cosine + 1) / 2).clamp_min(0).pow(t - 1)
    f_hat, w_hat = feat / nf[:, None], weight / nw[:, None]
    df_hat, dw_hat = dcos @ w_hat, dcos.t() @ f_hat
    # a norm clamped to EPS is a constant: autograd of F.normalize gives such a row no radial term
    f_rad = torch.where(nf[:, None] > EPS, f_hat, torch.zeros_like(f_hat))
    w_rad = torch.where(nw[:, None] > EPS, w_hat, torch.zeros_like(w_hat))
    dfeat = (df_hat - f_rad * (f_hat * df_hat).sum(dim=1, keepdim=True)) / nf[:, None]
    dweight = (dw_hat - w_rad * (w_hat * dw_hat).sum(dim=1, keepdim=True)) / nw[:, None]
    return dfeat, dweight, dlogits.sum(dim=0)


class OracleBceOps:
    """CPU stand-in for fedfr_b200.bce_head._CudaBceOps (host-logic tests only)."""

    def fwd(self, feat, weight, bias, labels, m, r, t):
        logits, gt, cosine, nf, nw = forward(feat, weight, bias, labels, m, r, t)
        return logits, gt, cosine, 1.0 / nf, 1.0 / nw

    def bwd(self, feat, weight, cosine, inv_nf, inv_nw, dlogits, r, t, need_dfeat, need_dbias):
        dfeat, dweight, dbias = backward(feat, weight, cosine, 1.0 / inv_nf, 1.0 / inv_nw, dlogits, r, t)
        return (dfeat if need_dfeat else None), dweight, (dbias if need_dbias else None)
