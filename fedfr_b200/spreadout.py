"""``SpreadOut_Module`` (server.py:48-63) on the fused kernels.

The reference pushes the class centres of all clients apart with
``loss = sum_{i != j} relu(normalize(FC)_i . normalize(FC)_j - margin)^2`` (``mode='mean'``: the mean over the
N (N - 1) off-diagonal pairs) and runs a few SGD steps on ``FC`` (server.py:340-371).  It materialises the ``[N, N]``
similarity, its boolean mask and their autograd temporaries; here the similarity is a tcgen05 GEMM whose epilogue keeps
``H = relu(sim - margin)`` (bf16, off the diagonal) and sums ``H^2``, and the gradient ``4 H . w_hat`` is the dx GEMM on
that scratch.  Same constructor, attribute (``FC``) and ``forward()`` as the reference; there is no unfused fallback.
"""
import torch

from . import _native as N


class _SpreadOutLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, fc, margin, mean):
        if not fc.is_cuda or fc.dim() != 2:
            raise RuntimeError("fedfr_b200.SpreadOut_Module needs a 2-D CUDA tensor (sm_100); there is no CPU fallback")
        w = fc.detach().to(torch.float32).contiguous()
        n, emb = w.shape
        dev = w.device
        st = torch.cuda.current_stream(dev).cuda_stream
        w_hat = torch.empty((n, emb), dtype=torch.bfloat16, device=dev)
        inv_norm = torch.empty(n, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.pfc_normalize_rows(N.ptr(w), None, n, emb, N.ptr(w_hat), None, N.ptr(inv_norm), st), "pfc_normalize_rows")
            n_part = N.lib.pfc_spreadout_num_partials(n, emb)
            part = torch.empty((2, n_part, n), dtype=torch.float32, device=dev)
            hw = torch.empty((n, emb), dtype=torch.float32, device=dev)
            nbytes = N.lib.pfc_spreadout_workspace_bytes(n, emb)
            ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            off = (-ws.data_ptr()) % 1024
            N.check(N.lib.pfc_spreadout(N.ptr(w_hat), n, emb, float(margin), N.ptr(part[0]), N.ptr(part[1]), N.ptr(hw), ws.data_ptr() + off,
                                        ws.numel() - off, st), "pfc_spreadout")
        scale = 1.0 / (n * (n - 1)) if mean and n > 1 else 1.0
        loss = part[1].sum(dtype=torch.float64).to(torch.float32) * scale
        # d loss / d w_hat_i = 4 sum_j H_ij w_hat_j; normalize backward: (g - w_hat (w_hat . g)) / |w|
        w_unit = w * inv_norm[:, None]
        g = hw * (4.0 * scale)
        grad_fc = (g - w_unit * (w_unit * g).sum(dim=1, keepdim=True)) * inv_norm[:, None]
        ctx.save_for_backward(grad_fc)
        ctx.fc_dtype = fc.dtype
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (grad_fc,) = ctx.saved_tensors
        return (grad_fc * grad_out).to(ctx.fc_dtype), None, None


class SpreadOut_Module(torch.nn.Module):
    """Drop-in for server.py:48-63 (same constructor arguments; ``local`` is accepted and unused, as in the reference)."""

    def __init__(self, all_FC, margin=0.7, local=False, mode='sum'):
        super(SpreadOut_Module, self).__init__()
        self.FC = torch.nn.Parameter(all_FC)
        self.margin = margin
        self.mode = mode

    def forward(self):
        if self.mode not in ('sum', 'mean'):
            return None                                        # server.py:57-61 leaves `loss` as the relu tensor otherwise; not supported
        return _SpreadOutLoss.apply(self.FC, self.margin, self.mode == 'mean')
