"""Autograd-facing loss functions and the fused optimizer of the mutual-learning step
(train.py:129-132,191-272), computed by the kernels of cmlpl_b200/csrc/losses.cu."""
from __future__ import annotations

import torch

from . import ops


class _CEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, probs, mask):
        loss, dz = ops.ce_fwd_bwd(logits.contiguous(), labels, probs, mask, 1.0, True)
        ctx.save_for_backward(dz)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dz,) = ctx.saved_tensors
        return dz * g, None, None, None


def cross_entropy(logits, labels):
    """torch.nn.CrossEntropyLoss()(logits, labels) (train.py:129,191)."""
    return _CEFn.apply(logits, labels.contiguous(), None, None)


def soft_cross_entropy(logits, probs, mask):
    """mean_i( -sum_c log_softmax(z)_ic * p_ic * mask_i ) with p, mask detached (train.py:239-242)."""
    return _CEFn.apply(logits, None, probs.detach().contiguous(), mask.detach().contiguous())


class _GraphContrastFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, f_row, f_col, p1, p, T, grad_side):
        loss, df = ops.graph_contrast(f_row.detach().contiguous(), f_col.detach().contiguous(), p1.contiguous(),
                                      p.contiguous(), T, grad_side, 1.0, True)
        ctx.save_for_backward(df)
        ctx.grad_side = grad_side
        return loss

    @staticmethod
    def backward(ctx, g):
        (df,) = ctx.saved_tensors
        if ctx.grad_side == 0:
            return df * g, None, None, None, None, None
        return None, df * g, None, None, None, None


def graph_contrast(f_row, f_col, probs1, probs, T, grad_side):
    """Pseudo-label-graph contrastive loss (train.py:246-265).  grad_side=0: gradient to the row
    features (loss_contrast); 1: to the column features (loss_contrast1).  The other operand and the
    pseudo-label probabilities are treated as constants, as in the reference (detach / no_grad)."""
    return _GraphContrastFn.apply(f_row, f_col, probs1.detach(), probs.detach(), float(T), int(grad_side))


_NORMALIZE_EPS = 1e-12                                # F.normalize's default eps


class _NTXentFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, emb_i, emb_j, T):
        bs = emb_i.size(0)
        x = torch.cat([emb_i, emb_j], 0).contiguous()
        z, norm = ops.l2norm(x, _NORMALIZE_EPS)       # F.normalize (models.py:23-24): a zero row stays finite
        loss, dz = ops.ntxent(z, bs, T, True)
        dx = ops.l2norm_bwd(z, norm, dz, _NORMALIZE_EPS)
        ctx.save_for_backward(dx)
        ctx.bs = bs
        return loss

    @staticmethod
    def backward(ctx, g):
        (dx,) = ctx.saved_tensors
        return dx[:ctx.bs] * g, dx[ctx.bs:] * g, None


def nt_xent(emb_i, emb_j, temperature=0.5):
    return _NTXentFn.apply(emb_i, emb_j, float(temperature))


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) with default betas/eps/no weight decay (train.py:131-132), all
    tensors of a group updated by one cmlpl_adam_multi_f32 launch per 16 tensors.  Parameters whose
    .grad is None are skipped exactly like torch does (feat_ss* in BaseNet2)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))

    @torch.no_grad()
    def step(self, closure=None):
        for group in self.param_groups:
            ps, gs, ms, vs = [], [], [], []
            step = None
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if not st:
                    st["step"] = 0
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                st["step"] += 1
                step = st["step"] if step is None else step
                if st["step"] != step:      # tensors that joined late get their own launch
                    ops.adam_multi([p], [p.grad.contiguous()], [st["exp_avg"]], [st["exp_avg_sq"]], group["lr"],
                                   *group["betas"], group["eps"], st["step"])
                    continue
                ps.append(p); gs.append(p.grad.contiguous()); ms.append(st["exp_avg"]); vs.append(st["exp_avg_sq"])
            if ps:
                ops.adam_multi(ps, gs, ms, vs, group["lr"], *group["betas"], group["eps"], step)
        # the kernel writes through raw pointers: bump the version counters ourselves so that everything keyed on
        # them (BaseNet2.packed_weights' cache, autograd's saved-tensor checks) sees the update
        touched = [p for group in self.param_groups for p in group["params"] if p.grad is not None]
        if touched:
            torch._C._increment_version(touched)        # takes an iterable of tensors
