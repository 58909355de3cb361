"""The loss on logits, restated in float64 on top of the restatement of oracle/ppn_loss.py.  TEST INFRASTRUCTURE.

The head the loss sees is s = sigmoid(x) of every channel of the logits x (model.py:133-136).  ``loss_terms`` applies
a float64 sigmoid and then the restated loss, so the kernels' terms on logits are held to the same float64
specification as on the sigmoid output.  ``grad_logits`` is the gradient the kernels form, written out as they form
it: the float64 gradient with respect to s, times (1 - s), times s.  A CPU test holds it to torch autograd through
torch.sigmoid.
"""
from __future__ import annotations

import torch

from oracle import ppn_loss as L


def loss_terms(logits, *targets, cfg):
    """(L_resp, L_iou, L_coor, L_size, L_limb) of sigmoid(logits), in float64; targets in the criterion's order."""
    return L.loss_terms(torch.sigmoid(logits.double()), *[t.double() for t in targets], cfg)


def grad_logits(logits, targets, cfg, grad_loss):
    """d(sum_t grad_loss[t] * L_t)/d(logits) in float64 by the chain rule: (dL/ds * (1 - s)) * s."""
    s = torch.sigmoid(logits.detach().double())
    return (L.autograd_grad(s, targets, cfg, grad_loss) * (1 - s)) * s


def terms_chunked(cfg, logits, targets, chunk=None):
    """loss_terms over the batch chunk by chunk (sum of chunk means * chunk size / B), as a numpy float64 [5]."""
    B = logits.shape[0]
    chunk = chunk or B
    acc = torch.zeros(5, dtype=torch.float64, device=logits.device)
    for b0 in range(0, B, chunk):
        sl = slice(b0, min(B, b0 + chunk))
        acc += torch.stack(loss_terms(logits[sl], *[t[sl] for t in targets], cfg=cfg)) * (sl.stop - sl.start)
    return (acc / B).cpu().numpy()
