"""Stage-2 evaluation heads on graph embeddings (K12; SURVEY 8f n4): the kNN classifier of `evaluate` and the
one-sample-per-step MLP of `evaluate_mlp` (Code/sage+gat+diffpool/train_triplet.py:80-85, 148-180)."""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from ._lib import call, ptr, stream_ptr


def knn_predict(train_emb: torch.Tensor, train_labels: torch.Tensor, query_emb: torch.Tensor, k: int = 3,
                num_classes: Optional[int] = None) -> torch.Tensor:
    """KNeighborsClassifier(n_neighbors=k).fit(train).predict(query): int64 [Q]."""
    return knn_classify(train_emb, train_labels, query_emb, k=k, num_classes=num_classes)[0]


def knn_classify(train_emb: torch.Tensor, train_labels: torch.Tensor, query_emb: torch.Tensor,
                 query_labels: Optional[torch.Tensor] = None, k: int = 3, num_classes: Optional[int] = None,
                 status: Optional[torch.Tensor] = None):
    """knn_predict for up to 1,024 classes and k <= 32, with the correct count reduced on the device: (pred int64 [Q],
    correct int64 [1] or None).  `status`: an int32 device word that a label outside [0, num_classes) sets bit 8 in
    (tsg.nn.check_fused_status raises on it); such a label is read clamped."""
    train_emb = train_emb.contiguous().float(); query_emb = query_emb.contiguous().float()
    train_labels = train_labels.contiguous().to(torch.int64)
    if num_classes is None:
        num_classes = int(train_labels.max().item()) + 1
    pred = torch.empty(query_emb.size(0), dtype=torch.int64, device=query_emb.device)
    correct = None
    if query_labels is not None:
        query_labels = query_labels.contiguous().to(torch.int64)
        correct = torch.empty(1, dtype=torch.int64, device=query_emb.device)
    call("tsg_knn_classify", ptr(train_emb), ptr(train_labels), ptr(query_emb), ptr(query_labels), train_emb.size(0),
         query_emb.size(0), train_emb.size(1), int(k), int(num_classes), ptr(pred), ptr(correct), ptr(status),
         stream_ptr())
    return pred, correct


class Mlp1Classifier:
    """`pred_model` of evaluate_mlp: Linear(in,64) / LeakyReLU / Linear(64,32) / LeakyReLU / Linear(32,classes),
    Adam(lr=1e-3), trained on one embedding per step in the given order (train_triplet.py:148-165).  The
    parameters are initialised by torch's own nn.Linear initialiser (same RNG stream as the reference)."""

    def __init__(self, in_feat: int, device, hidden1: int = 64, hidden2: int = 32, num_classes: int = 2,
                 lr: float = 1e-3, slope: float = 0.01):
        layers = [nn.Linear(in_feat, hidden1), nn.LeakyReLU(slope), nn.Linear(hidden1, hidden2), nn.LeakyReLU(slope),
                  nn.Linear(hidden2, num_classes)]
        self.dims = (in_feat, hidden1, hidden2, num_classes)
        self.lr, self.slope, self.step = lr, slope, 0
        flat = torch.cat([p.detach().reshape(-1) for l in layers if isinstance(l, nn.Linear) for p in (l.weight, l.bias)])
        self.params = flat.to(device).contiguous()
        self.m = torch.zeros_like(self.params); self.v = torch.zeros_like(self.params)

    def views(self):
        D, H1, H2, C = self.dims
        o, out = 0, []
        for r, c in ((H1, D), (H2, H1), (C, H2)):
            out.append(self.params[o:o + r * c].view(r, c)); o += r * c
            out.append(self.params[o:o + r]); o += r
        return out

    def fit(self, emb: torch.Tensor, labels: torch.Tensor, want_losses: bool = False):
        emb = emb.contiguous().float(); labels = labels.contiguous().to(torch.int64)
        D, H1, H2, C = self.dims
        losses = torch.empty(emb.size(0), dtype=torch.float32, device=emb.device) if want_losses else None
        call("tsg_mlp1_train", ptr(emb), ptr(labels), emb.size(0), D, H1, H2, C, ptr(self.params), ptr(self.m), ptr(self.v),
             self.step, self.lr, 0.9, 0.999, 1e-8, self.slope, ptr(losses), stream_ptr())
        self.step += emb.size(0)
        return losses

    def logits(self, emb: torch.Tensor) -> torch.Tensor:
        w1, b1, w2, b2, w3, b3 = self.views()
        h = torch.nn.functional.leaky_relu(emb @ w1.t() + b1, self.slope)
        h = torch.nn.functional.leaky_relu(h @ w2.t() + b2, self.slope)
        return h @ w3.t() + b3

    def predict(self, emb: torch.Tensor) -> torch.Tensor:
        return self.logits(emb).argmax(dim=1)

    def score(self, emb: torch.Tensor, labels: torch.Tensor, status: Optional[torch.Tensor] = None) -> torch.Tensor:
        """#(argmax of the logits == labels) over the rows of `emb` through tsg_mlp1_predict: int64 [1] on the device.
        The logits are the trainer's own forward arithmetic (bitwise); `status` as in knn_classify."""
        return mlp1_predict(self, emb, labels, status=status)[2]


def mlp1_predict(clf: Mlp1Classifier, emb: torch.Tensor, labels: Optional[torch.Tensor] = None,
                 want_logits: bool = False, status: Optional[torch.Tensor] = None):
    """The classifier's forward over every row of `emb` (tsg_mlp1_predict): (pred int64 [Q] = first-index argmax,
    logits [Q, classes] or None, correct int64 [1] or None)."""
    emb = emb.contiguous().float()
    D, H1, H2, C = clf.dims
    Q, dev = emb.size(0), emb.device
    pred = torch.empty(Q, dtype=torch.int64, device=dev)
    logits = torch.empty(Q, C, dtype=torch.float32, device=dev) if want_logits else None
    correct = None
    if labels is not None:
        labels = labels.contiguous().to(torch.int64)
        correct = torch.empty(1, dtype=torch.int64, device=dev)
    call("tsg_mlp1_predict", ptr(emb), ptr(labels), Q, D, H1, H2, C, ptr(clf.params), clf.slope, ptr(pred), ptr(logits),
         ptr(correct), ptr(status), stream_ptr())
    return pred, logits, correct
