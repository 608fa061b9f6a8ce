"""The oracle in multi-label mode, for the multi-label parity tests.

The reference picks its loss by dataset (train.py:317-320): BCEWithLogitsLoss(reduction='sum') for yelp, whose labels
are [N, C] 0/1, CrossEntropyLoss(reduction='sum') otherwise.  The oracle's loop (oracle/train.py) builds
CrossEntropyLoss; `multilabel_loss()` makes the loss it builds follow the rank of the targets instead, which for the
graphs here selects the same loss as the reference's dataset test.
"""
import contextlib

import torch

from oracle.train import OracleArgs

_CE = torch.nn.CrossEntropyLoss


class LossByLabelRank(torch.nn.Module):
    def __init__(self, reduction="mean", **kw):
        super().__init__()
        self.ce = _CE(reduction=reduction, **kw)
        self.bce = torch.nn.BCEWithLogitsLoss(reduction=reduction)

    def forward(self, logits, target):
        return self.bce(logits, target) if target.dim() == 2 else self.ce(logits, target)


@contextlib.contextmanager
def multilabel_loss():
    torch.nn.CrossEntropyLoss = LossByLabelRank
    try:
        yield
    finally:
        torch.nn.CrossEntropyLoss = _CE


def fixture_oracle_args(fx, g) -> OracleArgs:
    c = fx["config"]
    return OracleArgs(n_layers=c["n_layers"], n_hidden=c["n_hidden"], n_linear=c.get("n_linear", 0), n_feat=g.n_feat,
                      n_class=c["n_class"], n_train=int(g.train_mask.sum()), dropout=0.0, lr=c["lr"],
                      n_epochs=c["n_epochs"], seed=c["seed"], enable_pipeline=c.get("enable_pipeline", False),
                      use_pp=c.get("use_pp", False))
