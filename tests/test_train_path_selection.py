"""train() of the four recommenders chooses between the fused engine and the reference-shaped loop from host-side facts
alone: the optimizer handed in, gradient export, args.fused / ARLIB_B200_FUSED, the batch size and what the model's
engine accepts.  Driven on CPU stand-ins: the model is a small module with the parameters of each encoder, the fused
path is recorded by patching ``_train_fused``, and the loop runs zero batches (``_epoch_batches`` yields none)."""
import importlib
import types

import pytest
import torch

CLASSES = ["LightGCN", "NGCF", "SimGCL", "XSimGCL"]
U, I, D = 3, 5, 8


class _Model(torch.nn.Module):
    """the two embedding tables, plus NGCF's w1_k / w2_k when ``ngcf_layers`` is given; calling it returns the tables"""

    def __init__(self, ngcf_layers=None):
        super().__init__()
        self.embedding_dict = torch.nn.ParameterDict({'user_emb': torch.nn.Parameter(torch.zeros(U, D)),
                                                      'item_emb': torch.nn.Parameter(torch.zeros(I, D))})
        self.sparse_norm_adj = torch.zeros(U + I, U + I)
        if ngcf_layers is not None:
            self.layers = ngcf_layers
            self.W = torch.nn.ParameterDict({'w%d_%d' % (a, k): torch.nn.Parameter(torch.zeros(D, D))
                                             for k in range(ngcf_layers) for a in (1, 2)})

    def cuda(self):
        return self

    def forward(self):
        return self.embedding_dict['user_emb'], self.embedding_dict['item_emb']


def _rec(name, monkeypatch, ngcf_layers=2, layer_cl=1, **args):
    """(recommender built without __init__, the list of paths its train() calls take)"""
    cls = getattr(importlib.import_module("arlib_b200.recommender." + name), name)
    rec = cls.__new__(cls)
    rec.args = types.SimpleNamespace(**{"batch_size": 2048, "lRate": 0.01, "emb_size": D, "maxEpoch": 1, "reg": 1e-4,
                                        "seed": 0, **args})
    rec.data = types.SimpleNamespace(user_num=U, item_num=I)
    rec.model = _Model(ngcf_layers if name == "NGCF" else None)
    if name in ("SimGCL", "XSimGCL"):
        rec.n_layers, rec.cl_rate, rec.eps = 2, 0.2, 0.1
    if name == "XSimGCL":
        rec.layer_cl, rec.temp = layer_cl, 0.1
    rec.best_user_emb, rec.best_item_emb = rec.model()          # what evaluate() saves
    paths = []

    def no_batches(self, dev):
        paths.append("loop")
        yield from ()
    monkeypatch.delenv("ARLIB_B200_FUSED", raising=False)
    monkeypatch.setattr(cls, "_train_fused", lambda self, *a, **k: paths.append("fused"))
    monkeypatch.setattr(cls, "_epoch_batches", no_batches)
    monkeypatch.setattr(cls, "evaluate", lambda self, epoch: None)
    return rec, paths


def _train(rec, optimizer, export):
    return rec.train(Epoch=1, optimizer=optimizer, **({export: True} if export else {}))


def _check_optimizer_attribute(rec, name, path, optimizer):
    """only LightGCN's reference-shaped loop keeps its optimizer as ``self.optimizer``, like the reference"""
    if name == "LightGCN" and path == "loop" and optimizer is None:
        assert type(rec.optimizer) is torch.optim.Adam
    elif name == "LightGCN" and path == "loop":
        assert rec.optimizer is optimizer
    else:
        assert "optimizer" not in vars(rec)


OPTIMIZERS = {
    "none": lambda m: None,
    "adam": lambda m: torch.optim.Adam(m.parameters(), lr=0.003, betas=(0.8, 0.99), eps=1e-7),
    "adam-over-the-tables": lambda m: torch.optim.Adam([m.embedding_dict['user_emb'], m.embedding_dict['item_emb']]),
    "sgd": lambda m: torch.optim.SGD(m.parameters(), lr=0.1),
    "adamw": lambda m: torch.optim.AdamW(m.parameters(), lr=0.1),
    "amsgrad": lambda m: torch.optim.Adam(m.parameters(), lr=0.1, amsgrad=True),
    "weight-decay": lambda m: torch.optim.Adam(m.parameters(), lr=0.1, weight_decay=1e-4),
    "stale": lambda m: torch.optim.Adam([torch.nn.Parameter(torch.zeros(U, D)), torch.nn.Parameter(torch.zeros(I, D))]),
}


@pytest.mark.parametrize("export", [None, "requires_adjgrad", "requires_embgrad"])
@pytest.mark.parametrize("opt", list(OPTIMIZERS))
@pytest.mark.parametrize("name", CLASSES)
def test_the_optimizer_selects_the_path(name, opt, export, monkeypatch):
    """the engine stands in for no optimizer or a plain Adam over exactly model.parameters() (for NGCF that includes the
    weight matrices, so an Adam over the two tables keeps the loop), and only when no gradient is exported"""
    rec, paths = _rec(name, monkeypatch)
    optimizer = OPTIMIZERS[opt](rec.model)
    out = _train(rec, optimizer, export)
    fusable = opt in ("none", "adam") or (opt == "adam-over-the-tables" and name != "NGCF")
    path = "fused" if fusable and export is None else "loop"
    assert paths == [path]
    assert (out is None) == (export is None)
    _check_optimizer_attribute(rec, name, path, optimizer)


CONFIGS = {
    "args.fused=False": dict(fused=False),
    "ARLIB_B200_FUSED=0": dict(),
    "3B>16384": dict(batch_size=6000),
    "layer_cl=0": dict(layer_cl=0),
    "layer_cl=n_layers": dict(layer_cl=2),
    "ngcf-without-layers": dict(ngcf_layers=0),
}


@pytest.mark.parametrize("export", [None, "requires_adjgrad", "requires_embgrad"])
@pytest.mark.parametrize("opt", ["none", "adam"])
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("name", CLASSES)
def test_the_configuration_selects_the_path(name, config, opt, export, monkeypatch):
    """args.fused / ARLIB_B200_FUSED off and batches the fused grouping cannot sort keep the loop for every model;
    XSimGCL's engine needs 1 <= layer_cl < n_layers and NGCF's at least one layer (other models ignore those)"""
    rec, paths = _rec(name, monkeypatch, **CONFIGS[config])
    if config == "ARLIB_B200_FUSED=0":
        monkeypatch.setenv("ARLIB_B200_FUSED", "0")
    optimizer = OPTIMIZERS[opt](rec.model)
    _train(rec, optimizer, export)
    rejected = config in ("args.fused=False", "ARLIB_B200_FUSED=0", "3B>16384") or \
        (name == "XSimGCL" and config.startswith("layer_cl")) or (name == "NGCF" and config == "ngcf-without-layers")
    path = "loop" if rejected or export else "fused"
    assert paths == [path]
    _check_optimizer_attribute(rec, name, path, optimizer)
