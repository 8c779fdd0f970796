"""LightGCN -- drop-in for the reference's recommender/LightGCN.py.

``train()`` (GraphRecommender) runs arlib_b200.engine.LightGCNEngine on its fused path -- 2L+5 kernels per batch
replayed from a CUDA graph -- and otherwise the reference loop on torch autograd, with the encoder forward/backward on
the agcf SpMM kernels and ``.grad`` populated on the real nn.Parameters.
"""
import torch  # noqa: F401

from ..encoder import LGCN_Encoder, TorchGraphInterface  # noqa: F401  (re-exported like the reference module)
from ..engine import LightGCNEngine
from ..util.loss import bpr_l2_fused, bpr_loss, l2_reg_loss  # noqa: F401
from ..util.sampler import next_batch_pairwise  # noqa: F401
from ._base import GraphRecommender


class LightGCN(GraphRecommender):
    model_name = "LightGCN"
    PRINT_EVERY = 1000
    KEEPS_OPTIMIZER = True

    def _build_model(self):
        return LGCN_Encoder(self.data, self.args.emb_size, self.args.n_layers)

    def _fused_engine(self, model, table, adam, seed):
        return LightGCNEngine(model._graph, table, self.data.user_num, model.layers, adam["lr"], self.args.reg,
                              self.args.batch_size, len(self.data.training_data), betas=adam["betas"],
                              adam_eps=adam["eps"])
