"""NGCF -- drop-in for the reference's recommender/NGCF.py (train loop :31-79, encoder :163-212).

``train()`` (GraphRecommender) runs arlib_b200.engine.NGCFEngine on its fused path -- one propagation per layer
(A (E W1) = (A E) W1) + the fused dense layer kernels of csrc/ngcf.cu, forward and backward, Adam on the table fused into
the last SpMM, replayed from a CUDA graph; a caller's Adam over all 2 + 2L parameters hands its state to the engine and
gets it back.  Otherwise, and for a model without layers, the reference loop on torch autograd with the propagations on
the agcf SpMM and the loss on the fused BPR kernels."""
import torch  # noqa: F401

from ..encoder import NGCF_Encoder, TorchGraphInterface  # noqa: F401
from ..engine import NGCFEngine
from ..util.loss import bpr_l2_fused, bpr_loss, l2_reg_loss  # noqa: F401
from ._base import GraphRecommender


class NGCF(GraphRecommender):
    model_name = "NGCF"

    def _build_model(self):
        return NGCF_Encoder(self.data, self.args.emb_size, self.args.n_layers)

    def _adam_slots(self, model, eng, n_users):
        """the tables', then w1_k / w2_k -> row blocks [0, d) / [d, 2d) of layer k in the engine's packed moments"""
        d = model.latent_size
        slots = super()._adam_slots(model, eng, n_users)
        for k in range(model.layers):
            slots.append((model.W['w1_%d' % k], eng.Wm[k, :d], eng.Wv[k, :d]))
            slots.append((model.W['w2_%d' % k], eng.Wm[k, d:], eng.Wv[k, d:]))
        return slots

    def _engine_accepts(self, model):
        return model.layers >= 1

    def _fused_engine(self, model, table, adam, seed):
        return NGCFEngine(model._graph, table, model.weight_table(), self.data.user_num, adam["lr"], self.args.reg,
                          self.args.batch_size, len(self.data.training_data), betas=adam["betas"], adam_eps=adam["eps"])
