"""SimGCL -- drop-in for the reference's recommender/SimGCL.py (class :18-85, encoder
:169-219).  Hyper-parameters are hard-coded like the reference (:31-33: 2 layers,
cl_rate 0.2, eps 0.1, tau 0.2); ``args.n_layers`` is ignored.  Three propagations per
step (1 clean + 2 noise-perturbed) run on agcf_spmm_csr_f32 with the noise fused
into the epilogue.  The fused path of ``train()`` (GraphRecommender) runs
arlib_b200.engine.ContrastiveEngine, with the perturbation noise drawn by Philox in
the SpMM epilogue instead of torch.rand_like."""
import torch

from ..encoder import SimGCL_Encoder, TorchGraphInterface  # noqa: F401
from ..engine import ContrastiveEngine
from ..util.loss import bpr_l2_fused, bpr_loss, l2_reg_loss  # noqa: F401
from ._base import GraphRecommender


class SimGCL(GraphRecommender):
    model_name = "SimGCL"
    LOSS_LABELS = ('rec_loss:', 'cl_loss')

    def _build_model(self):
        self.n_layers = 2
        self.cl_rate = 0.2
        self.eps = 0.1
        return SimGCL_Encoder(self.data, self.args.emb_size, self.eps, self.n_layers)

    def _batch_loss(self, model, user_idx, pos_idx, neg_idx):
        rec_user_emb, rec_item_emb = model()
        rec_l2, parts = bpr_l2_fused(rec_user_emb, rec_item_emb, user_idx, pos_idx, neg_idx, self.args.reg,
                                     return_parts=True)
        cl_loss = self.cl_rate * model.cal_cl_loss([user_idx, pos_idx])
        return rec_l2 + cl_loss, (parts[1], cl_loss)

    def _fused_engine(self, model, table, adam, seed):
        return ContrastiveEngine(model._graph, table, self.data.user_num, "simgcl", self.n_layers, self.eps, self.cl_rate,
                                 0.2, adam["lr"], self.args.reg, self.args.batch_size, len(self.data.training_data),
                                 noise_seed=self._next_noise_seed(seed), betas=adam["betas"], adam_eps=adam["eps"])

    def _engine_losses(self, eng):
        return torch.stack(eng.losses(), 1)
