"""XSimGCL -- drop-in for the reference's recommender/XSimGCL.py (class :18-95, encoder
:179-223).  Hard-coded hyper-parameters like the reference (:32-36: 2 layers, cl_rate
0.2, eps 0.1, layer_cl 1, tau 0.1).  One noise-perturbed propagation per step on
agcf_spmm_csr_f32 (noise fused into the epilogue, the layer_cl view kept).  The fused
path of ``train()`` (GraphRecommender) runs arlib_b200.engine.ContrastiveEngine when
1 <= layer_cl < n_layers, with the perturbation noise drawn by Philox in the SpMM
epilogue instead of torch.rand_like."""
import torch

from ..encoder import TorchGraphInterface, XSimGCL_Encoder, unique_ids_like_reference  # noqa: F401
from ..engine import ContrastiveEngine
from ..util.loss import InfoNCE, bpr_l2_fused, bpr_loss, l2_reg_loss  # noqa: F401
from ._base import GraphRecommender


class XSimGCL(GraphRecommender):
    model_name = "XSimGCL"
    LOSS_LABELS = ('rec_loss:', 'cl_loss')

    def _build_model(self):
        self.n_layers = 2
        self.cl_rate = 0.2
        self.eps = 0.1
        self.layer_cl = 1
        self.temp = 0.1
        return XSimGCL_Encoder(self.data, self.args.emb_size, self.eps, self.n_layers, self.layer_cl)

    def cal_cl_loss(self, idx, user_view1, user_view2, item_view1, item_view2):
        """recommender/XSimGCL.py:39-44 (ids pass through float32 like torch.Tensor(list))"""
        dev = user_view1.device
        u_idx, i_idx = unique_ids_like_reference(idx[0], dev), unique_ids_like_reference(idx[1], dev)
        return InfoNCE(user_view1[u_idx], user_view2[u_idx], self.temp) + \
            InfoNCE(item_view1[i_idx], item_view2[i_idx], self.temp)

    def _batch_loss(self, model, user_idx, pos_idx, neg_idx):
        rec_user_emb, rec_item_emb, cl_user_emb, cl_item_emb = model(True)
        rec_l2, parts = bpr_l2_fused(rec_user_emb, rec_item_emb, user_idx, pos_idx, neg_idx, self.args.reg,
                                     return_parts=True)
        cl_loss = self.cl_rate * self.cal_cl_loss([user_idx, pos_idx], rec_user_emb, cl_user_emb, rec_item_emb,
                                                  cl_item_emb)
        return rec_l2 + cl_loss, (parts[1], cl_loss)

    def _engine_accepts(self, model):
        return 1 <= self.layer_cl < self.n_layers

    def _fused_engine(self, model, table, adam, seed):
        return ContrastiveEngine(model._graph, table, self.data.user_num, "xsimgcl", self.n_layers, self.eps,
                                 self.cl_rate, self.temp, adam["lr"], self.args.reg, self.args.batch_size,
                                 len(self.data.training_data), layer_cl=self.layer_cl,
                                 noise_seed=self._next_noise_seed(seed), betas=adam["betas"], adam_eps=adam["eps"])

    def _engine_losses(self, eng):
        return torch.stack(eng.losses(), 1)
