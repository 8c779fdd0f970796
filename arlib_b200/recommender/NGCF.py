"""NGCF -- drop-in for the reference's recommender/NGCF.py (train loop :31-79, encoder :163-212).

``train()`` has two paths with the same mathematics:
  * fused (the recommender's own optimizer, or the caller's plain torch.optim.Adam over exactly ``model.parameters()``;
    no gradient export; d in FUSED_WIDTHS): arlib_b200.engine.NGCFEngine -- one propagation per layer
    (A (E W1) = (A E) W1) + the fused dense layer kernels of csrc/ngcf.cu, forward and backward, Adam on the table fused
    into the last SpMM, replayed from a CUDA graph; a caller's optimizer hands its state to the engine and gets it back;
  * general (any other optimizer, requires_adjgrad / requires_embgrad, the other widths): the reference loop on torch
    autograd with the propagations on the agcf SpMM and the loss on the fused BPR kernels."""
import torch

from ..encoder import NGCF_Encoder, TorchGraphInterface  # noqa: F401
from ..util.loss import bpr_l2_fused, bpr_loss, l2_reg_loss  # noqa: F401
from ._base import GraphRecommender

# widths the fused engine trains at: those where it measured faster than the reference-shaped loop (DESIGN.md 4.7)
FUSED_WIDTHS = (8, 16, 32, 64, 128, 256)


class NGCF(GraphRecommender):
    model_name = "NGCF"

    def _build_model(self):
        return NGCF_Encoder(self.data, self.args.emb_size, self.args.n_layers)

    def train(self, requires_adjgrad=False, requires_embgrad=False, gradIterationNum=10, Epoch=0, optimizer=None,
              evalNum=5):
        self.bestPerformance = []
        model = self.model.cuda()
        exports = requires_adjgrad or requires_embgrad
        adam = self._fusable_adam_all(optimizer, model) if optimizer is not None and not exports else None
        if (optimizer is None or adam is not None) and not exports and self._fused_ok() \
                and int(self.args.emb_size) in FUSED_WIDTHS and model.layers >= 1:
            self._train_fused_ngcf(model, Epoch if Epoch else self.args.maxEpoch, evalNum, optimizer, adam)
            self.user_emb, self.item_emb = self.best_user_emb, self.best_item_emb
            return None
        if optimizer is None:
            optimizer = torch.optim.Adam(model.parameters(), lr=self.args.lRate)
        self._grad_buffers(requires_adjgrad, requires_embgrad, model)
        maxEpoch = Epoch if Epoch else self.args.maxEpoch
        dev = model.embedding_dict['user_emb'].device
        for epoch in range(maxEpoch):
            for n, batch in enumerate(self._epoch_batches(dev)):
                user_idx, pos_idx, neg_idx = batch
                model.train()
                rec_user_emb, rec_item_emb = model()
                # the three gathers + bpr_loss + l2_reg_loss(reg, user_emb, pos_item_emb) of the reference, one fused op
                batch_loss = bpr_l2_fused(rec_user_emb, rec_item_emb, user_idx, pos_idx, neg_idx, self.args.reg)
                optimizer.zero_grad()
                batch_loss.backward()
                self._accumulate_grads(requires_adjgrad, requires_embgrad, maxEpoch, epoch, gradIterationNum)
                optimizer.step()
                if n % 100 == 0:
                    print('training:', epoch + 1, 'batch', n, 'batch_loss:', batch_loss.item())
            model.eval()
            with torch.no_grad():
                self.user_emb, self.item_emb = self.model()
            if epoch % evalNum == 0:
                self.evaluate(epoch)
        self.user_emb, self.item_emb = self.best_user_emb, self.best_item_emb
        return self._train_returns(requires_adjgrad, requires_embgrad)

    def _adam_slots(self, model, eng, n_users):
        """the tables', then w1_k / w2_k -> row blocks [0, d) / [d, 2d) of layer k in the engine's packed moments"""
        d = model.latent_size
        slots = super()._adam_slots(model, eng, n_users)
        for k in range(model.layers):
            slots.append((model.W['w1_%d' % k], eng.Wm[k, :d], eng.Wv[k, :d]))
            slots.append((model.W['w2_%d' % k], eng.Wm[k, d:], eng.Wv[k, d:]))
        return slots

    def _train_fused_ngcf(self, model, maxEpoch, evalNum, optimizer=None, adam=None):
        """optimizer / adam: the caller's plain torch.optim.Adam over all of model.parameters() (_fusable_adam_all); the
        engine starts from its state and hands it back, so the caller can keep stepping it."""
        from ..engine import NGCFEngine
        from ..util.sampler import next_batch_pairwise
        table, W = model.parameter_table(), model.weight_table()
        dev = table.device
        adam = adam or {"lr": self.args.lRate, "betas": (0.9, 0.999), "eps": 1e-8}
        eng = NGCFEngine(model._graph, table, W, self.data.user_num, adam["lr"], self.args.reg, self.args.batch_size,
                         len(self.data.training_data), betas=adam["betas"], adam_eps=adam["eps"])
        if optimizer is not None:
            self._adam_state_to_engine(optimizer, model, eng, self.data.user_num)
        mode = self._sampler_mode()
        ts = self._device_train_set(dev) if mode == 'device' else None
        seed = int(getattr(self.args, 'seed', 0) or 0)
        for epoch in range(maxEpoch):
            if mode == 'device':
                eng.sample_epoch(ts, seed, self._next_sample_epoch())
            else:                                   # host sampler: the reference's RNG consumption
                us, is_, js = [], [], []
                for u, i, j in next_batch_pairwise(self.data, self.args.batch_size):
                    us += u; is_ += i; js += j
                eng.set_triples(us, is_, js)
            losses = eng.run_steps(0, use_graph=self._graph_pays_off(maxEpoch))
            for k, v in enumerate(losses[::100, 0].cpu().tolist()):
                print('training:', epoch + 1, 'batch', k * 100, 'batch_loss:', v)
            model.eval()
            with torch.no_grad():
                f = eng.forward_table(out=torch.empty_like(table))
                self.user_emb, self.item_emb = f[:self.data.user_num], f[self.data.user_num:]
            if epoch % evalNum == 0:
                self.evaluate(epoch)
        self.last_train_losses = eng.out4[:eng.n_batches].clone()
        if optimizer is not None:
            self._adam_state_from_engine(optimizer, model, eng, self.data.user_num)
