"""Trainer / evaluator shell shared by the four graph-CF recommenders.

Reference: recommender/LightGCN.py:17-161 -- ``save / predict / evaluate / test`` are
byte-identical across the reference's recommenders (SURVEY.md 2), so they live here
once.  Public surface kept: ``X(args, data)`` (re-callable on a live instance),
``train(requires_adjgrad, requires_embgrad, gradIterationNum, Epoch, optimizer,
evalNum)``, ``model``, ``user_emb / item_emb / best_user_emb / best_item_emb``,
``predict(user) -> np.ndarray``, ``test() -> (rec_list, [str])``, ``evaluate(epoch)``,
``save()``, ``data / args / topN / max_N / bestPerformance / recOutput``.

``train()`` is written once here and has two paths with the same mathematics:
  * fused (no gradient export; the recommender's own optimizer, or the caller's plain torch.optim.Adam over exactly
    ``model.parameters()``): ``_train_fused`` runs the model's engine from arlib_b200.engine -- on-device Philox
    sampling (or the host sampler for seed parity), one CUDA-graph replay per epoch, Adam state owned by the engine
    and handed back to a caller's optimizer;
  * general (any other optimizer, requires_adjgrad / requires_embgrad): the reference loop on torch autograd, with the
    propagations on the agcf SpMM kernels and ``.grad`` populated on the real nn.Parameters.
A model class supplies ``_build_model`` and what differs between the models: the batch loss of the general path
(``_batch_loss``), its engine (``_fused_engine``, ``_engine_accepts``, ``_engine_losses``) and its print line
(``LOSS_LABELS``, ``PRINT_EVERY``).
"""
from __future__ import annotations

import os
import sys

import torch

from .. import ops
from ..evaluator import FullRankEvaluator
from ..util.loss import bpr_l2_fused


class GraphRecommender(object):
    model_name = "GraphRecommender"
    # the reference's print line of a training batch: the labels of the printed losses, every PRINT_EVERY batches
    LOSS_LABELS = ('batch_loss:',)
    PRINT_EVERY = 100
    # the reference's LightGCN keeps its optimizer as self.optimizer and the others do not; the drop-ins mirror the
    # reference's attribute set because callers pickle the whole object (ARLib.py:127-131)
    KEEPS_OPTIMIZER = False

    def __init__(self, args, data):
        print("Recommender: " + self.model_name)
        self.data = data
        self.args = args
        self.bestPerformance = []
        self.recOutput = []
        self.topN = [int(num) for num in self.args.topK.split(',')]
        self.max_N = max(self.topN)
        # the row kernels hold a row as d/4 float4 lanes and are compiled for these widths only (csrc/common.cuh);
        # there is no fallback path by design, so say so here instead of failing inside the first propagation
        if int(self.args.emb_size) not in (8, 16, 32, 64, 128, 256):
            raise ValueError("arlib_b200: emb_size must be one of 8, 16, 32, 64, 128, 256 (got %r); the sm_100a kernels "
                             "are compiled for these widths and there is no CPU / generic fallback" % (self.args.emb_size,))
        self._evaluator = None
        self._train_set = None                # device mirrors are derived from ``data``: a re-__init__ drops both
        self.model = self._build_model()

    def _build_model(self):
        raise NotImplementedError

    # the evaluator holds device mirrors of data.test_set / training_set_u; it is
    # rebuilt whenever the data object changed shape (attacks mutate it in place)
    def _get_evaluator(self):
        key = (id(self.data), len(self.data.test_set), len(self.data.training_data), self.data.user_num,
               self.data.item_num)
        ev = self._evaluator
        if ev is None or ev[0] != key:
            dev = self.model.embedding_dict['user_emb'].device
            ev = (key, FullRankEvaluator(self.data, dev))
            self._evaluator = ev
        return ev[1]

    def __getstate__(self):           # device mirrors are derived data: keep pickles / deepcopies lean
        st = dict(self.__dict__)
        st['_evaluator'] = None
        st['_train_set'] = None
        return st

    def _sampler_mode(self):
        return str(getattr(self.args, 'sampler', os.environ.get('ARLIB_B200_SAMPLER', 'device'))).lower()

    def _fused_ok(self):
        """the fused engines take the batch sizes the single-CTA grouping sorts (3 B <= 16384) and are switched off
        by args.fused = False / ARLIB_B200_FUSED=0 (then the reference-shaped loop runs on the same kernels)"""
        on = getattr(self.args, 'fused', os.environ.get('ARLIB_B200_FUSED', '1'))
        return str(on).lower() not in ('0', 'false') and 3 * self.args.batch_size <= 16384

    # --------------------------------------------------- caller's torch.optim.Adam on the fused engines
    @staticmethod
    def _fusable_adam(optimizer, model):
        """The attacks hand ``train()`` their own optimizer (18 call sites, e.g. attack/White/CLeaR.py:145-146), nearly
        always ``torch.optim.Adam(model.parameters(), lr)``.  If it is exactly that -- plain Adam (no amsgrad / weight
        decay / maximize), ONE param group whose tensors ARE the set ``model.parameters()`` (the two embedding tables,
        and NGCF's 2L weight matrices), state either empty or initialised for all of them at one step count -- the fused
        engine can stand in for ``optimizer.step()``: it starts from the optimizer's state and writes it back; the
        result is its {lr, betas, eps}.  Anything else (another optimizer class, a subset of the parameters, stale
        parameters built before a re-``__init__`` -- a reference quirk callers rely on, SURVEY.md 8b) returns None and
        takes the reference-shaped loop."""
        if type(optimizer) is not torch.optim.Adam or len(optimizer.param_groups) != 1:
            return None
        g = optimizer.param_groups[0]
        params, want = list(g['params']), list(model.parameters())
        if len(params) != len(want) or {id(a) for a in params} != {id(b) for b in want}:
            return None
        if g.get('amsgrad') or g.get('weight_decay', 0) != 0 or g.get('maximize') or g.get('differentiable'):
            return None
        if torch.is_tensor(g['lr']) or g.get('decoupled_weight_decay'):
            return None
        steps = [float(optimizer.state[p]['step']) for p in params if len(optimizer.state.get(p, {}))]
        if 0 < len(steps) < len(params) or len(set(steps)) > 1:
            return None
        return {"lr": float(g['lr']), "betas": (float(g['betas'][0]), float(g['betas'][1])), "eps": float(g['eps'])}

    def _adam_slots(self, model, eng, n_users):
        """(parameter, the engine's exp_avg of it, the engine's exp_avg_sq of it) for every parameter the engine steps"""
        return [(model.embedding_dict['user_emb'], eng.m[:n_users], eng.v[:n_users]),
                (model.embedding_dict['item_emb'], eng.m[n_users:], eng.v[n_users:])]

    def _adam_state_to_engine(self, optimizer, model, eng, n_users):
        slots = self._adam_slots(model, eng, n_users)
        states = [optimizer.state.get(p, {}) for p, _, _ in slots]
        if all(len(st) for st in states):
            for (_, m, v), st in zip(slots, states):
                m.copy_(st['exp_avg']); v.copy_(st['exp_avg_sq'])
            eng.step_dev.fill_(int(float(states[0]['step'])))
            eng._refresh_adam_coefs()

    def _adam_state_from_engine(self, optimizer, model, eng, n_users):
        g = optimizer.param_groups[0]
        steps = int(eng.step_dev.item())
        for p, m, v in self._adam_slots(model, eng, n_users):
            st = optimizer.state[p]
            if len(st) == 0:                                  # what torch.optim.Adam._init_group creates lazily
                on_dev = bool(g.get('capturable') or g.get('fused'))
                st['step'] = torch.zeros((), dtype=torch.float32, device=p.device) if on_dev else torch.tensor(0.0)
                st['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            st['exp_avg'].copy_(m); st['exp_avg_sq'].copy_(v)
            st['step'].fill_(float(steps))

    @staticmethod
    def _graph_pays_off(max_epoch):
        """Capturing + instantiating the CUDA graph of an epoch costs ~0.3 s (torch empties its cache, thousands of
        kernel nodes); the eager launch sequence is GPU-bound at the named shapes (7 launches, ~60 us of CPU, per
        >= 150 us step).  The graph is worth it when it is replayed for several epochs -- not for the 1-2 epoch
        re-entries of the attack loops (measured at ml-1M shape, 490 batches: 0.133 s with a captured graph, 0.086 s eager
        per train(Epoch=1) call)."""
        return max_epoch >= 5

    def _next_sample_epoch(self):
        """Philox stream id of the next sampled epoch: keeps counting across train() calls on one instance (an
        attack that retrains the same recommender must not see the same triples again, like the reference's
        global Python RNG that simply keeps advancing)."""
        k = getattr(self, '_epochs_sampled', 0)
        self._epochs_sampled = k + 1
        return k

    def _next_noise_seed(self, seed):
        """Philox key of the perturbation noise of ONE train() call.  The engine's counter is (key, step, stream, row)
        and its step restarts at 0 with every engine, so the key mixes in a per-instance call counter: an attack that
        re-enters train(Epoch=1) must not replay the same perturbations per step index (the reference's
        torch.rand_like stream simply keeps advancing, recommender/SimGCL.py:204)."""
        k = getattr(self, '_noise_calls', 0)
        self._noise_calls = k + 1
        return ((seed * 2654435761 + 12345) ^ (k * 0x9E3779B97F4A7C15)) & 0xffffffffffffffff or 1

    def _device_train_set(self, dev):
        """Device mirror of data.training_data / training_set_u for the Philox sampler, rebuilt only when the data
        object changed (attacks append fake users' rows and re-enter train() many times; the O(E) Python pass over
        the rows would otherwise dominate a fused epoch)."""
        from ..engine import DeviceTrainSet
        key = (id(self.data), len(self.data.training_data), self.data.user_num, self.data.item_num, str(dev))
        cached = getattr(self, '_train_set', None)
        if cached is None or cached[0] != key:
            cached = (key, DeviceTrainSet(self.data, dev))
            self._train_set = cached
        return cached[1]

    def _epoch_batches(self, dev):
        """The batches of one epoch for the reference-shaped training loop (caller's optimizer, gradient export):
        ``(user_idx, pos_idx, neg_idx)`` as device LongTensors drawn by the on-device
        Philox sampler (agcf_bpr_sample_epoch, util/sampler.py:4-30), or -- sampler mode 'host' -- the reference's
        Python lists from util.sampler.next_batch_pairwise (same RNG consumption, in-place shuffle)."""
        from ..util.sampler import next_batch_pairwise
        B = self.args.batch_size
        if self._sampler_mode() != 'device':
            yield from next_batch_pairwise(self.data, B)
            return
        ts = self._device_train_set(dev)
        n = ts.n_edges
        u, i, j = (torch.empty(max(n, 1), dtype=torch.int32, device=dev) for _ in range(3))
        seed = int(getattr(self.args, 'seed', 0) or 0)
        ops.bpr_sample_epoch(ts.e_user, ts.e_item, ts.rej_rowptr, ts.rej_items, ts.n_items, seed,
                             self._next_sample_epoch(), u, i, j)
        u, i, j = u.long(), i.long(), j.long()
        for lo in range(0, n, B):
            yield u[lo:lo + B], i[lo:lo + B], j[lo:lo + B]

    # ------------------------------------------------------------------ reference API
    def save(self):
        """recommender/LightGCN.py:82-84"""
        with torch.no_grad():
            self.best_user_emb, self.best_item_emb = self.model.forward()

    def predict(self, u):
        """recommender/LightGCN.py:86-90 -- un-masked fp32 scores of one user, on the host."""
        with torch.no_grad():
            uid = self.data.get_user_id(u)
            rows = torch.tensor([uid], dtype=torch.int32, device=self.item_emb.device)
            score = ops.score_rows(self.user_emb.detach().contiguous(), rows, self.item_emb.detach().contiguous())
            return score[0].cpu().numpy()

    def evaluate(self, epoch):
        """recommender/LightGCN.py:92-135 -- keep-best by majority vote over the 4 metrics."""
        print('Evaluating the model...')
        ev = self._get_evaluator()
        with torch.no_grad():
            _, idx = ev.topk(self.user_emb, self.item_emb, self.max_N)
        measure = ev.measure(idx, [self.max_N])
        performance = {}
        for m in measure[1:]:
            k, v = m.strip().split(':')
            performance[k] = float(v)
        if len(self.bestPerformance) > 0:
            count = 0
            for k in self.bestPerformance[1]:
                if self.bestPerformance[1][k] > performance[k]:
                    count += 1
                else:
                    count -= 1
            if count < 0:
                self.bestPerformance[1] = performance
                self.bestPerformance[0] = epoch + 1
                self.save()
        else:
            self.bestPerformance.append(epoch + 1)
            self.bestPerformance.append(performance)
            self.save()
        print('-' * 120)
        print('Real-Time Ranking Performance ' + ' (Top-' + str(self.max_N) + ' Item Recommendation)')
        measure = [m.strip() for m in measure[1:]]
        print('*Current Performance*')
        print('Epoch:', str(epoch + 1) + ',', '  |  '.join(measure))
        bp = ''
        bp += 'Hit Ratio' + ':' + str(self.bestPerformance[1]['Hit Ratio']) + '  |  '
        bp += 'Precision' + ':' + str(self.bestPerformance[1]['Precision']) + '  |  '
        bp += 'Recall' + ':' + str(self.bestPerformance[1]['Recall']) + '  |  '
        bp += 'NDCG' + ':' + str(self.bestPerformance[1]['NDCG'])
        print('*Best Performance* ')
        print('Epoch:', str(self.bestPerformance[0]) + ',', bp)
        print('-' * 120)
        return measure

    def test(self):
        """recommender/LightGCN.py:137-161 -> (rec_list, metric strings)."""
        ev = self._get_evaluator()
        with torch.no_grad():
            rec_list, measure = ev.test(self.user_emb, self.item_emb, self.topN, self.max_N)
        sys.stdout.write('\rProgress: [{}]100%\n'.format('+' * 50))
        return rec_list, measure

    # ------------------------------------------------------------------ training
    def train(self, requires_adjgrad=False, requires_embgrad=False, gradIterationNum=10, Epoch=0, optimizer=None,
              evalNum=5):
        """The reference's ``train()`` of all four recommenders: the fused engine when nothing is exported and the
        engine can stand in for the optimizer, otherwise the reference-shaped loop."""
        self.bestPerformance = []
        model = self.model.cuda()
        maxEpoch = Epoch if Epoch else self.args.maxEpoch
        exports = requires_adjgrad or requires_embgrad
        adam = self._fusable_adam(optimizer, model) if optimizer is not None and not exports else None
        if (optimizer is None or adam is not None) and not exports and self._fused_ok() and self._engine_accepts(model):
            self._train_fused(model, maxEpoch, evalNum, optimizer, adam)
            self.user_emb, self.item_emb = self.best_user_emb, self.best_item_emb
            return None
        if optimizer is None:
            optimizer = torch.optim.Adam(model.parameters(), lr=self.args.lRate)
        if self.KEEPS_OPTIMIZER:
            self.optimizer = optimizer
        self._grad_buffers(requires_adjgrad, requires_embgrad, model)
        dev = model.embedding_dict['user_emb'].device
        for epoch in range(maxEpoch):
            for n, (user_idx, pos_idx, neg_idx) in enumerate(self._epoch_batches(dev)):
                model.train()
                batch_loss, shown = self._batch_loss(model, user_idx, pos_idx, neg_idx)
                optimizer.zero_grad()
                batch_loss.backward()
                self._accumulate_grads(requires_adjgrad, requires_embgrad, maxEpoch, epoch, gradIterationNum)
                optimizer.step()
                if n % self.PRINT_EVERY == 0:
                    self._print_losses(epoch, n, [t.item() for t in shown])
            model.eval()
            with torch.no_grad():
                self.user_emb, self.item_emb = self.model()
            if epoch % evalNum == 0:
                self.evaluate(epoch)
        self.user_emb, self.item_emb = self.best_user_emb, self.best_item_emb
        return self._train_returns(requires_adjgrad, requires_embgrad)

    def _print_losses(self, epoch, n, values):
        pairs = [x for label, v in zip(self.LOSS_LABELS, values) for x in (label, v)]
        print('training:', epoch + 1, 'batch', n, *pairs)

    def _batch_loss(self, model, user_idx, pos_idx, neg_idx):
        """(loss to backpropagate, the tensors printed under LOSS_LABELS) of one batch of the reference-shaped loop.
        BPR + L2 of LightGCN and NGCF: the three gathers + bpr_loss + l2_reg_loss(reg, user_emb, pos_item_emb) of the
        reference, one fused op."""
        rec_user_emb, rec_item_emb = model()
        batch_loss = bpr_l2_fused(rec_user_emb, rec_item_emb, user_idx, pos_idx, neg_idx, self.args.reg)
        return batch_loss, (batch_loss,)

    def _fused_engine(self, model, table, adam, seed):
        """the model's fused training engine (arlib_b200.engine) over ``table``, with Adam's {lr, betas, eps}"""
        raise NotImplementedError

    def _engine_accepts(self, model):
        """whether ``_fused_engine`` can train this model's configuration"""
        return True

    def _engine_losses(self, eng):
        """the engine's per-batch losses of the last epoch, [n_batches, k]; the first len(LOSS_LABELS) columns are the
        printed ones.  Kept as ``last_train_losses``."""
        return eng.out4[:eng.n_batches]

    def _train_fused(self, model, maxEpoch, evalNum, optimizer=None, adam=None):
        """train() on the model's fused engine.  optimizer / adam: the caller's plain torch.optim.Adam over
        model.parameters() (_fusable_adam); the engine starts from its state and hands it back, so the caller can keep
        stepping it."""
        from ..util.sampler import next_batch_pairwise
        table = model.parameter_table()
        dev = table.device
        seed = int(getattr(self.args, 'seed', 0) or 0)
        adam = adam or {"lr": self.args.lRate, "betas": (0.9, 0.999), "eps": 1e-8}
        eng = self._fused_engine(model, table, adam, seed)
        if optimizer is not None:
            self._adam_state_to_engine(optimizer, model, eng, self.data.user_num)
        mode = self._sampler_mode()
        ts = self._device_train_set(dev) if mode == 'device' else None
        every, shown = self.PRINT_EVERY, len(self.LOSS_LABELS)
        for epoch in range(maxEpoch):
            if mode == 'device':
                eng.sample_epoch(ts, seed, self._next_sample_epoch())
            else:                                   # host sampler: the reference's RNG consumption
                us, is_, js = [], [], []
                for u, i, j in next_batch_pairwise(self.data, self.args.batch_size):
                    us += u; is_ += i; js += j
                eng.set_triples(us, is_, js)
            eng.run_steps(0, use_graph=self._graph_pays_off(maxEpoch))
            for k, values in enumerate(self._engine_losses(eng)[::every, :shown].cpu().tolist()):
                self._print_losses(epoch, k * every, values)
            model.eval()
            with torch.no_grad():
                f = eng.forward_table(out=torch.empty_like(table))
                self.user_emb, self.item_emb = f[:self.data.user_num], f[self.data.user_num:]
            if epoch % evalNum == 0:
                self.evaluate(epoch)
        self.last_train_losses = self._engine_losses(eng).clone()
        if optimizer is not None:
            self._adam_state_from_engine(optimizer, model, eng, self.data.user_num)

    def _grad_buffers(self, requires_adjgrad, requires_embgrad, model):
        """recommender/LightGCN.py:36-43.  The reference allocates a DENSE N x N Matgrad
        (20 GB at Gowalla shape); here the adjacency gradient is accumulated on the stored
        pattern and only densified on return."""
        if requires_embgrad:
            model.requires_grad = True
            dev = model.embedding_dict['user_emb'].device
            self.usergrad = torch.zeros((self.data.user_num, self.args.emb_size), device=dev)
            self.itemgrad = torch.zeros((self.data.item_num, self.args.emb_size), device=dev)
        elif requires_adjgrad:
            self.model.sparse_norm_adj.requires_grad = True
            self.Matgrad = None

    def _accumulate_grads(self, requires_adjgrad, requires_embgrad, maxEpoch, epoch, gradIterationNum):
        """recommender/LightGCN.py:58-62"""
        if requires_adjgrad and maxEpoch - epoch < gradIterationNum:
            g = self.model.sparse_norm_adj.grad
            self.Matgrad = g.clone() if self.Matgrad is None else self.Matgrad + g
        elif requires_embgrad and maxEpoch - epoch < gradIterationNum:
            self.usergrad += self.model.embedding_dict["user_emb"].grad
            self.itemgrad += self.model.embedding_dict["item_emb"].grad

    def _train_returns(self, requires_adjgrad, requires_embgrad):
        """recommender/LightGCN.py:74-80"""
        if requires_adjgrad:
            n = self.data.user_num + self.data.item_num
            dense = self.Matgrad.to_dense() if self.Matgrad is not None else \
                torch.zeros((n, n), device=self.user_emb.device)
            mat = (dense + dense.T)[:self.data.user_num, self.data.user_num:]
        if requires_adjgrad and requires_embgrad:
            return mat, self.user_emb, self.item_emb, self.usergrad, self.itemgrad
        elif requires_adjgrad:
            return mat
        elif requires_embgrad:
            return self.user_emb, self.item_emb, self.usergrad, self.itemgrad
