"""Trainer / evaluator shell shared by the four graph-CF recommenders.

Reference: recommender/LightGCN.py:17-161 -- ``save / predict / evaluate / test`` are
byte-identical across the reference's recommenders (SURVEY.md 2), so they live here
once.  Public surface kept: ``X(args, data)`` (re-callable on a live instance),
``train(requires_adjgrad, requires_embgrad, gradIterationNum, Epoch, optimizer,
evalNum)``, ``model``, ``user_emb / item_emb / best_user_emb / best_item_emb``,
``predict(user) -> np.ndarray``, ``test() -> (rec_list, [str])``, ``evaluate(epoch)``,
``save()``, ``data / args / topN / max_N / bestPerformance / recOutput``.
"""
from __future__ import annotations

import os
import sys

import torch

from .. import ops
from ..evaluator import FullRankEvaluator


class GraphRecommender(object):
    model_name = "GraphRecommender"

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
        decay / maximize), ONE param group whose tensors ARE the model's two embedding parameters -- the fused engine
        can stand in for ``optimizer.step()``: it starts from the optimizer's state and writes it back.  Anything
        else (another optimizer class, stale parameters built before a re-``__init__`` -- a reference quirk callers
        rely on, SURVEY.md 8b) returns None and takes the reference-shaped loop."""
        if len(list(model.parameters())) != 2:
            return None
        return GraphRecommender._plain_adam(optimizer, [model.embedding_dict['user_emb'], model.embedding_dict['item_emb']])

    @staticmethod
    def _fusable_adam_all(optimizer, model):
        """``_fusable_adam`` for a model with parameters besides the two tables (NGCF's 2L weight matrices): the one
        param group must hold exactly the set ``model.parameters()``, every one of which the fused engine steps."""
        return GraphRecommender._plain_adam(optimizer, list(model.parameters()))

    @staticmethod
    def _plain_adam(optimizer, want):
        """{lr, betas, eps} of a plain torch.optim.Adam with one param group over exactly the tensors ``want`` whose state
        is either empty or initialised for all of them at one step count; None for anything else."""
        if type(optimizer) is not torch.optim.Adam or len(optimizer.param_groups) != 1:
            return None
        g = optimizer.param_groups[0]
        params = list(g['params'])
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
        """The batches of one epoch for the reference-shaped training loops (caller's optimizer, gradient export,
        NGCF / SimGCL / XSimGCL): ``(user_idx, pos_idx, neg_idx)`` as device LongTensors drawn by the on-device
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
    def _train_fused_contrastive(self, model, maxEpoch, evalNum, kind, layer_cl=1, optimizer=None, adam=None):
        """SimGCL / XSimGCL training when the recommender owns the optimizer and no gradient is exported: the fused
        engine (arlib_b200.engine.ContrastiveEngine) -- device sampling (or the host sampler for seed parity), one
        CUDA-graph replay per epoch, Adam state owned by the engine.  Same mathematics as the reference loop
        (recommender/SimGCL.py:36-85, XSimGCL.py:46-95); the perturbation noise comes from Philox in the SpMM
        epilogue instead of torch.rand_like."""
        from ..engine import ContrastiveEngine
        from ..util.sampler import next_batch_pairwise
        table = model.parameter_table()
        dev = table.device
        seed = int(getattr(self.args, 'seed', 0) or 0)
        tau = self.temp if kind == "xsimgcl" else 0.2
        adam = adam or {"lr": self.args.lRate, "betas": (0.9, 0.999), "eps": 1e-8}
        eng = ContrastiveEngine(model._graph, table, self.data.user_num, kind, self.n_layers, self.eps, self.cl_rate, tau,
                                adam["lr"], self.args.reg, self.args.batch_size, len(self.data.training_data),
                                layer_cl=layer_cl, noise_seed=self._next_noise_seed(seed),
                                betas=adam["betas"], adam_eps=adam["eps"])
        if optimizer is not None:
            self._adam_state_to_engine(optimizer, model, eng, self.data.user_num)
        mode = self._sampler_mode()
        ts = self._device_train_set(dev) if mode == 'device' else None
        for epoch in range(maxEpoch):
            if mode == 'device':
                eng.sample_epoch(ts, seed, self._next_sample_epoch())
            else:
                us, is_, js = [], [], []
                for u, i, j in next_batch_pairwise(self.data, self.args.batch_size):
                    us += u; is_ += i; js += j
                eng.set_triples(us, is_, js)
            eng.run_steps(0, use_graph=self._graph_pays_off(maxEpoch))
            rec, cl = eng.losses()
            rec, cl = rec[::100].cpu().tolist(), cl[::100].cpu().tolist()
            for k, (r, c) in enumerate(zip(rec, cl)):
                print('training:', epoch + 1, 'batch', k * 100, 'rec_loss:', r, 'cl_loss', c)
            model.eval()
            with torch.no_grad():
                f = eng.forward_table(out=torch.empty_like(table))
                self.user_emb, self.item_emb = f[:self.data.user_num], f[self.data.user_num:]
            if epoch % evalNum == 0:
                self.evaluate(epoch)
        self.last_train_losses = torch.stack(eng.losses(), 1).clone()
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
