"""NGCF's caller's-Adam recogniser (GraphRecommender._fusable_adam) and the state handover between a
torch.optim.Adam over all 2 + 2L parameters and the fused engine's packed moments, on CPU tensors."""
import torch


def _ngcf_like(d=4, L=2, n_users=3, n_items=5):
    m = torch.nn.Module()
    m.embedding_dict = torch.nn.ParameterDict({'user_emb': torch.nn.Parameter(torch.zeros(n_users, d)),
                                               'item_emb': torch.nn.Parameter(torch.zeros(n_items, d))})
    packed = torch.zeros(L, 2 * d, d)
    m.W = torch.nn.ParameterDict({})
    for k in range(L):
        m.W['w1_%d' % k] = torch.nn.Parameter(packed[k, :d])
        m.W['w2_%d' % k] = torch.nn.Parameter(packed[k, d:])
    m.latent_size, m.layers = d, L
    return m


def test_single_recogniser_accepts_exactly_plain_adam_over_all_parameters():
    from arlib_b200.recommender._base import GraphRecommender
    f = GraphRecommender._fusable_adam
    m = _ngcf_like()
    got = f(torch.optim.Adam(m.parameters(), lr=0.003, betas=(0.8, 0.99), eps=1e-7), m)
    assert got == {"lr": 0.003, "betas": (0.8, 0.99), "eps": 1e-7}
    assert f(torch.optim.Adam(list(m.parameters())[::-1], lr=0.1), m) is not None          # the set, in any order
    e, W = m.embedding_dict, m.W
    tables = [e['user_emb'], e['item_emb']]
    for bad in (torch.optim.SGD(m.parameters(), lr=0.1),
                torch.optim.AdamW(m.parameters(), lr=0.1),
                torch.optim.Adam(m.parameters(), lr=0.1, amsgrad=True),
                torch.optim.Adam(m.parameters(), lr=0.1, weight_decay=1e-4),
                torch.optim.Adam(m.parameters(), lr=0.1, maximize=True),
                torch.optim.Adam(m.parameters(), lr=torch.tensor(0.1)),
                torch.optim.Adam(tables, lr=0.1),                                             # the two tables only
                torch.optim.Adam(tables + [W['w1_0'], W['w2_0'], W['w1_1']], lr=0.1),         # one weight missing
                torch.optim.Adam([{'params': tables}, {'params': list(W.values())}], lr=0.1),
                torch.optim.Adam([torch.nn.Parameter(p.detach().clone()) for p in m.parameters()], lr=0.1)):  # stale
        assert f(bad, m) is None, bad
    # state: half-initialised, or initialised at unequal steps
    for steps in ([3.0, None, 3.0, 3.0, 3.0, 3.0], [3.0, 3.0, 3.0, 3.0, 3.0, 2.0]):
        opt = torch.optim.Adam(m.parameters(), lr=0.1)
        for p, s in zip(m.parameters(), steps):
            if s is not None:
                opt.state[p] = {'step': torch.tensor(s), 'exp_avg': torch.zeros_like(p), 'exp_avg_sq': torch.zeros_like(p)}
        assert f(opt, m) is None, steps
    opt = torch.optim.Adam(m.parameters(), lr=0.1)
    for p in m.parameters():
        opt.state[p] = {'step': torch.tensor(7.0), 'exp_avg': torch.zeros_like(p), 'exp_avg_sq': torch.zeros_like(p)}
    assert f(opt, m) is not None


class _FakeEngine:
    def __init__(self, n, d, L):
        self.m, self.v = torch.zeros(n, d), torch.zeros(n, d)
        self.Wm, self.Wv = torch.zeros(L, 2 * d, d), torch.zeros(L, 2 * d, d)
        self.step_dev = torch.zeros(1, dtype=torch.int32)
        self.refreshed = 0

    def _refresh_adam_coefs(self):
        self.refreshed += 1


def test_state_handover_maps_every_parameter_to_the_packed_moments():
    from arlib_b200.recommender.NGCF import NGCF
    d, L, U, I = 4, 2, 3, 5
    m = _ngcf_like(d, L, U, I)
    rec = NGCF.__new__(NGCF)
    opt = torch.optim.Adam(m.parameters(), lr=0.1)
    eng = _FakeEngine(U + I, d, L)
    rec._adam_state_to_engine(opt, m, eng, U)                  # no state yet: the engine keeps its zeros
    assert eng.refreshed == 0 and int(eng.step_dev) == 0
    # engine -> optimizer: state created lazily, each parameter's block of the packed moments
    eng.m.copy_(torch.arange((U + I) * d, dtype=torch.float32).view(U + I, d))
    eng.v.copy_(eng.m * 2)
    eng.Wm.copy_(torch.arange(L * 2 * d * d, dtype=torch.float32).view(L, 2 * d, d) + 1000)
    eng.Wv.copy_(eng.Wm * 3)
    eng.step_dev.fill_(11)
    rec._adam_state_from_engine(opt, m, eng, U)
    e, W = m.embedding_dict, m.W
    want = {e['user_emb']: eng.m[:U], e['item_emb']: eng.m[U:]}
    for k in range(L):
        want[W['w1_%d' % k]] = eng.Wm[k, :d]
        want[W['w2_%d' % k]] = eng.Wm[k, d:]
    assert len(opt.state) == 2 + 2 * L
    for p, ref in want.items():
        st = opt.state[p]
        assert float(st['step']) == 11.0 and torch.equal(st['exp_avg'], ref)
    assert torch.equal(opt.state[W['w2_1']]['exp_avg_sq'], eng.Wv[1, d:])
    # optimizer -> a fresh engine: the same blocks and the step counter
    eng2 = _FakeEngine(U + I, d, L)
    rec._adam_state_to_engine(opt, m, eng2, U)
    assert torch.equal(eng2.m, eng.m) and torch.equal(eng2.v, eng.v)
    assert torch.equal(eng2.Wm, eng.Wm) and torch.equal(eng2.Wv, eng.Wv)
    assert int(eng2.step_dev) == 11 and eng2.refreshed == 1
    # and the optimizer still steps on its own afterwards
    for p in m.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    assert float(opt.state[W['w1_0']]['step']) == 12.0
