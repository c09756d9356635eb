"""rl.ValueNetwork.forward_views / forward_both / RecordRing.experience_values: the value network on gathered views of ONE
perspective-0 feature batch (astro_value_forward_views, value_forward_kernel with an index and a view per output).

- The PyTorch form (autograd, CPU, float64) is the gather, the column exchange of ship 1's view and forward_torch; under
  autograd forward_both back-propagates exactly as before.  Bad inputs raise before anything is evaluated.
- On the GPU every output equals astro_value_forward on the materialised view, bit for bit: forward_both on
  observe(shared=True) equals forward() on observe(), forward_views equals the kernel on the gathered tensor (index -1 and
  all-masked items included), experience_values equals the network on experiences()' feature tensors, and the plain path
  (no index, no view) is the identity gather.  The new forms stay within forward64's bound and launch value_forward_kernel
  alone."""
import numpy as np
import pytest

from astro_b200 import core
from tests import helpers as H
from tests.test_value_network_forms import _batch, _feature_batch, form_of, forward64, make_net, net_params

SWAP = [0, 6, 7, 8, 9, 10, 1, 2, 3, 4, 5, 11, 12, 13, 14]


def _views_by_hand(x, index, view):
    """x [M, N, D] -> [E, N, D]: item index[e] (all -1 for index -1), ship 1's columns where view[e] is set, one by one."""
    import torch
    out = []
    for e, i in enumerate(index.tolist()):
        item = torch.full_like(x[0], -1.0) if i == -1 else x[i]
        if view is not None and int(view[e]):
            item = item[:, SWAP]
        out.append(item)
    return torch.stack(out)


def _random_views(M, E, seed, device='cpu', with_view=True):
    import torch
    g = torch.Generator().manual_seed(seed)
    index = torch.randint(-1, M, (E,), generator=g)
    index[:4] = torch.tensor([-1, 0, M - 1, 0])                 # terminal, repeats, the last item
    view = torch.randint(0, 2, (E,), generator=g).to(torch.uint8) if with_view else None
    return index.to(device), None if view is None else view.to(device)


# ------------------------------------------------------------------ CPU: the PyTorch form

def test_torch_form_equals_forward_torch_on_gathered_rows():
    """forward_views in PyTorch (CPU float32 and float64, duel and solo) = forward_torch on the rows gathered one by one:
    repeats, index -1, both views; E = 0 gives [0, nout]."""
    import torch
    for S, dtype in ((2, torch.float32), (2, torch.float64), (1, torch.float32)):
        net = make_net(S, 6, 3.0, 4 + S).to(dtype)
        x = torch.from_numpy(_feature_batch(40, 13, S, 7)[0]).to(dtype)
        index, view = _random_views(40, 203, S, with_view=S == 2)
        assert (index == -1).any() and len(set(index.tolist())) < 200
        with torch.no_grad():
            got = net.forward_views(x, index, view)
            want = net.forward_torch(_views_by_hand(x, index, view))
            assert got.shape == (203, 6) and got.dtype == dtype and torch.equal(got, want), S
            assert net.forward_views(x, index[:0], None if view is None else view[:0]).shape == (0, 6)
    # forward_both's pairs are forward_views of (item, ship 0), (item, ship 1)
    net = make_net(2, 6, 1.0, 2)
    x = torch.from_numpy(_feature_batch(20, 9, 2, 3)[0])
    with torch.no_grad():
        both = net.forward_both(x)
        views = net.forward_views(x, torch.arange(20).repeat_interleave(2), torch.arange(40).remainder(2).to(torch.uint8))
    assert float((both.reshape(40, 6) - views).abs().max()) <= 1e-6


def _forward_both_before(net, x):
    """forward_both as it was before the kernel routing (the first layer's weight with exchanged columns)."""
    import torch
    swap = torch.tensor(SWAP, device=x.device)
    w = torch.cat((net.f0.weight, net.f0.weight[:, swap]), dim=0)
    b = torch.cat((net.f0.bias, net.f0.bias), dim=0)
    h = torch.nn.functional.linear(x, w, b).unflatten(-1, (2, -1)).movedim(-2, -3)
    for layer in net.f:
        h = layer(net.activation(h))
    h = net.pool(h, features=x.unsqueeze(-3))
    for layer in net.v:
        h = net.activation(layer(h))
    return torch.tanh(net.v0(h))


def test_forward_both_under_autograd_backpropagates_as_before():
    """With autograd on, forward_both is the PyTorch code it was: the same outputs and the same gradients for every
    parameter and for the features; solo features still raise."""
    import torch
    grads = []
    for fn in (lambda n, x: n.forward_both(x), _forward_both_before):
        net = make_net(2, 6, 3.0, 9)
        x = torch.from_numpy(_feature_batch(24, 11, 2, 5)[0]).reshape(2, 12, 11, 15).requires_grad_()
        q = fn(net, x)
        (q * torch.linspace(-1, 1, q.numel()).reshape(q.shape)).sum().backward()
        grads.append([q.detach()] + [p.grad for p in net.parameters()] + [x.grad])
    assert grads[0][0].shape == (2, 12, 2, 6)
    for a, b in zip(*grads):
        assert torch.equal(a, b)
    with pytest.raises(ValueError):
        make_net(1, 6, 1.0, 1).forward_both(torch.zeros((4, 8, 10)))


def test_forward_views_rejects_bad_inputs_before_evaluating(monkeypatch):
    """dtype, shape, device and range errors raise ValueError before the network is evaluated."""
    import torch
    from astro_b200 import rl
    net, solo = make_net(2, 6, 1.0, 1), make_net(1, 6, 1.0, 1)
    monkeypatch.setattr(rl.ValueNetwork, 'forward_torch', lambda self, x: pytest.fail('evaluated'))
    x, xs = torch.zeros((5, 8, 15)), torch.zeros((5, 8, 10))
    i, v = torch.tensor([0, 4, -1]), torch.tensor([0, 1, 1], dtype=torch.uint8)
    bad = [(net, x[0], i, v), (net, xs, i, None), (net, x[:, :0], i, v), (net, x.long(), i, v),
           (net, x, i.int(), v), (net, x, i[None], v[None]), (net, x, [0, 1], None),
           (net, x, i, v.bool()), (net, x, i, v[:2]), (solo, xs, i, v),
           (net, x, torch.tensor([0, 5]), None), (net, x, torch.tensor([-2, 0]), None), (net, x[:0], torch.tensor([-1, 0]), None)]
    for n, xx, ii, vv in bad:
        with pytest.raises(ValueError):
            n.forward_views(xx, ii, vv)
    with pytest.raises(ValueError, match='outside -1 .. 4'):
        net.forward_views(x, torch.tensor([3, 5, -1]), None)


def test_views_abi_refuses_bad_arguments_before_touching_the_batch():
    """astro_value_forward_views checks its arguments before the batch handle: negative sizes, rows < 1, more outputs than
    items without an index (output e would read item e past the buffer, or through a NULL features pointer when there are
    no items) and missing features / q_out pointers are ASTRO_E_INVALID with a message naming them; arguments that pass
    reach the handle check."""
    from astro_b200 import _native as nat
    L, p = nat.lib(), 1 << 20                     # (p: a stand-in pointer, never dereferenced on these paths)
    for args, msg in (((-1, 8, None, None, 4, p), b'n_out >= 0'), ((100, 8, None, None, -4, p), b'n_out >= 0'),
                      ((100, 0, None, None, 4, p), b'rows >= 1'), ((100, 8, None, None, 200, p), b'n_out <= n_items'),
                      ((0, 8, None, None, 4, p), b'n_out <= n_items'), ((100, 8, p, None, 4, None), b'null features or q_out')):
        n_items, rows, index, view, n_out, q = args
        features = None if n_items == 0 else p
        assert L.astro_value_forward_views(None, features, n_items, rows, index, view, n_out, q, None) == -1, args
        assert msg in L.astro_last_error(), (args, L.astro_last_error())
    assert L.astro_value_forward_views(None, None, 100, 8, None, None, 4, p, None) == -1
    assert L.astro_last_error() == b'null features or q_out'
    for args in ((p, 100, 8, None, None, 100, p), (p, 100, 8, None, None, 40, p), (None, 0, 8, p, None, 4, p)):
        assert L.astro_value_forward_views(None, *args, None) == -1 and L.astro_last_error() == b'null batch handle', args


# ------------------------------------------------------------------ GPU: bit for bit against the materialised views

def _value_form(din):
    return ('value_forward_kernel', din)


@pytest.mark.gpu
@pytest.mark.parametrize('PL', [4, 8])
def test_forward_both_equals_forward_on_both_views_bit_for_bit(PL):
    """forward_both(observe(shared=True)) == forward(observe()) (value_forward_kernel on the two-view tensor) on both views,
    bit for bit: 1005 games (not a multiple of 16), finished games, bullet caps 4, 32 and 100, n_rows at the default and 8
    more; forward_both launches value_forward_kernel<15> alone."""
    import torch

    def run():
        for K in (4, 32, 100):
            games = _batch(32, 2, PL, 1005, K, seed=K + PL)
            assert games.get_arrays()['finished'].any()
            net = make_net(2, 6, 3.0, K).cuda()
            default = -(-(PL + K) // 4) * 4
            for n_rows in (default, default + 8):
                full = games.observe(n_rows)
                shared = games.observe(n_rows, shared=True)
                with torch.no_grad():
                    want = net(full)
                    got = net.forward_both(shared)
                assert got.shape == want.shape == (1005, 2, 6)
                assert torch.equal(got, want), (K, n_rows, float((got - want).abs().max()))
    _, forms = H.launched(run, form_of)
    assert {f for f in forms if f[0] != 'observe_kernel'} == {_value_form(15)}, forms


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [5, 13, 36])
def test_forward_views_equal_the_kernel_on_the_gathered_tensor(rows):
    """forward_views with random indices (repeats, -1, both views; 1003 outputs: a ragged last group) == value_forward on
    the materialised gather, bit for bit, duel and solo; all-masked items (no live row) among the gathered ones.  Indices
    outside -1 .. M - 1 passed to the library directly give NaN rows and leave every other row as it was."""
    import torch
    from astro_b200 import _native as nat
    from astro_b200 import rl
    for S in (2, 1):
        x_h, _ = _feature_batch(300, rows, S, 11 * rows + S)
        x = torch.from_numpy(x_h).cuda()
        index, view = _random_views(300, 1003, rows + S, 'cuda', with_view=S == 2)
        masked = (x[index.clamp(min=0), :, 0] < 0).all(dim=1) & (index >= 0)
        assert masked.any() and (index == -1).any()
        net = make_net(S, 6, 3.0, rows).cuda()
        with torch.no_grad():
            got = net.forward_views(x, index, view)
            g = rl._games(S == 1, 32, 32, x.device.index)
            want = g.value_forward(rl.ValueNetwork._gather_views(x, index, view).contiguous())
        assert torch.equal(got, want), (S, float((got - want).abs().max()))
        # out of range through the C ABI: NaN rows, nothing read
        bad = index.clone()
        bad[5], bad[6], bad[1002] = 300, -2, 1 << 40
        q = torch.zeros_like(got)
        nat.check(nat.lib().astro_value_forward_views(g._h, x.data_ptr(), 300, rows, bad.data_ptr(),
                                                      None if view is None else view.data_ptr(), 1003, q.data_ptr(),
                                                      g._stream()))
        nan = torch.zeros(1003, dtype=torch.bool, device='cuda')
        nan[[5, 6, 1002]] = True
        assert q[nan].isnan().all() and torch.equal(q[~nan], got[~nan])


@pytest.mark.gpu
def test_forward_views_within_the_float64_bound():
    """forward_views and forward_both stay within forward64's bound B of the float64 network on the materialised views, at
    weight scales 1, 3 and 10 and nout 1, 6 and 8, with hot rows, all-masked items and index -1; only
    value_forward_kernel<15> is launched."""
    import torch

    def run():
        worst = 0.0
        for c, (scale, nout) in enumerate(((1, 6), (3, 8), (10, 1), (1, 1), (3, 6), (10, 8))):
            x_h, _ = _feature_batch(257, 21, 2, 40 + c)
            x = torch.from_numpy(x_h).cuda()
            index, view = _random_views(257, 777, c, 'cuda')
            net = make_net(2, nout, float(scale), 20 + c, route=True).cuda()
            with torch.no_grad():
                got = torch.cat((net.forward_views(x, index, view), net.forward_both(x).reshape(-1, nout)))
            idx = np.concatenate([index.cpu().numpy(), np.arange(257).repeat(2)])
            vw = np.concatenate([view.cpu().numpy(), np.tile([0, 1], 257)])
            xm = np.where((idx < 0)[:, None, None], np.float32(-1), x_h[np.maximum(idx, 0)])
            xm = np.where(vw[:, None, None] != 0, xm[..., SWAP], xm)
            want, B = forward64(net_params(net), xm)
            ratio = np.abs(got.cpu().numpy().astype(np.float64) - want) / B
            worst = max(worst, float(ratio.max()))
            assert (ratio <= 1).all(), (scale, nout, float(ratio.max()), np.argwhere(ratio > 1)[:4])
        print('worst |forward_views - float64| / B: %.3g' % worst)
    _, forms = H.launched(run, form_of)
    assert forms == {_value_form(15)}, forms


@pytest.mark.gpu
@pytest.mark.parametrize('din', [15, 10])
def test_plain_path_equals_identity_views(din):
    """astro_value_forward (no index, no view) == forward_views with index = arange(n) and view 0, bit for bit; the library
    refuses a view array on solo features, negative sizes, rows < 1 and missing pointers, launching nothing."""
    import torch
    from astro_b200 import _native as nat
    from astro_b200 import rl
    S = 1 if din == 10 else 2
    x = torch.from_numpy(_feature_batch(1031, 36, S, din)[0]).cuda()
    net = make_net(S, 8, 3.0, din).cuda()
    g = rl._games(S == 1, 32, 32, x.device.index)
    with torch.no_grad():
        plain = net(x)
        ar = torch.arange(1031, device='cuda')
        assert torch.equal(net.forward_views(x, ar, None), plain)
        if S == 2:
            assert torch.equal(net.forward_views(x, ar, torch.zeros(1031, dtype=torch.uint8, device='cuda')), plain)
    L, h, st = nat.lib(), g._h, g._stream()
    q = torch.zeros((4, 8), device='cuda')
    v = torch.zeros(4, dtype=torch.uint8, device='cuda')
    before = g.launches
    if S == 1:
        assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, ar.data_ptr(), v.data_ptr(), 4, q.data_ptr(), st) == -1
    assert L.astro_value_forward_views(h, x.data_ptr(), -1, 36, None, None, 4, q.data_ptr(), st) == -1
    assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, None, None, -4, q.data_ptr(), st) == -1
    assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 0, None, None, 4, q.data_ptr(), st) == -1
    assert L.astro_value_forward_views(h, None, 1031, 36, None, None, 4, q.data_ptr(), st) == -1
    assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, None, None, 4, None, st) == -1
    assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, None, None, 0, None, st) == 0
    assert L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, None, None, 1032, q.data_ptr(), st) == -1   # item 1031
    assert L.astro_value_forward_views(h, None, 0, 36, None, None, 4, q.data_ptr(), st) == -1
    with pytest.raises(ValueError):
        net.forward_views(x, torch.tensor([0, 1031], device='cuda'), None)
    assert g.launches == before
    # without an index and fewer outputs than items: the first n_out items, as the plain path gives them
    head = torch.full((1000, 8), float('nan'), device='cuda')
    nat.check(L.astro_value_forward_views(h, x.data_ptr(), 1031, 36, None, None, 1000, head.data_ptr(), st))
    assert torch.equal(head, plain[:1000])
    # no items at all, every index -1: the all -1 item, with nothing read (features NULL)
    neg = torch.full((5,), -1, dtype=torch.int64, device='cuda')
    q5 = torch.full((5, 8), float('nan'), device='cuda')
    nat.check(L.astro_value_forward_views(h, None, 0, 36, neg.data_ptr(), None, 5, q5.data_ptr(), st))
    with torch.no_grad():
        assert torch.equal(q5, net(torch.full((5, 36, din), -1.0, device='cuda')))
    from astro_b200.batched import BatchedGames
    fresh = BatchedGames(core.SOLO_CONFIG if S == 1 else core.DEFAULT_CONFIG, 32)
    assert L.astro_value_forward_views(fresh._h, x.data_ptr(), 1031, 36, None, None, 4, q.data_ptr(), st) == -3   # no weights


# ------------------------------------------------------------------ GPU: recorded rings

@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['pool', 'fresh', 'solo'])
def test_experience_values_equal_the_network_on_experiences(mode):
    """Three consecutive windows of 100 explore ticks (n_steps 100, a ring of 201 rows): experience_values == net on
    experiences()' features / next_features, bit for bit, with identical pairs and metadata, carried and terminal pairs
    among them; its peak allocation stays below one E x n_rows x D float32 tensor.  A 4-slot batch with a reset pool, the
    same in fresh-game mode, and solo games (no view array)."""
    import torch
    from tests.test_rollout_record import _batch as ring_batch, _net
    cfg = core.DEFAULT_CONFIG._replace(solo=True) if mode == 'solo' else core.DEFAULT_CONFIG
    N, T, n_steps = 1024, 100, 100
    net = _net(cfg.solo)
    g = ring_batch(cfg, N, net, fresh=mode == 'fresh')
    ring = g.record_ring(n_steps + T + 1)
    carry = None
    n_carried = n_terminal = 0
    for w in range(3):
        s0 = g.step_index
        g.rollout_device(T, bots='explore', record=ring)
        rew, dis, nxt, carry = g.nstep_experiences(ring.window_events(T), carry, n_steps=n_steps, discount=0.995)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with torch.no_grad():
            got = ring.experience_values(net, rew, dis, nxt, n_steps)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        exp = ring.experiences(rew, dis, nxt, n_steps)
        E = int(exp['terminal'].shape[0])
        assert E > 0 and peak < E * ring.n_rows * ring.D * 4, (peak, E)
        with torch.no_grad():
            want_q, want_n = net(exp['features']), net(exp['next_features'])
        assert torch.equal(got['q'], want_q) and torch.equal(got['next_q'], want_n), w
        for key in ('action', 'reward', 'discount', 'terminal', 'game', 'ship', 'tick'):
            assert torch.equal(got[key], exp[key]), (w, key)
        n_carried += int((got['tick'] < s0).sum())
        n_terminal += int(got['terminal'].sum())
    assert n_carried > 0 and n_terminal > 0
