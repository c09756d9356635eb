"""Every observation and value-network kernel instantiation, each checked against the oracle's features or against a float64
network with a derived error bound.

observe_impl / astro_policy_controls / astro_value_forward (astro_b200.cu) choose observe_kernel<R, S, BOTH, PL> (12 forms),
policy_mma_kernel<R, S, PL> (8) and value_forward_kernel<DIN> (2) from the batch layout.  LEDGER lists all 22 and the tests
that launch each one; a CPU test holds it to the symbols of the built library, and every GPU test asserts, through
torch.profiler, that it launched exactly the network forms it is about.

- observe: bit for bit against a vectorised restatement of the oracle's ao_features (itself checked against ao_features
  on sampled games, bearing edge cases included), at bullet caps up to the largest n_rows the staging buffer takes, with
  ragged batches, finished games and every planet / bullet count; n_rows one step past the limit is refused unlaunched.
- policy_mma_kernel and value_forward_kernel: within the bound B of forward64() of the float64 network, at weight scales
  1, 3 and 10 and nout 1, 6 and 8; the control equals the float64 argmax wherever the top two are more than 2B apart, and
  exact ties take the lower index.  A planted "hot" row, one object per game whose feature alone sets one unit's maximum,
  swept over every position of the 8-row chunks, makes a dropped, repeated or foreign row change the outputs by far
  more than B."""
import re

import numpy as np
import pytest

from astro_b200 import core
from oracle import astro_oracle as ao
from tests import helpers as H


# ------------------------------------------------------------------ kernel names and the ledger

_FORM = re.compile(r'\b(observe_kernel|policy_mma_kernel|value_forward_kernel)<([^<>]*)>')


def form_of(name):
    """A network kernel's name, as CUPTI writes it (`observe_kernel<float, 2, true, 4>`) or as cu++filt does
    (`observe_kernel<float, (int)2, (bool)1, (int)4>`), as a tuple: ('observe_kernel', 'float', 2, 1, 4).  None for any
    other kernel."""
    m = _FORM.search(name)
    if m is None:
        return None
    out = [m.group(1)]
    for a in m.group(2).split(','):
        a = re.sub(r'^\((?:int|bool)\)', '', a.strip())
        out.append({'true': 1, 'false': 0}.get(a, int(a) if a.isdigit() else a))
    return tuple(out)


OBSERVE_CASES = [(r, S, view, PL) for r in ('float', 'double') for S, view in ((1, 'solo'), (2, 'both'), (2, 'shared'))
                 for PL in (4, 8)]
POLICY_CASES = [(r, S, PL) for r in ('float', 'double') for S in (1, 2) for PL in (4, 8)]


def observe_form(r, S, view, PL):
    return ('observe_kernel', r, S, int(view == 'both'), PL)


def policy_form(r, S, PL):
    return ('policy_mma_kernel', r, S, PL)


def value_form(din):
    return ('value_forward_kernel', din)


PRODUCTION_POLICY = policy_form('float', 2, 4)


def _ledger():
    led = {}

    def add(test, *forms):
        for f in forms:
            led.setdefault(f, []).append(test)
    for c in OBSERVE_CASES:
        add('test_observe_matches_the_oracle_bit_for_bit', observe_form(*c))
    for c in POLICY_CASES:
        add('test_policy_matches_the_float64_network', policy_form(*c))
    add('test_policy_hot_row_over_every_chunk_offset', PRODUCTION_POLICY, policy_form('double', 1, 8))
    add('test_policy_ties_take_the_lower_index_and_masks_write_their_columns', PRODUCTION_POLICY)
    for din in (10, 15):
        add('test_value_forward_matches_the_float64_network', value_form(din))
    return {f: tuple(t) for f, t in led.items()}


LEDGER = _ledger()


def test_network_kernel_names_parse_in_both_spellings():
    assert form_of('void (anonymous namespace)::observe_kernel<float, 2, true, 4>(const void *, int)') \
        == ('observe_kernel', 'float', 2, 1, 4)
    assert form_of('void <unnamed>::observe_kernel<double, (int)1, (bool)0, (int)8>(const void *, int)') \
        == ('observe_kernel', 'double', 1, 0, 8)
    assert form_of('void <unnamed>::policy_mma_kernel<float, (int)2, (int)4>(const void *)') == PRODUCTION_POLICY
    assert form_of('void (anonymous namespace)::policy_mma_kernel<double, 1, 8>(const void *)') \
        == ('policy_mma_kernel', 'double', 1, 8)
    assert form_of('void <unnamed>::value_forward_kernel<(int)15>(const float *)') == value_form(15)
    assert form_of('void (anonymous namespace)::value_forward_kernel<10>(const float *)') == value_form(10)
    assert form_of('void <unnamed>::tick_kernel<double, (int)1, (bool)0, (int)8>(<unnamed>::TickParams)') is None


def test_library_network_forms_equal_the_ledger():
    """The built library's observe / policy / value-forward instantiations are exactly the ledger's 22 keys, and every test
    the ledger names exists here: a form added to the library without a test that launches it fails here, with no GPU."""
    forms = [f for f in map(form_of, H.library_kernel_names()) if f is not None]
    assert len(forms) == len(set(forms)) == 22
    assert set(forms) == set(LEDGER), (sorted(set(forms) - set(LEDGER)), sorted(set(LEDGER) - set(forms)))
    for form, tests in LEDGER.items():
        assert tests, form
        for t in tests:
            assert callable(globals().get(t)) and t.startswith('test_'), (form, t)


def _expect(forms, fn):
    """fn() must launch exactly the network forms `forms`, each at least once, and each must be in the ledger under the
    calling test."""
    import inspect
    test = next(f.function for f in inspect.stack(0) if f.function.startswith('test_'))
    for f in forms:
        assert test in LEDGER[f], (test, f)
    result, got = H.launched(fn, form_of)
    assert got == set(forms), (sorted(set(forms) - got), sorted(got - set(forms)))
    return result


# ------------------------------------------------------------------ games and the feature reference

def edge_bearings():
    """Bearings where util.norm_angle's floored remainder turns: 0, +-pi, (2k - 1) pi and 2 pi k with their float64
    neighbours, the float32 roundings of all of them, and values at the +-71,476 rad guard of set_arrays."""
    pi, up, dn = np.pi, (lambda v: np.nextafter(v, np.inf)), (lambda v: np.nextafter(v, -np.inf))
    vals = [0.0, -0.0, 71476.0, -71476.0, dn(71476.0), up(-71476.0), 71475.5, -71475.5, 71471.0, -71471.0]
    for k in (1, 2, 3, 7, 50, 11375, 11376):
        for c in (2 * pi * k, (2 * k - 1) * pi):
            for v in (c, -c):
                vals += [v, up(v), dn(v)]
    vals = np.array(vals)
    vals = np.concatenate([vals, vals.astype(np.float32).astype(np.float64)])
    return vals[np.abs(vals) <= 71476.0]


def features_ref(arr, S, n_rows):
    """The padded feature tensor [n, S, n_rows, D] float32 of get_arrays() output `arr`: view q = game seen by ship q
    (core.roll_ships), rows = planets, bullets, then -1 (finished games: all -1) — ao_features for every game and view."""
    ships, planets, bullets = arr['ships'], arr['planets'], arr['bullets']
    n, PL, K = ships.shape[0], planets.shape[1], bullets.shape[1]
    D = 1 + 5 * S + 4
    npl = np.where(arr['finished'], 0, arr['n_planets']).astype(np.int64)
    nb = np.where(arr['finished'], 0, arr['n_bullets']).astype(np.int64)
    sf = np.empty((n, S, 5), dtype=np.float32)
    sf[..., :4] = ships[..., :4]
    sf[..., 4] = ao.norm_angle(ships[..., 4]) / np.pi
    objs = np.concatenate([planets, bullets, np.zeros((n, 1, 4))], axis=1)
    r = np.arange(n_rows)[None, :]
    live = r < (npl + nb)[:, None]
    src = np.where(live, np.where(r < npl[:, None], r, PL + r - npl[:, None]), PL + K)
    obj = np.take_along_axis(objs, src[..., None], axis=1).astype(np.float32)
    out = np.empty((n, S, n_rows, D), dtype=np.float32)
    for q in range(S):
        out[:, q, :, 0] = np.where(r < npl[:, None], 0.0, 1.0)
        for k in range(S):
            out[:, q, :, 1 + 5 * k:6 + 5 * k] = sf[:, (k + q) % S][:, None, :]
        out[:, q, :, 1 + 5 * S:] = obj
    out[np.broadcast_to(~live[:, None, :], out.shape[:3])] = -1.0
    return out


def random_games(n, S, PL, K, seed, fin=0.05):
    """set_arrays() inputs of n games: random ships (one bearing in three an edge_bearings() value), every planet count
    1..PL, bullet counts over 0..K with 0 and K frequent, and a share `fin` of finished games."""
    r = np.random.RandomState(seed)
    ships = np.concatenate([r.uniform(-1, 1, (n, S, 2)), r.uniform(-0.3, 0.3, (n, S, 2)), r.uniform(-250, 250, (n, S, 1))], axis=2)
    b = ships[..., 4].reshape(-1)
    e = edge_bearings()
    sel = np.arange(0, b.size, 3)
    b[sel] = e[np.arange(sel.size) % e.size]
    ships[..., 4] = b.reshape(n, S)
    planets = np.concatenate([r.uniform(-0.8, 0.8, (n, PL, 2)), r.uniform(-0.1, 0.1, (n, PL, 2))], axis=2)
    npl = 1 + r.permutation(np.arange(n) % PL)
    nb = r.randint(0, K + 1, n)
    nb[r.rand(n) < 0.1] = K
    nb[r.rand(n) < 0.1] = 0
    bullets = np.concatenate([r.uniform(-1.3, 1.3, (n, K, 2)), r.uniform(-2, 2, (n, K, 2))], axis=2)
    return ships, planets, npl, bullets, nb, r.rand(n) < fin


def _config(S, PL):
    cfg = core.SOLO_CONFIG if S == 1 else core.DEFAULT_CONFIG
    return cfg._replace(max_planets=PL)


def _batch(precision, S, PL, N, K, seed, fin=0.05):
    from astro_b200.batched import BatchedGames
    g = BatchedGames(_config(S, PL), N, bullet_cap=K, precision=precision, seed=seed)
    ships, planets, npl, bullets, nb, finished = random_games(N, S, PL, K, seed, fin)
    g.set_arrays(ships, planets, npl, bullets, nb, np.zeros(N, dtype=np.int64), finished=finished)
    return g


def test_feature_reference_equals_ao_features():
    """features_ref == ao_features, bit for bit, on sampled games of every layout: both ship counts, 4 and 8 planet
    slots, bullet caps 0, 33 and 208, the bearing edge cases, finished games, default and larger n_rows."""
    n_edge = 0
    for S in (1, 2):
        for PL in (4, 8):
            for K in (0, 33, 208):
                ships, planets, npl, bullets, nb, fin = random_games(150, S, PL, K, S * 100 + PL + K, fin=0.1)
                for f32 in (False, True):
                    sh = ships.astype(np.float32).astype(np.float64) if f32 else ships
                    arr = dict(ships=sh, planets=planets, bullets=bullets, n_planets=npl, n_bullets=nb, finished=fin)
                    for n_rows in (PL + K, PL + K + 7):
                        got = features_ref(arr, S, n_rows)
                        for g in range(150):
                            for me in range(S):
                                if fin[g]:
                                    assert (got[g, me] == -1).all()
                                    continue
                                want = ao.features(S, sh[g], planets[g, :npl[g]], bullets[g, :nb[g]], me, n_rows)
                                assert H.same_bits(got[g, me], want), (S, PL, K, g, me)
                    n_edge += int(np.isin(sh[..., 4], edge_bearings()).sum())
    assert n_edge > 1000
    # the bearing feature turns where it should: -1 at -pi, +pi and 3 pi; just above pi wraps to just above -1
    v = (ao.norm_angle(np.array([np.pi, -np.pi, 3 * np.pi, np.pi + 1e-6])) / np.pi).astype(np.float32)
    assert (v[:3] == -1).all() and -1 < v[3] < -0.9999


# ------------------------------------------------------------------ the float64 network and its error bound

U = 2.0 ** -22


def net_params(net):
    """(weight, bias) of f0, f[0], f[1], v[0], v[1], v0 as float64 arrays of the float32 values."""
    return [(l.weight.detach().double().cpu().numpy(), l.bias.detach().double().cpu().numpy())
            for l in (net.f0, net.f[0], net.f[1], net.v[0], net.v[1], net.v0)]


def _e16(v):
    """Bound on |v - (hi + lo)| for the kernel's FP16 pair of a value of magnitude v (see forward64)."""
    return U * v + np.minimum(2.0 ** -25, 2.0 ** -11 * v)


def _injected(W, b, a, n_mma):
    """Bound on what one layer's arithmetic adds to its outputs (see forward64), a = the float64 input."""
    A, aW = np.abs(a), np.abs(W)
    M = A @ aW.T
    return 1.01 * (U * M + _e16(A) @ aW.T + A @ _e16(aW).T + (n_mma / 2 + 0.25) * U * (np.abs(b) + M))


def _softsign(z):
    """softsign, its slope, and the bound on the kernel's rounding of it."""
    s = z / (1.0 + np.abs(z))
    return s, 1.0 / (1.0 + np.abs(z)) ** 2, ROUND * np.abs(s)


def _absmv(M, v):
    return np.einsum('...jk,...k->...j', np.abs(M), v)


ROUND = 1.25 * U


def forward64(P, x, rows_chunk=1 << 14):
    """rl.ValueNetwork.forward of parameters P (net_params) on features x [n, rows, D] (float32) in float64, masked_max's
    x - 1e9 pad included, and a bound B with |kernel - float64| <= B per output.  Returns (q, B), [n, nout] each.

    What each step of the kernel adds (per layer y = b + sum_k w_k a_k, a its float32 input, w and b float32 weights):
    * FP16 split.  The kernel takes a = a_hi + a_lo + da, w = w_hi + w_lo + dw (each part FP16, the lo part what the hi part
      dropped, rounded) and sums a_lo w_hi + a_hi w_lo + a_hi w_hi: exact products of 11-bit operands.  What is dropped,
      a_lo w_lo + (a_hi + a_lo) dw + da w, is at most 2^-22 |a||w| + |a| e16(|w|) + e16(|a|) |w| (x 1.01), where
      e16(v) = 2^-22 v + min(2^-25, 2^-11 v): |a - a_hi| <= 2^-11 |a|, and rounding that to FP16 costs 2^-11 of it, or, in
      FP16's subnormal range, half its spacing 2^-24: the 2^-25 floor of each lo operand.
    * Accumulation (an assumption, not a measurement): each m16n8k16 adds its 16 exact products to its fp32 accumulator
      with an error of at most 2^-23 (|c| + sum |p|), one unit in the 24th bit of the magnitude sum (truncation as well
      as rounding); a layer takes n_mma of them (3 for f0: one k-step of three products; 6 for a 32-wide layer), plus
      half a unit for the value head's fma of the bias: (n_mma / 2 + 1 / 4) 2^-22 (|b| + sum |w| |a|).
    * Activations: the kernel's softsign (fast reciprocal) and tanhf are within 2 ulp of the function of their float32
      input, and the rounding of 1 + |x| moves softsign by at most half an ulp more: 1.25 x 2^-22 |v|.
    * Max-pool is 1-Lipschitz per unit: its error is at most the largest error of the rows it pools.  A padding row's
      x - 1e9 is rounded to float32 (2^-24 (1e9 + |x|)); it decides the maximum only for an item without a live row.
    Each of these reaches the outputs through the network's Jacobian from that point on, evaluated at the float64 values:
    B = sum over the steps of |J| e (absolute values of the composed Jacobian, not the product of absolute weights, which
    would be loose by about sqrt(32) per layer), the pool taken as above.  This is the first-order bound: what it drops
    is quadratic in errors of relative size ~1e-5, which the factor 1.05 covers; the softsign and tanh slopes (at most 1,
    1 / (1 + |z|)^2 far out) are what keep the 1e9 path bounded."""
    (W0, b0), (W1, b1), (W2, b2), (V1, c1), (V2, c2), (V0, c0) = P
    n, R, _ = x.shape
    step = max(1, rows_chunk // max(R, 1))
    qs, bs = [], []
    for i in range(0, n, step):
        xc = x[i:i + step]
        a = xc.astype(np.float64)
        z0 = a @ W0.T + b0
        s0, d0, r0 = _softsign(z0)
        z1 = s0 @ W1.T + b1
        s1, d1, r1 = _softsign(z1)
        z2 = s1 @ W2.T + b2
        J1 = W2 * d1[..., None, :]                                   # dz2 / dz1, per row
        J0 = (J1 @ W1) * d0[..., None, :]                            # dz2 / dz0
        e = (_injected(W2, b2, s1, 6) + _absmv(J1, _injected(W1, b1, s0, 6)) + r1 @ np.abs(W2).T
             + _absmv(J1 @ W1, r0) + _absmv(J0, _injected(W0, b0, a, 3)))
        pad = (xc[..., 0] < 0)[..., None]
        none = pad.all(axis=1, keepdims=True)
        e = np.where(pad, np.where(none, e + 2.0 ** -24 * (1e9 + np.abs(z2)), 0.0), e).max(axis=1)
        p = (z2 - 1e9 * pad).max(axis=1)
        z3 = p @ V1.T + c1
        s3, d3, r3 = _softsign(z3)
        z4 = s3 @ V2.T + c2
        s4, d4, r4 = _softsign(z4)
        z5 = s4 @ V0.T + c0
        q = np.tanh(z5)
        G = (1.0 - q ** 2)[..., None] * V0                          # dq / ds4
        B = ROUND * np.abs(q) + (1.0 - q ** 2) * _injected(V0, c0, s4, 6) + _absmv(G, r4)
        G = G * d4[..., None, :]                                     # dq / dz4
        B += _absmv(G, _injected(V2, c2, s3, 6))
        G = G @ V2                                                   # dq / ds3
        B += _absmv(G, r3)
        G = G * d3[..., None, :]                                     # dq / dz3
        B += _absmv(G, _injected(V1, c1, p, 6)) + _absmv(G @ V1, e)
        qs.append(q)
        bs.append(1.05 * B + 2.0 ** -140)
    return np.concatenate(qs), np.concatenate(bs)


def make_net(S, nout, scale, seed, route=False):
    """rl.ValueNetwork on the CPU, every parameter times `scale`.  route=True: unit 0 reads the object's dx alone
    (f0 row 0 = dx, f[0] and f[1] row 0 = 3 x unit 0, no bias), so the row of the largest dx holds unit 0's maximum after
    every per-object layer, and the head reads unit 0 with three times its usual weight."""
    import torch
    from astro_b200 import rl
    torch.manual_seed(seed)
    net = rl.ValueNetwork(solo=S == 1, nout=nout)
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(scale)
        if route:
            net.f0.weight[0] = 0.0
            net.f0.weight[0, 1 + 5 * S + 2] = 1.0
            net.f0.bias[0] = 0.0
            for layer in net.f:
                layer.weight[0] = 0.0
                layer.weight[0, 0] = 3.0
                layer.bias[0] = 0.0
            net.v[0].weight[:, 0] *= 3.0
    return net


def _synthetic_features(n, S, K, seed):
    ships, planets, npl, bullets, nb, fin = random_games(n, S, 4, K, seed, fin=0.0)
    arr = dict(ships=ships.astype(np.float32).astype(np.float64), planets=planets, bullets=bullets, n_planets=npl,
               n_bullets=nb, finished=fin)
    return features_ref(arr, S, 4 + K).reshape(n * S, 4 + K, -1)


def test_forward64_is_the_value_network_in_float64():
    """forward64's values are rl.ValueNetwork.forward_torch run in float64 on the same features (padding and an item
    without a live row included)."""
    import torch
    for S in (1, 2):
        x = _synthetic_features(64, S, 12, 3 + S)
        x[5] = -1.0                                          # no live row: the 1e9 path
        net = make_net(S, 6, 3.0, 1 + S)
        q, B = forward64(net_params(net), x)
        with torch.no_grad():
            want = net.double().forward_torch(torch.from_numpy(x).double()).numpy()
        assert np.abs(q - want).max() <= 1e-12
        assert (B > 0).all() and B[np.arange(len(B)) != 5].max() < 1e-3


def _emulate(P, x, form):
    """The kernel's network in numpy on items with a live row: float32 activations, each m16n8k16 as 16 exact products
    summed and rounded once to float32 into the accumulator; form 'three' = the kernel's split (a_lo w_hi, a_hi w_lo,
    a_hi w_hi), 'two' = without a_lo w_hi, 'hi' = a_hi w_hi alone."""
    def split(v):
        hi = v.astype(np.float16).astype(np.float32)
        return hi.astype(np.float64), (v - hi).astype(np.float16).astype(np.float64)

    terms = {'three': ((1, 0), (0, 1), (0, 0)), 'two': ((0, 1), (0, 0)), 'hi': ((0, 0),)}[form]

    def layer(W, b, a):
        k = -(-W.shape[1] // 16) * 16
        a = np.concatenate([a, np.zeros(a.shape[:-1] + (k - a.shape[-1],), np.float32)], axis=-1)
        W = np.concatenate([W.astype(np.float32), np.zeros((W.shape[0], k - W.shape[1]), np.float32)], axis=1)
        (ah, al), (wh, wl) = split(a), split(W)
        A, Wp = (ah, al), (wh, wl)
        acc = np.broadcast_to(b.astype(np.float32), a.shape[:-1] + (W.shape[0],)).copy()
        for s in range(0, k, 16):
            for ia, iw in terms:
                acc = (acc.astype(np.float64) + A[ia][..., s:s + 16] @ Wp[iw][:, s:s + 16].T).astype(np.float32)
        return acc

    soft = lambda v: (v / (np.float32(1) + np.abs(v))).astype(np.float32)
    (W0, b0), (W1, b1), (W2, b2), (V1, c1), (V2, c2), (V0, c0) = P
    h = layer(W0, b0, x)
    h = layer(W2, b2, soft(layer(W1, b1, soft(h))))
    h = np.where((x[..., 0] < 0)[..., None], np.float32(-3e38), h).max(axis=1)
    h = layer(V2, c2, soft(layer(V1, c1, h)))
    return np.tanh(layer(V0, c0, soft(h)).astype(np.float64))


@pytest.mark.parametrize('scale', [1, 3, 10])
def test_bound_holds_for_the_kernel_split_and_fails_for_weaker_ones(scale):
    """The bound has teeth: an emulation of the kernel's three-product split stays within B on every output (at under
    2 % of it), while the two-product form (no a_lo w_hi) and the hi x hi form exceed B on most outputs at weight scale
    1 and on a third to a half of them at scales 3 and 10, where tanh saturates and B's worst case over the pooled rows
    weighs more."""
    for S in (1, 2):
        x = _synthetic_features(150, S, 40, 11 * scale + S)
        P = net_params(make_net(S, 8, float(scale), 7 * scale + S))
        q, B = forward64(P, x)
        err = {f: np.abs(_emulate(P, x, f) - q) for f in ('three', 'two', 'hi')}
        assert (err['three'] <= 0.02 * B).all(), float((err['three'] / B).max())
        assert (err['two'] > B).mean() > 0.25, (S, float((err['two'] > B).mean()))
        assert (err['hi'] > B).mean() > 0.4, (S, float((err['hi'] > B).mean()))
        if scale == 1:
            assert (err['two'] > B).mean() > 0.5 and (err['hi'] > B).mean() > 0.7


# ------------------------------------------------------------------ observe against the oracle, all 12 forms

# the largest n_rows the 200 KB staging buffer of an observe CTA (8 warps) takes, and the next n_rows with n_rows * D a
# multiple of 4
ROW_LIMIT = {'both': (212, 216), 'shared': (424, 428), 'solo': (638, 640)}


def _observe(games, view, n_rows):
    return games.observe(n_rows, shared=view == 'shared')


def _check_observe(games, view, n_rows):
    S = games.S
    got = _observe(games, view, n_rows).cpu().numpy()
    want = features_ref(games.get_arrays(), S, n_rows)
    if view == 'shared':
        want = want[:, 0]
    assert got.shape == want.shape and H.same_bits(got, want), (view, n_rows, np.argwhere(got.view(np.uint32) != want.view(np.uint32))[:4])


@pytest.mark.gpu
@pytest.mark.parametrize('r,S,view,PL', OBSERVE_CASES, ids=['%s S=%d %s PL=%d' % c for c in OBSERVE_CASES])
def test_observe_matches_the_oracle_bit_for_bit(r, S, view, PL):
    """observe() == ao_features for every game and view, bit for bit: 1005 games (a ragged last tile), finished games,
    every planet count, bullet counts 0..K, the bearing edge cases; bullet caps 0, 1, 31, 33, 64 at the default n_rows and
    8 rows more, and the largest cap at the largest n_rows the staging buffer takes (the launch with more than 48 KB of
    dynamic shared memory)."""
    limit = ROW_LIMIT[view][0]
    N = 1005

    def run():
        for K in (0, 1, 31, 33, 64, limit - PL):
            games = _batch(64 if r == 'double' else 32, S, PL, N, K, seed=K + PL)
            arr = games.get_arrays()
            live = ~arr['finished']
            assert arr['finished'].any() and set(arr['n_planets'][live]) == set(range(1, PL + 1))
            assert (arr['n_bullets'][live] == K).any() and (arr['n_bullets'][live] == 0).any()
            default = -(-(PL + K) // 4) * 4
            for n_rows in ((limit,) if K == limit - PL else (default, default + 8)):
                _check_observe(games, view, n_rows)
    _expect([observe_form(r, S, view, PL)], run)


@pytest.mark.gpu
@pytest.mark.parametrize('PL', [4, 8])
def test_observe_refuses_n_rows_past_the_staging_limit(PL):
    """n_rows one step past the staging limit (216 both views, 428 shared, 640 solo), or below planet slots + bullet cap,
    is refused before any launch; the limit itself is taken (test_observe_matches_the_oracle_bit_for_bit)."""
    from astro_b200 import _native as nat
    for S, view in ((1, 'solo'), (2, 'both'), (2, 'shared')):
        games = _batch(32, S, PL, 64, 8, seed=1)
        before = games.launches
        for n_rows in (ROW_LIMIT[view][1], PL + 4):
            with pytest.raises(nat.AstroError):
                _observe(games, view, n_rows)
        assert games.launches == before


# ------------------------------------------------------------------ policy_mma_kernel against the float64 network

WORST = {}


def _record(form, ratio):
    WORST[form] = max(WORST.get(form, 0.0), float(ratio))
    print('worst |kernel - float64| / B  %s: %.3g' % (form, WORST[form]))


def _policy_run(games, net, nout):
    import torch
    games.set_policy(net)
    q = torch.full((games.n_pad, games.S, nout), float('nan'), dtype=torch.float32, device=games.device)
    act = games.policy_controls(q_out=q)
    return q[:games.n].cpu().numpy().astype(np.float64), act[:games.n].cpu().numpy().astype(np.int64)


def _check_policy(games, net, nout, form):
    """q and the controls of policy_controls against forward64 on features_ref of the same state; returns (q, want, B)."""
    S, N = games.S, games.n
    arr = games.get_arrays()
    q, act = _policy_run(games, net, nout)
    fin = arr['finished']
    assert (q[fin] == 0).all() and (act[fin] == 2).all()
    live = ~fin
    rows = int((arr['n_planets'][live] + arr['n_bullets'][live]).max())
    x = features_ref(arr, S, rows)[live].reshape(-1, rows, 1 + 5 * S + 4)
    want, B = forward64(net_params(net), x)
    got = q[live].reshape(-1, nout)
    ratio = np.abs(got - want) / B
    _record(form, ratio.max())
    assert (ratio <= 1).all(), (float(ratio.max()), np.argwhere(ratio > 1)[:4])
    top = np.sort(want, axis=1)[:, ::-1]
    clear = (top[:, 0] - top[:, 1] > 2 * B.max(axis=1)) if nout > 1 else np.ones(len(want), bool)
    assert clear.sum() > 40                          # (tanh saturates at scale 10: most top-two gaps are tiny there)
    assert (act[live].reshape(-1)[clear] == want.argmax(axis=1)[clear]).all()
    return q, want, B


@pytest.mark.gpu
@pytest.mark.parametrize('r,S,PL', POLICY_CASES, ids=['%s S=%d PL=%d' % c for c in POLICY_CASES])
def test_policy_matches_the_float64_network(r, S, PL):
    """policy_controls' q within B of the float64 network on the oracle's features, controls = the float64 argmax where the
    top two are more than 2B apart, finished games control 2 and q 0: bullet caps 0, 32 and 400 (up to 51 chunks of 8
    rows per game), each with its own nout (1, 6, 8) and weight scale (1, 3, 10), so every form meets every nout and
    scale; ragged batches, every planet count, the bearing edge cases."""
    f = POLICY_CASES.index((r, S, PL))

    def run():
        for i, K in enumerate((0, 32, 400)):
            nout, scale = (1, 6, 8)[(i + f) % 3], (1, 3, 10)[(i + 2 * f) % 3]
            games = _batch(64 if r == 'double' else 32, S, PL, 1005 if K < 400 else 333, K, seed=17 * f + i)
            _check_policy(games, make_net(S, nout, float(scale), 5 * f + i), nout, policy_form(r, S, PL))
    _expect([policy_form(r, S, PL)], run)


def _plant_hot_rows(games, seed):
    """One object per live game gets dx = 20 + 30 u (distinct per game, far above every other |dx| <= 2): a fifth of the
    games at row 0, a fifth at the last row, the rest spread over all rows.  Returns the hot rows and the row counts."""
    r = np.random.RandomState(seed)
    arr = games.get_arrays()
    n = games.n
    npl, nb = arr['n_planets'], arr['n_bullets']
    rows = npl + nb
    g = np.arange(n)
    hot = np.where(g % 5 == 0, 0, np.where(g % 5 == 1, rows - 1, r.randint(0, 1 << 30, n) % rows))
    planets, bullets = arr['planets'].copy(), arr['bullets'].copy()
    val = 20.0 + 30.0 * r.rand(n)
    in_pl = hot < npl
    planets[g[in_pl], hot[in_pl], 2] = val[in_pl]
    bullets[g[~in_pl], (hot - npl)[~in_pl], 2] = val[~in_pl]
    games.set_arrays(arr['ships'], planets, npl, bullets, nb, arr['tick'], finished=arr['finished'])
    return hot, rows


@pytest.mark.gpu
def test_policy_hot_row_over_every_chunk_offset():
    """A hot row per game (unit 0's maximum, make_net(route=True)) at every offset of the 8-row chunks, at the first and
    the last row, at bullet list positions past 32 and 256 in tiles whose lists hold thousands of items: q within B, and
    the float64 network without the hot row differs from q by more than 8B on most outputs — a dropped, repeated or
    foreign row cannot pass."""
    def run():
        for form, (r, S, PL) in ((PRODUCTION_POLICY, ('float', 2, 4)), (policy_form('double', 1, 8), ('double', 1, 8))):
            games = _batch(64 if r == 'double' else 32, S, PL, 1005, 400, seed=3, fin=0.02)
            hot, rows = _plant_hot_rows(games, 4)
            live = ~games.get_arrays()['finished']
            npl = games.get_arrays()['n_planets']
            assert set((hot % 8)[live & (rows > 8)]) == set(range(8)) and (hot - npl > 256)[live].any()
            net = make_net(S, 6, 3.0, 9, route=True)
            q, want, B = _check_policy(games, net, 6, form)
            arr = games.get_arrays()
            rows_max = int(rows[live].max())
            x = features_ref(arr, S, rows_max)[live]
            x[np.arange(x.shape[0]), :, hot[live], 1 + 5 * S + 2] = 0.0           # the hot value gone
            cold, _ = forward64(net_params(net), x.reshape(-1, rows_max, x.shape[-1]))
            assert (np.abs(cold - want) > 8 * B).mean() > 0.8
    _expect([PRODUCTION_POLICY, policy_form('double', 1, 8)], run)


@pytest.mark.gpu
def test_policy_ties_take_the_lower_index_and_masks_write_their_columns():
    """Outputs with the same v0 row and bias are the same q bit for bit; where they hold the maximum the control is the
    lower index, as torch.argmax: a tie inside one lane's pair (6, 7) and across lanes (1, 4, 5).  ship_mask 1, 2 and 3
    write only their columns."""
    import torch

    def run():
        games = _batch(32, 2, 4, 1005, 32, seed=8)
        fin = games.get_arrays()['finished']
        for dup in ((6, 7), (1, 4, 5)):
            net = make_net(2, 8, 3.0, 12)
            with torch.no_grad():
                net.v0.bias[:] = -2.0
                for k in dup:
                    net.v0.weight[k] = net.v0.weight[dup[0]]
                    net.v0.bias[k] = 2.0
            q, act = _policy_run(games, net, 8)
            live = ~fin
            qd = q[live][..., list(dup)]
            assert (qd == qd[..., :1]).all()
            top = q[live].max(axis=-1)
            at_dup = qd[..., 0] == top
            assert at_dup.mean() > 0.9
            assert (act[live][at_dup] == dup[0]).all()
        full = games.policy_controls()
        for ships in ([0], [1], [0, 1]):
            out = torch.full((games.n_pad, 2), 9, dtype=torch.uint8, device=games.device)
            games.policy_controls(out=out, ships=ships)
            for s in range(2):
                assert (out[:, s] == (full[:, s] if s in ships else 9)).all(), (ships, s)
    _expect([PRODUCTION_POLICY], run)


# ------------------------------------------------------------------ value_forward_kernel against the float64 network

VF_CASES = [(1, 4099), (7, 17), (8, 16), (9, 15), (36, 4099), (404, 33), (1031, 1), (1031, 17)]


def _feature_batch(n, rows, S, seed):
    """Features [n, rows, D] with live-row patterns by item i: (i + i // 8) % 4 = prefix, sparse, last row only, none (so
    the two items of a tile pair differ); padding rows have flag -1 and random other columns.  One live row per item with
    a live row is hot (dx = 20 + 30 u), its position swept over every chunk offset.  Returns features and hot rows."""
    r = np.random.RandomState(seed)
    D = 1 + 5 * S + 4
    x = np.concatenate([r.randint(0, 2, (n, rows, 1)), r.uniform(-1, 1, (n, rows, 5 * S)),
                        r.uniform(-1.3, 1.3, (n, rows, 2)), r.uniform(-2, 2, (n, rows, 2))], axis=2).astype(np.float32)
    i = np.arange(n)
    pattern = (i + i // 8) % 4
    ri = np.arange(rows)[None, :]
    live = np.where(pattern[:, None] == 0, ri < r.randint(1, rows + 1, n)[:, None],
                    np.where(pattern[:, None] == 1, r.rand(n, rows) < 0.3,
                             np.where(pattern[:, None] == 2, ri == rows - 1, False)))
    live[(pattern == 1) & ~live.any(axis=1), 0] = True
    x[..., 0] = np.where(live, x[..., 0], -1.0)
    hot = np.full(n, -1)
    for k in np.nonzero(live.any(axis=1))[0]:
        cand = np.nonzero(live[k])[0]
        hot[k] = cand[(k * 5) % cand.size]
        x[k, hot[k], D - 2] = 20.0 + 30.0 * r.rand()
    assert x.shape[2] == D
    return x, hot


@pytest.mark.gpu
@pytest.mark.parametrize('din', [10, 15])
def test_value_forward_matches_the_float64_network(din):
    """value_forward within B of the float64 network: rows 1 .. 1031, items 1 .. 4099 (partial 16-item groups), prefix /
    sparse / last-row / no live rows (the 1e9 path and its scaled head), a hot row per item over the chunk offsets and the
    padding-chunk skip, nout 1, 6 and 8 and weight scales 1, 3 and 10; without the hot row the float64 outputs move by
    more than 8B on most items."""
    import torch
    from astro_b200.batched import BatchedGames
    S = 1 if din == 10 else 2
    games = BatchedGames(_config(S, 4), 32, bullet_cap=32)

    def run():
        offsets = set()
        for c, (rows, n) in enumerate(VF_CASES):
            nout, scale = (1, 6, 8)[c % 3], (1, 3, 10)[(c + din) % 3]
            x, hot = _feature_batch(n, rows, S, 31 * c + din)
            net = make_net(S, nout, float(scale), c + din, route=True)
            games.set_policy(net)
            q = games.value_forward(torch.from_numpy(x).cuda()).cpu().numpy().astype(np.float64)
            want, B = forward64(net_params(net), x)
            ratio = np.abs(q - want) / B
            _record(value_form(din), ratio.max())
            assert (ratio <= 1).all(), (rows, n, float(ratio.max()), np.argwhere(ratio > 1)[:4])
            has = hot >= 0
            offsets |= set(hot[has] % 8)
            if has.sum() >= 8:
                cold = x.copy()
                cold[np.nonzero(has)[0], hot[has], din - 2] = 0.0
                moved = np.abs(forward64(net_params(net), cold)[0] - want) > 8 * B
                assert moved[has].mean() > 0.8, (rows, n, float(moved[has].mean()))
        assert offsets == set(range(8))
    _expect([value_form(din)], run)
