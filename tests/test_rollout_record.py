"""The per-tick recording ring of device rollouts (astro_rollout_device_record, BatchedGames.record_ring): every tick's controls,
events and pre-step observation, byte for byte what a Python loop of step() calls sees, in every bot mode and on every path
of astro_rollout_device; recording changes no result; the Experience tensors built from the ring equal ones built by hand
from that loop."""
import ctypes as C

import numpy as np
import pytest

from astro_b200 import core, rng
from astro_b200 import _native as nat
from tests import helpers as H

pytestmark = pytest.mark.gpu

CALLS = (37, 43, 37, 43)          # 160 ticks: graph chunks of 16 and tail ticks in every call, a ring of 48 rows wraps
BOTS = [('script', 'script'), ('nothing', 'script'), ('policy', 'script'), ('policy', 'policy'), ('explore', 'script'),
        ('explore', 'explore'), ('stream', 'stream')]


def _net(solo=False):
    import torch
    from astro_b200 import rl
    torch.manual_seed(11)
    net = rl.ValueNetwork(solo=solo, nout=6).cuda()
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(3.0)
    return net


def _batch(cfg, N, net, fresh=False, K=32):
    from astro_b200.batched import BatchedGames
    g = BatchedGames(cfg, N, bullet_cap=K, precision=32, seed=13)
    if fresh:
        g.enable_fresh_games(quota=48)
    else:
        pool = H.make_pool(cfg, 256)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    g.reset_all()
    g.set_policy(net)
    g.set_exploration(1.0, 0.1, seed=5)
    return g


def _loop_tick(g, bots):
    """One tick of the loop of test_rollout_device_equals_tick_by_tick_loop; returns (controls [n_pad, S], events [n_pad])."""
    import torch
    if bots[0] == 'stream':
        ctl = torch.from_numpy(rng.actions(g.seed, np.arange(g.n_pad) + g.first_game, g.step_index, g.S).astype(np.uint8)).cuda()
        return ctl, g.step(None, auto_reset=True)[2].clone()
    a = g.script_controls() if 'script' in bots else torch.full((g.n_pad, g.S), 2, dtype=torch.uint8, device='cuda')
    for s, b in enumerate(bots):
        if b == 'nothing':
            a[:, s] = 2
    ships = [s for s, b in enumerate(bots) if b in ('policy', 'explore')]
    if ships:
        g.policy_controls(out=a, ships=ships)
    ships = [s for s, b in enumerate(bots) if b == 'explore']
    if ships:
        g.explore_controls(a, g._explore_state, 1.0, 0.1, seed=5, ships=ships)
    ctl = a.clone()
    ev = g.step(a, auto_reset=True)[2].clone()
    return ctl, ev


def _check_against_loop(cfg, bots, observations, N=2048, calls=CALLS, ring_rows=48):
    """Recorded rollout == Python loop, row by row, after every call; final state and statistics == an unrecorded rollout."""
    import torch
    net = _net(cfg.solo)
    bots = bots[:1] if cfg.solo else bots
    rec, loop, plain = (_batch(cfg, N, net) for _ in range(3))
    ring = rec.record_ring(ring_rows, observations=observations)
    for n in calls:
        s0 = rec.step_index
        want = []
        for k in range(n):
            obs = loop.observe(n_rows=ring.n_rows, shared=True).clone() if observations else None
            ctl, ev = _loop_tick(loop, bots)
            want.append((obs, ctl, ev))
        rec.rollout_device(n, bots=bots, record=ring)
        plain.rollout_device(n, bots=bots)
        for k, (obs, ctl, ev) in enumerate(want):
            row = (s0 + k) % ring_rows
            assert torch.equal(ring.controls[row], ctl), (bots, s0 + k)
            assert torch.equal(ring.events[row, :N], ev), (bots, s0 + k)
            if observations:
                assert torch.equal(ring.observations[row, :N], obs), (bots, s0 + k)
        if observations:
            after = loop.observe(n_rows=ring.n_rows, shared=True)
            assert torch.equal(ring.observations[(s0 + n) % ring_rows, :N], after), bots
    xa, xb, xc = rec.get_arrays(), plain.get_arrays(), loop.get_arrays()
    sa, sb, sc = rec.stats(), plain.stats(), loop.stats()
    assert sa == sb == sc and sa['env_steps'] == N * sum(calls)
    for k in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (xa[k] == xb[k]).all() and (xa[k] == xc[k]).all(), k
    return sa


@pytest.mark.parametrize('observations', [False, True])
@pytest.mark.parametrize('bots', BOTS)
@pytest.mark.parametrize('env', [None, 'ASTRO_FUSED_BOTS', 'ASTRO_LOOP_GRAPH'])
def test_recorded_rollout_equals_python_loop(bots, observations, env, monkeypatch):
    """Every ring row is what a Python loop of step() calls passed and got, with or without the in-tick bots and the captured
    graph chunks (each switched off in the environment: the same rings)."""
    if env:
        monkeypatch.setenv(env, '0')
    st = _check_against_loop(core.DEFAULT_CONFIG, bots, observations)
    assert st['episodes'] > 0


@pytest.mark.parametrize('bots', [('script', 'script'), ('policy', 'script')])
def test_recorded_rollout_in_an_eight_slot_batch(bots):
    """8 planet slots (max_planets 6): the 8-slot tick kernel records through the same tick body."""
    cfg = core.DEFAULT_CONFIG._replace(max_planets=6)
    for observations in (False, True):
        _check_against_loop(cfg, bots, observations, N=1024, calls=(37, 43))


@pytest.mark.parametrize('bot', ['script', 'nothing', 'policy'])
def test_recorded_rollout_of_solo_games(bot):
    cfg = core.DEFAULT_CONFIG._replace(solo=True)
    for observations in (False, True):
        _check_against_loop(cfg, (bot, bot), observations, N=1024, calls=(37, 43))


@pytest.mark.parametrize('bots,observations', [(('stream', 'stream'), False), (('script', 'script'), False),
                                               (('explore', 'explore'), True)])
def test_recorded_rollout_in_fresh_game_mode(bots, observations):
    """Fresh-game mode re-creates games from refills whose timing depends on the launch pattern, so the reference here is an
    unrecorded rollout of the same calls: identical final state and statistics, its last tick's events equal the ring's, the
    counter-stream controls are rng.actions, and each call's first and final observations are observe() of those states."""
    import torch
    cfg, N = core.DEFAULT_CONFIG, 2048
    net = _net()
    rec, plain = _batch(cfg, N, net, fresh=True), _batch(cfg, N, net, fresh=True)
    ring = rec.record_ring(48, observations=observations)
    ends = 0
    for n in CALLS:
        s0 = rec.step_index
        before = rec.observe(n_rows=ring.n_rows, shared=True).clone() if observations else None
        rec.rollout_device(n, bots=bots, record=ring)
        plain.rollout_device(n, bots=bots)
        assert torch.equal(ring.events[(s0 + n - 1) % 48], plain._events)
        ev = ring.window_events(n)
        ends += int(((ev & nat.EV_DONE_MASK) != 0).sum())
        if bots[0] == 'stream':
            for k in range(n):
                want = rng.actions(rec.seed, np.arange(rec.n_pad), s0 + k, 2).astype(np.uint8)
                assert (ring.controls[(s0 + k) % 48].cpu().numpy() == want).all()
        if observations:
            assert torch.equal(ring.observations[s0 % 48, :N], before)
            assert torch.equal(ring.observations[(s0 + n) % 48, :N], rec.observe(n_rows=ring.n_rows, shared=True))
    sa, sb = rec.stats(), plain.stats()
    assert sa == sb and sa['wins0'] + sa['wins1'] + sa['both_lost'] + sa['timeouts'] == ends > 0
    xa, xb = rec.get_arrays(), plain.get_arrays()
    for k in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (xa[k] == xb[k]).all(), k


def test_experiences_from_the_ring_equal_ones_built_from_the_loop():
    """Five windows of 100 explore-explore ticks, n_steps 100, a ring of 201 rows: the Experience tensors the ring builds from
    nstep_experiences equal the ones built by hand from a Python loop's log (features from observe(shared=False)[g, s], the
    row convention of test_nstep_experiences_match_the_reference_ingestion), and every terminal pair is flagged."""
    import torch
    cfg, N, W, T, n_steps = core.DEFAULT_CONFIG, 256, 5, 100, 100
    net = _net()
    rec, loop = _batch(cfg, N, net), _batch(cfg, N, net)
    ring = rec.record_ring(n_steps + T + 1)
    bots = ('explore', 'explore')
    feats, ctls, evs = [], [], []
    carry_r = carry_l = None
    n_terminal = 0
    for w in range(W):
        for k in range(T):
            feats.append(loop.observe(n_rows=ring.n_rows).clone())
            ctl, ev = _loop_tick(loop, bots)
            ctls.append(ctl)
            evs.append(ev)
        feats.append(loop.observe(n_rows=ring.n_rows).clone())        # (replaced by the next window's first tick: the same)
        rec.rollout_device(T, bots=bots, record=ring)
        ev_l = torch.stack(evs[w * T:(w + 1) * T]).contiguous()
        ev_r = ring.window_events(T)
        assert torch.equal(ev_r, ev_l)
        rew, dis, nxt, carry_r = rec.nstep_experiences(ev_r, carry_r, n_steps=n_steps, discount=0.995)
        got = ring.experiences(rew, dis, nxt, n_steps)
        rew_l, dis_l, nxt_l, carry_l = loop.nstep_experiences(ev_l, carry_l, n_steps=n_steps, discount=0.995)
        # by hand, from the loop's log
        t0 = w * T
        row, game, ship = (nxt_l >= -1).nonzero(as_tuple=True)
        tick = t0 + row - n_steps
        assert int(tick.min()) >= 0
        nx = nxt_l[row, game, ship]
        terminal = nx == -1
        log = torch.stack(feats[:t0 + T + 1])                      # [ticks + 1, n, S, rows, D]: the last entry is the state after
        feats = feats[:t0 + T]
        want_f = log[tick, game, ship]
        want_n = log[t0 + nx.clamp(min=0), game, ship]
        want_n[terminal] = -1.0
        want = dict(features=want_f, action=torch.stack(ctls)[tick, game, ship], reward=rew_l[row, game, ship],
                    discount=dis_l[row, game, ship], next_features=want_n, terminal=terminal, game=game, ship=ship, tick=tick)
        for key, v in want.items():
            assert torch.equal(got[key], v), (w, key)
        # each terminal pair is flagged: its game ended within n_steps ticks of the pair's tick, and every pair whose new
        # state is None is one
        done = (torch.stack(evs) & nat.EV_DONE_MASK) != 0                                   # [ticks, n]
        span = torch.arange(n_steps, device='cuda')
        t_idx = (tick[terminal, None] + span[None, :]).clamp(max=done.shape[0] - 1)
        assert done[t_idx, game[terminal, None]].any(dim=1).all()
        n_terminal += int(terminal.sum())
    assert n_terminal > 0


def test_recording_fast_paths_keep_their_launches():
    """Recording without observations costs no launch: scripted games keep the in-tick bot form with many ticks per launch
    (no script kernel), the counter stream keeps the fused form."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from tests.test_tick_forms import form_of
    cfg, N, n = core.DEFAULT_CONFIG, 2048, 100
    net = _net()
    # (the last tick of a counter-stream call is a launch of its own, the one-tick form: it writes the call's `events`)
    for bots, forms in ((('script', 'script'), {('tick_f32_kernel', 2, 1, 1, 1, 0)}),
                        (('stream', 'stream'), {('tick_f32_kernel', 2, 1, 1, 0, 0), ('tick_f32_kernel', 2, 1, 0, 0, 0)})):
        g = _batch(cfg, N, net)
        ring = g.record_ring(128, observations=False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            g.rollout_device(n, bots=bots, record=ring)
            torch.cuda.synchronize()
        counts = {}
        for e in prof.key_averages():
            counts[e.key] = counts.get(e.key, 0) + e.count
        assert counts, 'the profiler returned no kernel records'
        ticks = {form_of(k): c for k, c in counts.items() if form_of(k) is not None}
        assert set(ticks) == forms and sum(ticks.values()) == 2, (bots, ticks)   # n - 1 ticks in one launch, then the last
        assert not any('script_kernel' in k or 'observe_kernel' in k for k in counts), counts
        assert int((ring.events[:n] & nat.EV_SKIPPED).sum()) == 0 and int(ring.controls[:n].max()) <= 5


def test_record_errors():
    """Misuse of astro_rollout_device_record returns ASTRO_E_INVALID with a message naming the problem."""
    import torch
    L = nat.lib()
    cfg, N = core.DEFAULT_CONFIG, 64
    g = _batch(cfg, N, _net())
    h, st = g._h, g._stream()
    ring = g.record_ring(8)

    def call(games, n, r, flags=nat.TICK_AUTO_RESET):
        return L.astro_rollout_device_record(games._h, n, 1, 1, 0.1, 0.45, games._actions.data_ptr(), C.byref(r), flags, st)

    def struct(**kw):
        f = dict(ticks=8, n_rows=ring.n_rows, controls=ring.controls.data_ptr(), events=ring.events.data_ptr(),
                 observations=ring.observations.data_ptr())
        f.update(kw)
        return nat.AstroRecordRing(f['ticks'], f['n_rows'], f['controls'], f['events'], f['observations'])

    assert call(g, 8, struct()) == -1 and b'ring of at least' in L.astro_last_error()
    assert call(g, 7, struct(controls=None)) == -1 and b'controls and events' in L.astro_last_error()
    assert call(g, 7, struct(events=None)) == -1 and b'controls and events' in L.astro_last_error()
    assert call(g, 7, struct(n_rows=4)) == -1 and b'n_rows' in L.astro_last_error()
    assert call(g, 7, struct(observations=ring.observations.data_ptr() + 4)) == -1 and b'16-byte aligned' in L.astro_last_error()
    assert call(g, 7, struct(), nat.TICK_AUTO_RESET | nat.TICK_GENERIC_KERNEL) == -1 and b'ASTRO_TICK_GENERIC_KERNEL' in L.astro_last_error()
    from astro_b200.batched import BatchedGames
    g64 = BatchedGames(cfg, N, bullet_cap=32, precision=64)
    assert call(g64, 7, struct()) == -1 and b'float32' in L.astro_last_error()
    with pytest.raises(nat.AstroError, match='ring of at least'):
        g.rollout_device(8, bots='script', record=ring)          # (the library's error, through the Python layer)
    assert call(g, 7, struct()) == 0                           # a working call after the failures
    torch.cuda.synchronize()
