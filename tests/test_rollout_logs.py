"""Game logs of device rollouts (logs.GameRecorder.rollout, RecordRing.follow_states, astro_rollout_device_follow).

A RecordRing that follows a few games receives their states from follow_kernel<S, PL> (4 forms) before every tick of
rollout_device, next to every tick's controls and event byte.  GameRecorder.rollout turns those rows into core.Games.
The reference is GameRecorder.step on a Python loop of step() calls driving a twin batch: the same finished Games bit
for bit and byte-identical .jsonl files, in every bot pairing, with and without the captured graph chunks and the in-tick
bots, in 8-slot and solo batches; fresh-game mode against get_states at the call boundaries; the logged ticks against
the oracle; following changes no result, and misuse of the entry point launches nothing."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from astro_b200 import _native as nat
from astro_b200 import core, logs
from oracle import astro_oracle as ao
from tests import helpers as H
from tests.test_rollout_record import CALLS, _batch, _loop_tick, _net

TOL = 1e-5                        # the float32 tick's policy (DESIGN §3, test_tick_forms)
BOTS = [('stream', 'stream'), ('script', 'script'), ('script', 'nothing'), ('policy', 'script'), ('explore', 'explore')]

# ------------------------------------------------------------------ kernel names and the ledger

_FORM = re.compile(r'\bfollow_kernel<([^<>]*)>')


def form_of(name):
    """follow_kernel<2, 4> (CUPTI) or follow_kernel<(int)2, (int)4> (cu++filt) -> ('follow_kernel', 2, 4); None for any
    other kernel."""
    m = _FORM.search(name)
    if m is None:
        return None
    return ('follow_kernel',) + tuple(int(re.sub(r'^\(int\)', '', a.strip())) for a in m.group(1).split(','))


LEDGER = {('follow_kernel', S, PL): ('test_each_follow_form_is_launched',) for S in (1, 2) for PL in (4, 8)}


def test_follow_kernel_names_parse_in_both_spellings():
    assert form_of('void (anonymous namespace)::follow_kernel<2, 4>(const void *, int)') == ('follow_kernel', 2, 4)
    assert form_of('void <unnamed>::follow_kernel<(int)1, (int)8>(const void *, int)') == ('follow_kernel', 1, 8)
    assert form_of('void <unnamed>::export_kernel<float, (int)2, (int)4>(const void *)') is None
    assert form_of('void (anonymous namespace)::tick_f32_kernel<2, true, false, false, true>(TickParams)') is None


def test_library_follow_forms_equal_the_ledger():
    """The built library holds exactly the 4 follow_kernel forms, and each is launched by a test of this file."""
    forms = [f for f in map(form_of, H.library_kernel_names()) if f is not None]
    assert len(forms) == len(set(forms)) == 4
    assert set(forms) == set(LEDGER)
    for form, tests in LEDGER.items():
        for t in tests:
            assert callable(globals().get(t)) and t.startswith('test_'), (form, t)


@pytest.mark.gpu
@pytest.mark.parametrize('S,PL', [(S, PL) for S in (1, 2) for PL in (4, 8)])
@pytest.mark.parametrize('bot', ['script', 'policy'])
def test_each_follow_form_is_launched(S, PL, bot):
    """A followed rollout of each batch layout launches exactly its follow_kernel form, seen by torch.profiler.  The profiler
    runs in a process of its own (tests/follow_worker.py), so that no CUPTI session of this file precedes the exact launch
    counts other test files take in this process."""
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'follow_worker.py')
    r = subprocess.run([sys.executable, worker, str(int(S == 1)), '4' if PL == 4 else '6', bot], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-3000:])
    names = json.loads(r.stdout.strip().splitlines()[-1])
    assert names, 'the profiler returned no kernel records'
    assert {f for f in map(form_of, names) if f is not None} == {('follow_kernel', S, PL)}, names


# ------------------------------------------------------------------ the reference: GameRecorder.step on a step() loop

class _Logged:
    """A batch whose step() goes through a GameRecorder; every tick, event_rewards of the events step() returns must equal
    its reward tensor (every game that was stepped)."""

    def __init__(self, games, recorder):
        self._g, self._rec = games, recorder

    def __getattr__(self, k):
        return getattr(self._g, k)

    def step(self, actions, **kw):
        out = self._rec.step(actions, **kw)
        ev = out[2].cpu().numpy()
        stepped = (ev & nat.EV_SKIPPED) == 0
        want = out[0].cpu().numpy()
        got = logs.event_rewards(ev, self._g.S, self._g.config.solo)
        assert got.dtype == want.dtype and np.array_equal(got[stepped], want[stepped])
        return out


def _scout(cfg, N, net, bots, calls, extra=(0, 31, 33, 1000)):
    """Games to follow: up to 24 that end within the calls (found on an unfollowed twin; the rollouts are deterministic)
    and a few fixed slots."""
    g = _batch(cfg, N, net)
    ring = g.record_ring(max(calls) + 1, observations=False)
    ended = np.zeros(g.n_pad, dtype=bool)
    for n in calls:
        g.rollout_device(n, bots=bots, record=ring)
        ended |= ((ring.window_events(n) & nat.EV_DONE_MASK) != 0).any(0).cpu().numpy()
    hits = np.nonzero(ended[:N])[0]
    pick = hits[np.linspace(0, hits.size - 1, min(24, hits.size)).astype(int)] if hits.size else hits
    return sorted(set(int(i) for i in pick) | set(i for i in extra if i < N))


def _same_state(a, b):
    assert (a is None) == (b is None)
    if a is None:
        return
    for x, y in ((a.ships.x, b.ships.x), (a.ships.dx, b.ships.dx), (a.ships.b, b.ships.b), (a.planets.x, b.planets.x),
                 (a.planets.dx, b.planets.dx), (a.bullets.x, b.bullets.x), (a.bullets.dx, b.bullets.dx)):
        assert x.dtype == y.dtype == np.float64 and H.same_bits(x, y)
    assert a.planets.b is b.planets.b is None and a.bullets.b is b.bullets.b is None
    assert (a.reload, a.t) == (b.reload, b.t)


def _same_ticks(ta, tb):
    assert len(ta) == len(tb)
    for t, u in zip(ta, tb):
        _same_state(t.state, u.state)
        assert t.control.dtype == u.control.dtype and np.array_equal(t.control, u.control)
        assert t.reward.dtype == u.reward.dtype == np.float32 and np.array_equal(t.reward.view(np.uint32), u.reward.view(np.uint32))
        assert t.bot_data == u.bot_data


def _same_logs(dev, loop):
    assert len(dev.finished) == len(loop.finished)
    for a, b in zip(dev.finished, loop.finished):
        assert a.config == b.config and a.winner == b.winner
        _same_ticks(a.ticks, b.ticks)
    for i in dev.indices:                                      # the games still in progress
        _same_ticks(dev._ticks[i], loop._ticks[i])
    assert [os.path.basename(p) for p in dev.paths] == [os.path.basename(p) for p in loop.paths]
    for p, q in zip(dev.paths, loop.paths):
        with open(p, 'rb') as f, open(q, 'rb') as h:
            assert f.read() == h.read(), p


def _check_logs(tmp_path, cfg, bots, N=2048, calls=CALLS, ring_rows=48):
    """GameRecorder.rollout on rollout_device calls == GameRecorder.step on a step() loop; returns the number of finished
    games."""
    net = _net(cfg.solo)
    bots = bots[:1] if cfg.solo else bots
    follow = _scout(cfg, N, net, bots, calls)
    dev, loop = _batch(cfg, N, net), _batch(cfg, N, net)
    ring = dev.record_ring(ring_rows, observations=False, follow=follow)
    rd = logs.GameRecorder(dev, follow, folder=str(tmp_path / 'device'), bot_data=['a', 'b'][:dev.S])
    rl = logs.GameRecorder(loop, follow, folder=str(tmp_path / 'loop'), bot_data=['a', 'b'][:dev.S])
    proxy = _Logged(loop, rl)
    for n in calls:
        for _ in range(n):
            _loop_tick(proxy, bots)
        rd.rollout(n, ring, bots=bots)
    _same_logs(rd, rl)
    assert dev.stats() == loop.stats()
    for p in rd.paths:
        g = core.load_log(p)
        assert len(g.ticks) > 0 and g.winner in (None, 0, 1)
    return len(rd.finished)


@pytest.mark.gpu
@pytest.mark.parametrize('env', [None, 'ASTRO_LOOP_GRAPH', 'ASTRO_FUSED_BOTS'])
@pytest.mark.parametrize('bots', BOTS)
def test_followed_rollout_equals_the_step_loop(bots, env, tmp_path, monkeypatch):
    """The logs of rollout_device calls of 37, 43, 37, 43 ticks (graph chunks, tail ticks, a ring of 48 rows that wraps)
    equal a step() loop's, bit for bit and byte for byte, with the graph chunks or the in-tick bots switched off."""
    if env:
        monkeypatch.setenv(env, '0')
    assert _check_logs(tmp_path, core.DEFAULT_CONFIG, bots) > 0


@pytest.mark.gpu
@pytest.mark.parametrize('bots', [('script', 'script'), ('policy', 'script')])
def test_followed_rollout_in_an_eight_slot_batch(bots, tmp_path):
    assert _check_logs(tmp_path, core.DEFAULT_CONFIG._replace(max_planets=6), bots, N=1024, calls=(37, 43)) > 0


@pytest.mark.gpu
@pytest.mark.parametrize('max_planets', [4, 6])
@pytest.mark.parametrize('bot', ['script', 'policy'])
def test_followed_rollout_of_solo_games(bot, max_planets, tmp_path):
    cfg = core.DEFAULT_CONFIG._replace(solo=True, max_planets=max_planets)
    _check_logs(tmp_path, cfg, (bot, bot), N=1024, calls=(37, 43))


@pytest.mark.gpu
@pytest.mark.parametrize('bots', [('stream', 'stream'), ('script', 'script'), ('explore', 'explore')])
def test_followed_rollout_in_fresh_game_mode(bots, monkeypatch):
    """Fresh-game refills happen between launches, so the reference is a twin with the same launch pattern: unfollowed,
    with the in-tick bots off for scripted games and recording observations for the counter stream (both take the
    per-tick loop, as following does).  The followed states at every call boundary are get_states of the twin, and the
    final arrays and statistics are the twin's."""
    cfg, N = core.DEFAULT_CONFIG, 2048
    net = _net()
    if bots[0] == 'script':
        monkeypatch.setenv('ASTRO_FUSED_BOTS', '0')
    follow = [0, 5, 31, 32, 77, 640, 1500, 2047]
    dev, twin = _batch(cfg, N, net, fresh=True), _batch(cfg, N, net, fresh=True)
    ring = dev.record_ring(48, observations=False, follow=follow)
    twin_ring = twin.record_ring(48, observations=True) if bots[0] == 'stream' else None
    rec = logs.GameRecorder(dev, follow)
    for n in CALLS:
        s0 = dev.step_index
        before = twin.get_states(follow)
        rec.rollout(n, ring, bots=bots)
        twin.rollout_device(n, bots=bots, record=twin_ring)
        for a, b in zip(ring.follow_states(s0), before):
            _same_state(a, b)
        for a, b in zip(ring.follow_states(s0 + n), twin.get_states(follow)):
            _same_state(a, b)
    assert dev.stats() == twin.stats()
    xa, xb = dev.get_arrays(), twin.get_arrays()
    for k in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (xa[k] == xb[k]).all(), k


# ------------------------------------------------------------------ against the oracle

def _oracle_batch(states, S, K):
    ob = ao.Batch(len(states), S, K)
    for j, s in enumerate(states):
        ob.ships[j, :, 0:2], ob.ships[j, :, 2:4], ob.ships[j, :, 4] = s.ships.x, s.ships.dx, s.ships.b
        p, nb = s.planets.x.shape[0], s.bullets.x.shape[0]
        ob.planets[j, :p, 0:2], ob.planets[j, :p, 2:4] = s.planets.x, s.planets.dx
        ob.np_[j] = p
        ob.bullets[j, :nb, 0:2], ob.bullets[j, :nb, 2:4] = s.bullets.x, s.bullets.dx
        ob.nb[j] = nb
        ob.reload[j], ob.t[j] = s.reload, s.t
    return ob


def _close(got, ref):
    err = np.abs(np.asarray(got) - np.asarray(ref)) / np.maximum(1.0, np.abs(ref))
    return err.size == 0 or float(err.max()) <= TOL


@pytest.mark.gpu
def test_logs_of_a_scripted_rollout_replay_through_the_oracle(tmp_path):
    """Every logged Tick of a scripted rollout, replayed through oracle.step_batch from its state and control: the reward
    is the logged one, the game ends exactly on its last Tick, and the next Tick's state is the oracle's (discrete
    outcomes exact, continuous state within 1e-5 * max(1, |ref|)); the ring's event bytes of the last call are the
    oracle's.  Every file round-trips through core.load_log."""
    cfg, N, K, calls = core.DEFAULT_CONFIG, 2048, 32, (37, 43)
    net = _net()
    follow = _scout(cfg, N, net, ('script', 'script'), calls)
    g = _batch(cfg, N, net, K=K)
    ring = g.record_ring(48, observations=False, follow=follow)
    rec = logs.GameRecorder(g, follow, folder=str(tmp_path))
    for n in calls:
        s0 = g.step_index
        rec.rollout(n, ring, bots='script')
    games = list(rec.finished) + [core.Game(cfg, None, rec._ticks[i]) for i in follow if rec._ticks[i]]
    assert rec.finished
    ticks = [t for gm in games for t in gm.ticks]
    o2, rew, done, ev = ao.step_batch(cfg, _oracle_batch([t.state for t in ticks], 2, K), np.stack([t.control for t in ticks]))
    k = 0
    for gi, gm in enumerate(games):
        for j, t in enumerate(gm.ticks):
            assert np.array_equal(rew[k].astype(np.float32), t.reward), (gi, j)
            last = j == len(gm.ticks) - 1
            assert bool(done[k]) == (last and gi < len(rec.finished)), (gi, j)
            if not last:
                nxt = gm.ticks[j + 1].state
                assert nxt.bullets.x.shape[0] == o2.nb[k] and nxt.planets.x.shape[0] == o2.np_[k], (gi, j)
                assert _close(nxt.t, o2.t[k]) and _close(nxt.reload, o2.reload[k]), (gi, j)
                assert _close(np.concatenate([nxt.ships.x, nxt.ships.dx, nxt.ships.b[:, None]], 1), o2.ships[k]), (gi, j)
                p, nb = o2.np_[k], o2.nb[k]
                assert _close(np.concatenate([nxt.planets.x, nxt.planets.dx], 1), o2.planets[k, :p]), (gi, j)
                assert _close(np.concatenate([nxt.bullets.x, nxt.bullets.dx], 1), o2.bullets[k, :nb]), (gi, j)
            k += 1
    # the event bytes of the last call's ticks, from the ring
    n = calls[-1]
    for s in range(s0, s0 + n):
        states = ring.follow_states(s)
        live = [j for j, st in enumerate(states) if st is not None]
        row = s % ring.ticks
        ctl = ring.controls[row].cpu().numpy()[[follow[j] for j in live]]
        _, _, _, ev_o = ao.step_batch(cfg, _oracle_batch([states[j] for j in live], 2, K), ctl)
        ev_r = ring.events[row].cpu().numpy()[[follow[j] for j in live]]
        assert np.array_equal(ev_r.astype(np.int64), ev_o.astype(np.int64)), s
    for p, gm in zip(rec.paths, rec.finished):
        back = core.load_log(p)
        assert back.winner == gm.winner and len(back.ticks) == len(gm.ticks)
        for t, u in zip(back.ticks, gm.ticks):
            assert np.array_equal(t.state.ships.x, u.state.ships.x) and np.array_equal(t.control, u.control)
            assert np.array_equal(t.reward, u.reward)


# ------------------------------------------------------------------ no side effects, misuse

@pytest.mark.gpu
@pytest.mark.parametrize('bots', [('script', 'script'), ('stream', 'stream'), ('policy', 'script')])
def test_following_changes_no_result(bots):
    """Final arrays, statistics and every controls / events row of a followed rollout equal those of the same rollout
    recorded without following."""
    import torch
    cfg, N = core.DEFAULT_CONFIG, 2048
    net = _net()
    a, b = _batch(cfg, N, net), _batch(cfg, N, net)
    ra = a.record_ring(48, observations=False, follow=[3, 64, 2000])
    rb = b.record_ring(48, observations=False)
    for n in CALLS:
        s0 = a.step_index
        a.rollout_device(n, bots=bots, record=ra)
        b.rollout_device(n, bots=bots, record=rb)
        rows = ra._rows(s0, n)
        assert torch.equal(ra.controls[rows], rb.controls[rows]) and torch.equal(ra.events[rows], rb.events[rows])
    assert a.stats() == b.stats()
    xa, xb = a.get_arrays(), b.get_arrays()
    for k in xa:
        assert (xa[k] == xb[k]).all(), k


def _call(L, g, n, ring, follow, flags=nat.TICK_AUTO_RESET):
    return L.astro_rollout_device_follow(g._h, n, 1, 1, 0.1, 0.45, g._actions.data_ptr(), ring, follow, flags, g._stream())


@pytest.mark.gpu
def test_out_of_range_index_is_a_finished_row():
    """A hand-built follow ring whose index holds games outside 0..n_games-1: those rows say finished, tick -1, all zero;
    the valid slot holds get_states' state."""
    import torch
    L = nat.lib()
    cfg, N = core.DEFAULT_CONFIG, 64
    g = _batch(cfg, N, _net())
    ring = g.record_ring(8, observations=False)
    idx = torch.tensor([-1, 5, g.n_pad, 1 << 30], dtype=torch.int32, device='cuda')
    m, R = 4, 8
    sh = torch.full((R, m, 2, 5), 7.0, device='cuda')
    pl = torch.full((R, m, g.PL, 4), 7.0, device='cuda')
    bl = torch.full((R, m, g.K, 4), 7.0, device='cuda')
    info = torch.full((R, m, 4), 7, dtype=torch.int32, device='cuda')
    f = nat.AstroFollowRing(m, 0, idx.data_ptr(), sh.data_ptr(), pl.data_ptr(), bl.data_ptr(), info.data_ptr())
    want = g.get_arrays([5])
    before = g.launches
    assert _call(L, g, 0, C.byref(ring._ring), C.byref(f)) == 0, L.astro_last_error()
    assert g.launches == before + 1                              # the follow kernel after the call's (no) ticks
    row = g.step_index % R
    inf = info[row].cpu().numpy()
    for j in (0, 2, 3):
        assert list(inf[j]) == [0, 0, -1, 1]
        assert float(sh[row, j].abs().sum() + pl[row, j].abs().sum() + bl[row, j].abs().sum()) == 0.0
    assert list(inf[1]) == [want['n_planets'][0], want['n_bullets'][0], want['tick'][0], 0]
    assert np.array_equal(sh[row, 1].cpu().numpy().astype(np.float64), want['ships'][0])
    assert np.array_equal(pl[row, 1].cpu().numpy().astype(np.float64), want['planets'][0])
    assert np.array_equal(bl[row, 1].cpu().numpy().astype(np.float64), want['bullets'][0])
    others = [r for r in range(R) if r != row]
    assert bool((info[others] == 7).all())                       # no other row was written


@pytest.mark.gpu
def test_follow_errors_launch_nothing():
    """Misuse of astro_rollout_device_follow returns ASTRO_E_INVALID with a message naming the problem and launches
    nothing (the library's launch counter); a good call afterwards works."""
    import torch
    L = nat.lib()
    cfg, N = core.DEFAULT_CONFIG, 64
    g = _batch(cfg, N, _net())
    ring = g.record_ring(8, observations=False, follow=[1, 2])
    rr = C.byref(ring._ring)

    def fstruct(**kw):
        f = dict(m=2, index=ring._follow_index.data_ptr(), ships=ring.follow_ships.data_ptr(),
                 planets=ring.follow_planets.data_ptr(), bullets=ring.follow_bullets.data_ptr(), info=ring.follow_info.data_ptr())
        f.update(kw)
        return C.byref(nat.AstroFollowRing(f['m'], 0, f['index'], f['ships'], f['planets'], f['bullets'], f['info']))

    from astro_b200.batched import BatchedGames
    g64 = BatchedGames(cfg, N, bullet_cap=32, precision=64)
    cases = [(g, 7, rr, None, nat.TICK_AUTO_RESET, b'follow ring is required'),
             (g, 7, None, fstruct(), nat.TICK_AUTO_RESET, b'recording ring'),
             (g, 7, rr, fstruct(m=0), nat.TICK_AUTO_RESET, b'at least one game'),
             (g, 7, rr, fstruct(index=None), nat.TICK_AUTO_RESET, b'arrays are required'),
             (g, 7, rr, fstruct(ships=None), nat.TICK_AUTO_RESET, b'arrays are required'),
             (g, 7, rr, fstruct(planets=None), nat.TICK_AUTO_RESET, b'arrays are required'),
             (g, 7, rr, fstruct(bullets=None), nat.TICK_AUTO_RESET, b'arrays are required'),
             (g, 7, rr, fstruct(info=None), nat.TICK_AUTO_RESET, b'arrays are required'),
             (g, 7, rr, fstruct(ships=ring.follow_ships.data_ptr() + 2), nat.TICK_AUTO_RESET, b'4-byte aligned'),
             (g, 7, rr, fstruct(info=ring.follow_info.data_ptr() + 1), nat.TICK_AUTO_RESET, b'4-byte aligned'),
             (g, 8, rr, fstruct(), nat.TICK_AUTO_RESET, b'ring of at least'),
             (g, 7, rr, fstruct(), nat.TICK_AUTO_RESET | nat.TICK_GENERIC_KERNEL, b'ASTRO_TICK_GENERIC_KERNEL'),
             (g64, 7, rr, fstruct(), nat.TICK_AUTO_RESET, b'float32')]
    for games, n, r, f, flags, msg in cases:
        before = games.launches
        rc = _call(L, games, n, r, f, flags)
        assert rc == -1 and msg in L.astro_last_error(), (msg, rc, L.astro_last_error())
        assert games.launches == before, msg
    with pytest.raises(ValueError, match='distinct'):
        g.record_ring(8, follow=[1, 1])
    with pytest.raises(IndexError):
        g.record_ring(8, follow=[N])
    with pytest.raises(ValueError, match='follows games'):
        logs.GameRecorder(g, [2, 1]).rollout(3, ring, bots='script')
    before = g.launches
    assert _call(L, g, 7, rr, fstruct()) == 0 and g.launches > before
    torch.cuda.synchronize()
