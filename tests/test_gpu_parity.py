"""Parity of the CUDA path (through the C ABI) against the oracle and the committed golden
vectors of the reference.  Bar: every discrete outcome (done, hit flags, timeout, fire ticks,
bullet counts and order, rewards) bit-exact; continuous state bit-exact in the float64
validation build and within |d| <= 1e-5 * max(1, |ref|) per tick in the float32 build
(north-star tolerance; measured errors are ~1e-7)."""
import collections
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from astro_b200 import core, rng
from astro_b200 import _native as nat
from oracle import astro_oracle as ao
from tests import helpers as H

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _games(*a, **k):
    from astro_b200.batched import BatchedGames
    return BatchedGames(*a, **k)


def _close(got, ref):
    return np.abs(got - ref) <= TOL * np.maximum(1.0, np.abs(ref))


# ------------------------------------------------------------------ golden trajectories, f64

def test_golden_trajectories_f64_free_running():
    """All 39 reference games, replayed free-running from tick 0 in the float64 build: every
    pre-step state, reward and terminal matches the reference bit for bit."""
    z, meta = H.load_traj()
    groups = collections.defaultdict(list)
    for m in meta:
        groups[tuple(sorted((k, v) for k, v in m['config'].items() if k != 'seed'))].append(m)
    checked = 0
    for _, ms in groups.items():
        cfg = H.config_from(ms[0]['config'])
        S = ms[0]['nships']
        n = len(ms)
        games = _games(cfg, n, bullet_cap=32, precision=64)
        off = {m['game']: np.concatenate([[0], np.cumsum(z['g%d_nb' % m['game']])]) for m in ms}
        games.set_states([H.state_from_arrays(z['g%d_ships' % m['game']][0], z['g%d_planets' % m['game']][0],
                                              np.zeros((0, 4)), 0.0, 0.0) for m in ms])
        T = max(m['nticks'] for m in ms)
        for k in range(T):
            arr = games.get_arrays()
            ctl = np.full((n, S), 2, dtype=np.uint8)
            for i, m in enumerate(ms):
                g = m['game']
                if k >= m['nticks']:
                    continue
                P, B = m['nplanets'], int(z['g%d_nb' % g][k])
                assert not arr['finished'][i] and arr['n_bullets'][i] == B and arr['n_planets'][i] == P, (g, k)
                assert H.same_bits(arr['ships'][i], z['g%d_ships' % g][k]), (g, k)
                assert H.same_bits(arr['planets'][i, :P], z['g%d_planets' % g][k]), (g, k)
                assert H.same_bits(arr['bullets'][i, :B], z['g%d_bullets' % g][off[g][k]:off[g][k + 1]]), (g, k)
                assert games.schedule.reload[arr['tick'][i]] == z['g%d_reload' % g][k]
                assert games.schedule.t[arr['tick'][i]] == z['g%d_t' % g][k]
                ctl[i] = z['g%d_control' % g][k]
                checked += 1
            reward, done, events = games.step(ctl)
            reward, done = reward.cpu().numpy(), done.cpu().numpy()
            for i, m in enumerate(ms):
                g = m['game']
                if k >= m['nticks']:
                    continue
                assert H.same_bits(reward[i], z['g%d_reward' % g][k]), (g, k)
                assert bool(done[i]) == (k == m['nticks'] - 1 and not m['truncated']), (g, k)
            if k == T - 1:
                arr = games.get_arrays()
                for i, m in enumerate(ms):
                    g = m['game']
                    if m['truncated'] and m['nticks'] == T:
                        assert H.same_bits(arr['ships'][i], z['g%d_final_ships' % g])
                        B = arr['n_bullets'][i]
                        assert H.same_bits(arr['bullets'][i, :B], z['g%d_final_bullets' % g].reshape(-1, 4))
    assert checked > 6000


def test_golden_edges_f64_through_core_step():
    """70 single-step knife-edge / precedence cases through the drop-in core.step."""
    z = np.load(os.path.join(H.G, 'edges.npz'))
    meta = json.load(open(os.path.join(H.G, 'edges.json')))
    for c in meta:
        i = c['case']
        cfg = H.config_from(c['config'])
        state = H.state_from_arrays(z['c%d_ships' % i], z['c%d_planets' % i], z['c%d_bullets' % i], c['reload'], c['t'])
        nxt, reward = core.step(state, np.array(c['control']), cfg)
        assert (nxt is None) == c['done'], c['name']
        assert H.same_bits(reward, c['reward']), c['name']
        if nxt is not None:
            o = z['c%d_o_ships' % i]
            assert H.same_bits(nxt.ships.x, o[:, 0:2]) and H.same_bits(nxt.ships.dx, o[:, 2:4]), c['name']
            assert H.same_bits(nxt.ships.b, o[:, 4]), c['name']
            o = z['c%d_o_planets' % i]
            assert H.same_bits(nxt.planets.x, o[:, 0:2]) and H.same_bits(nxt.planets.dx, o[:, 2:4]), c['name']
            o = z['c%d_o_bullets' % i].reshape(-1, 4)
            assert H.same_bits(nxt.bullets.x, o[:, 0:2]) and H.same_bits(nxt.bullets.dx, o[:, 2:4]), c['name']
            assert nxt.reload == c['o_reload'] and nxt.t == c['o_t'], c['name']


def test_golden_edges_f32_discrete():
    """The same cases in the float32 build (inputs rounded to float32, oracle fed the rounded
    inputs): done / reward / bullet count exact, state within tolerance."""
    z = np.load(os.path.join(H.G, 'edges.npz'))
    meta = json.load(open(os.path.join(H.G, 'edges.json')))
    f32 = lambda a: np.asarray(a, dtype=np.float32).astype(np.float64)
    for c in meta:
        i = c['case']
        cfg = H.config_from(c['config'])
        S = 1 if cfg.solo else 2
        sh, pl, bl = f32(z['c%d_ships' % i]), f32(z['c%d_planets' % i]), f32(z['c%d_bullets' % i]).reshape(-1, 4)
        games = _games(cfg, 1, bullet_cap=32, precision=32)
        games.set_schedule_origin(c['reload'], c['t'])
        games.set_states([H.state_from_arrays(sh, pl, bl, c['reload'], c['t'])], ticks=[0])
        ref = ao.step_one(cfg, sh, pl, bl, c['reload'], c['t'], c['control'], bullet_cap=32)
        reward, done, events = games.step(np.array(c['control']).reshape(1, S))
        assert bool(done[0].item()) == ref['done'], c['name']
        assert (reward[0].cpu().numpy().astype(np.float64) == ref['reward']).all(), c['name']
        assert int(events[0].item()) == ref['events'], c['name']
        if not ref['done']:
            arr = games.get_arrays()
            B = ref['bullets'].shape[0]
            assert arr['n_bullets'][0] == B, c['name']
            assert _close(arr['ships'][0], ref['ships']).all(), c['name']
            assert _close(arr['planets'][0, :pl.shape[0]], ref['planets']).all(), c['name']
            assert _close(arr['bullets'][0, :B], ref['bullets']).all(), c['name']


# ------------------------------------------------------------------ config #2: 4,096 games

def _teacher_forced(cfg, N, K, ticks, precision, pool_size=512, seed=0, first_game=0, start=None, tick_flags=0):
    """GPU tick vs oracle, the oracle re-fed the GPU's state every tick; auto-reset on."""
    S = 1 if cfg.solo else 2
    pool = H.make_pool(cfg, pool_size)
    games = _games(cfg, N, bullet_cap=K, precision=precision, seed=seed, first_game=first_game)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    games.tick_flags = tick_flags
    if start is not None:
        start(games)
    rpool = {k: (v.astype(games.np_rdtype).astype(np.float64) if v.dtype != np.int32 else v) for k, v in pool.items()}
    ids = first_game + np.arange(N)
    arr = games.get_arrays()
    if start is None:
        pick = rng.pool_pick(seed, ids, np.zeros(N, dtype=np.uint32), pool_size)
        assert (arr['episode'] == 0).all() and (arr['ships'] == rpool['ships'][pick]).all()
        assert (arr['n_planets'] == rpool['np'][pick]).all() and (arr['n_bullets'] == 0).all()
    worst = 0.0
    n_done = n_fired = 0
    for k in range(ticks):
        ob, alive = H.oracle_batch_from(arr, S, K)
        ob.reload[:] = games.schedule.reload[arr['tick']]
        ob.t[:] = games.schedule.t[arr['tick']]
        ctl = rng.actions(seed, ids, k, S)
        o2, rew, done, ev = ao.step_batch(cfg, ob, ctl, alive)
        r_gpu, d_gpu, e_gpu = games.step(None, auto_reset=True)
        r_gpu, d_gpu, e_gpu = r_gpu.cpu().numpy(), d_gpu.cpu().numpy(), e_gpu.cpu().numpy()
        assert (e_gpu == ev).all(), (k, np.nonzero(e_gpu != ev)[0][:8], e_gpu[e_gpu != ev][:8], ev[e_gpu != ev][:8])
        assert (d_gpu == done).all(), k
        assert (r_gpu.astype(np.float64) == rew).all(), k
        new = games.get_arrays()
        live = done == 0
        assert (new['n_bullets'][live] == o2.nb[live]).all(), k
        assert (new['tick'][live] == arr['tick'][live] + 1).all(), k
        assert (new['n_planets'][live] == arr['n_planets'][live]).all(), k
        pm = (np.arange(4)[None, :] < o2.np_[:, None])[live]
        bm = (np.arange(K)[None, :] < o2.nb[:, None])[live]
        for name, got, ref, mask in (('ships', new['ships'][live], o2.ships[live], None),
                                     ('planets', new['planets'][live], o2.planets[live], pm),
                                     ('bullets', new['bullets'][live], o2.bullets[live], bm)):
            if mask is not None:
                got, ref = got[mask], ref[mask]
            if precision == 64:
                assert (H.bits(got) == H.bits(ref)).all(), (k, name)
            else:
                err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
                if err.size:
                    worst = max(worst, float(err.max()))
                assert (err <= TOL).all(), (k, name, float(err.max()))
        # games that ended were re-created from the pool in the same launch
        dead = ~live
        if dead.any():
            pick = rng.pool_pick(seed, ids[dead], np.full(int(dead.sum()), k + 1, dtype=np.uint32), pool_size)
            assert (new['episode'][dead] == arr['episode'][dead] + 1).all(), k
            assert (new['ships'][dead] == rpool['ships'][pick]).all(), k
            assert (new['n_planets'][dead] == rpool['np'][pick]).all(), k
            assert (new['n_bullets'][dead] == 0).all() and (new['tick'][dead] == 0).all(), k
            for j, p in zip(np.nonzero(dead)[0], pick):
                P = rpool['np'][p]
                assert (new['planets'][j, :P] == rpool['planets'][p, :P]).all(), k
        n_done += int(dead.sum())
        n_fired += int(((ev & nat.EV_FIRED) != 0).sum())
        arr = new
    return games, worst, n_done, n_fired


def test_config2_4096_games_f32_teacher_forced():
    """BASELINE config #2: 4,096 duel games, random actions, default planets, 1,000 ticks:
    discrete outcomes bit-exact against the oracle on identical inputs, continuous within 1e-5."""
    games, worst, n_done, n_fired = _teacher_forced(core.DEFAULT_CONFIG, 4096, 32, 1000, 32)
    assert n_done > 20000 and n_fired > 100000
    assert worst < 2e-6, worst
    st = games.stats()
    assert st['env_steps'] == 4096 * 1000 and st['episodes'] == n_done
    assert st['episodes'] == st['wins0'] + st['wins1'] + st['both_lost'] + st['timeouts']
    assert st['overflow'] == 0 and st['bullets_spawned'] == 2 * n_fired


@pytest.mark.parametrize('flags', [nat.TICK_GENERIC_KERNEL])
def test_kernel_variants_hold_the_same_parity(flags):
    """The A/B kernels (persistent; persistent with staged rows; generic template) pass
    the same teacher-forced check as the default kernel, incl. a ragged tile count."""
    _teacher_forced(core.DEFAULT_CONFIG, 4096 + 96, 32, 150, 32, tick_flags=flags)
    _teacher_forced(core.DEFAULT_CONFIG, 2048, 400, 4, 32, start=_stress_fill(400, 5), tick_flags=flags)


def test_4096_games_f64_teacher_forced_bit_exact():
    _teacher_forced(core.DEFAULT_CONFIG, 2048, 32, 300, 64)


def test_solo_games_both_builds():
    """Solo configs: one ship, no firing (reload_time=1000), timeout counts as a win."""
    cfg = core.SOLO_CONFIG._replace(max_time=3)
    for prec in (32, 64):
        games, worst, n_done, n_fired = _teacher_forced(cfg, 1024, 32, 200, prec, pool_size=128)
        assert n_fired == 0 and n_done > 0
        assert games.stats()['timeouts'] > 0


def test_f64_free_running_rollout_matches_oracle_rollout():
    """400 ticks free-running (no teacher) with auto-reset: float64 build == oracle rollout,
    bit for bit, and the device counters equal the oracle's."""
    cfg, N, K, T, M = core.DEFAULT_CONFIG, 2048, 32, 400, 256
    pool = H.make_pool(cfg, M)
    games = _games(cfg, N, bullet_cap=K, precision=64, seed=5, first_game=1000)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    ob, _ = H.oracle_batch_from(games.get_arrays(), 2, K)
    for _ in range(T):
        games.step(None, auto_reset=True)
    stats = ao.rollout(cfg, ob, pool, 5, 1000, 0, T, threads=4)
    arr = games.get_arrays()
    assert (arr['n_bullets'] == ob.nb).all() and (arr['episode'] == ob.episode).all()
    assert (H.bits(arr['ships']) == H.bits(ob.ships)).all()
    bm = np.arange(K)[None, :] < ob.nb[:, None]
    assert (H.bits(arr['bullets'][bm]) == H.bits(ob.bullets[bm])).all()
    pm = np.arange(4)[None, :] < ob.np_[:, None]
    assert (H.bits(arr['planets'][pm]) == H.bits(ob.planets[pm])).all()
    assert (games.schedule.t[arr['tick']] == ob.t).all() and (games.schedule.reload[arr['tick']] == ob.reload).all()
    st = games.stats()
    for i, name in enumerate(nat.STAT_NAMES[:8]):
        assert st[name] == stats[i], name


def test_f32_free_running_statistics_match_the_f64_build():
    """Free-running float32 against the float64 (reference-arithmetic) build on episode statistics: the same games,
    pool, counter-stream controls and pool picks for 600 ticks.  Individual float32 trajectories leave the float64
    ones after some tens of ticks (chaotic dynamics, SURVEY hard part 8), so what must agree is the distribution:
    episode count, win split, mean episode length and bullet traffic, within the sampling error of ~170,000 episodes
    (tolerances: 4 standard errors of a binomial share / 1 % on the totals), and the first ticks — before rounding
    differences can grow — game by game."""
    cfg, N, K, T, M = core.DEFAULT_CONFIG, 32768, 32, 600, 1024
    pool = H.make_pool(cfg, M)
    out = {}
    for precision in (32, 64):
        games = _games(cfg, N, bullet_cap=K, precision=precision, seed=21, first_game=4096)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        ev_early = []
        for k in range(30):
            ev_early.append(games.step(None, auto_reset=True)[2].cpu().numpy().copy())
        if precision == 32:
            games.step_many(T - 30, None, auto_reset=True)
        else:
            for _ in range(T - 30):
                games.step(None, auto_reset=True)
        out[precision] = (games.stats(), np.stack(ev_early))
    (a, ea), (b, eb) = out[32], out[64]
    assert a['env_steps'] == b['env_steps'] == N * T
    # the first 30 ticks: the same discrete events in (all but a handful of knife-edge) games
    assert (ea != eb).any(axis=0).mean() < 1e-3
    n = b['episodes']
    assert n > 100000 and abs(a['episodes'] - n) <= 0.01 * n                     # mean episode length within 1 %
    for key in ('wins0', 'wins1', 'both_lost'):
        pa, pb = a[key] / a['episodes'], b[key] / n
        assert abs(pa - pb) <= 4.0 * np.sqrt(2.0 * pb * (1.0 - pb) / n) + 1e-4, (key, pa, pb)
    assert a['timeouts'] == b['timeouts'] == 0 or abs(a['timeouts'] - b['timeouts']) <= 0.05 * b['timeouts'] + 5
    for key in ('bullets_in', 'bullets_out', 'planets_live'):
        assert abs(a[key] - b[key]) <= 0.01 * b[key], key


# ------------------------------------------------------------------ config #3: 65,536 games, full pools

_stress_fill = H.stress_fill


@pytest.mark.parametrize('K', [400, 32])
def test_config3_65536_games_max_bullet_pool(K):
    """BASELINE config #3 at its stated size: 65,536 games with pre-filled bullet pools (K=400 is the lossless
    bound of the default config, K=32 the production cap): despawn, spawn at capacity, cull and
    compaction order checked element-wise against the oracle for several ticks."""
    N = 65536
    games, worst, n_done, n_fired = _teacher_forced(core.DEFAULT_CONFIG, N, K, 6, 32, start=_stress_fill(K, 3))
    assert n_done > 0 and n_fired > 0
    st = games.stats()
    assert st['overflow'] > 0 and st['bullets_in'] > st['bullets_out']


def test_small_cap_overflow_policy():
    """K=4: newborn bullets beyond the cap are dropped from the end and flagged."""
    games, _, _, _ = _teacher_forced(core.DEFAULT_CONFIG, 2048, 4, 120, 32)
    assert games.stats()['overflow'] > 0


# ------------------------------------------------------------------ observations

def test_observe_matches_oracle_features():
    """observe() == get_features + roll_ships + to_batch for every game and both perspectives,
    float32 bit-exact (rl.py:43-99)."""
    cfg, N, K = core.DEFAULT_CONFIG, 2048, 32
    for prec in (32, 64):
        pool = H.make_pool(cfg, 256)
        games = _games(cfg, N, bullet_cap=K, precision=prec, seed=1)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        for _ in range(90):
            games.step(None, auto_reset=True)
        games.step(None, auto_reset=False)       # leaves a few finished games behind
        arr = games.get_arrays()
        obs = games.observe().cpu().numpy()
        assert obs.shape == (N, 2, 36, 15) and obs.dtype == np.float32
        assert arr['finished'].any()
        for g in range(N):
            for me in range(2):
                if arr['finished'][g]:
                    assert (obs[g, me] == -1).all()
                    continue
                P, B = arr['n_planets'][g], arr['n_bullets'][g]
                ref = ao.features(2, arr['ships'][g], arr['planets'][g, :P], arr['bullets'][g, :B], me, 36)
                assert (obs[g, me].view(np.uint32) == ref.view(np.uint32)).all(), (prec, g, me)


def test_features_api_matches_golden():
    """astro_b200.rl.ValueNetwork.get_features / get_features_batch vs the reference's outputs."""
    from astro_b200 import rl
    z, meta = H.load_traj()
    f = np.load(os.path.join(H.G, 'features.npz'))
    fm = json.load(open(os.path.join(H.G, 'features.json')))
    for e in fm[:12]:
        g = e['game']
        nb = z['g%d_nb' % g]
        off = np.concatenate([[0], np.cumsum(nb)])
        states = [H.state_from_arrays(z['g%d_ships' % g][k], z['g%d_planets' % g][k],
                                      z['g%d_bullets' % g][off[k]:off[k + 1]], 0.0, 0.0) for k in e['ticks']]
        for k, s in zip(e['ticks'], states):
            got = rl.ValueNetwork.get_features(s)
            ref = f['g%d_t%d_f0' % (g, k)]
            assert got.shape == ref.shape and (got.view(np.uint32) == ref.view(np.uint32)).all(), (g, k)
            if e['nships'] == 2:
                got = rl.ValueNetwork.get_features(core.roll_ships(s, 1))
                assert (got.view(np.uint32) == f['g%d_t%d_f1' % (g, k)].view(np.uint32)).all(), (g, k)
        got = rl.ValueNetwork.get_features_batch(states)
        assert (got.view(np.uint32) == f['g%d_batch' % g].view(np.uint32)).all(), g
        assert (rl.ValueNetwork.to_batch([rl.ValueNetwork.get_features(s) for s in states]) == got).all()


def test_rollout_host_pipelining_equals_tick_by_tick():
    """astro_rollout_host (controls of tick k+1 / events of tick k-1 copied while tick k runs)
    returns, tick for tick, the events of the unpipelined astro_tick_host and leaves the same state."""
    import torch
    cfg, N, K, T = core.DEFAULT_CONFIG, 8192, 32, 45
    pool = H.make_pool(cfg, 256)
    r = np.random.RandomState(3)
    actions = torch.from_numpy(r.randint(0, 6, (T, N, 2)).astype(np.uint8)).pin_memory()

    def fresh():
        g = _games(cfg, N, bullet_cap=K, precision=32, seed=4)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        for _ in range(30):
            g.step(None, auto_reset=True)
        return g
    a, b = fresh(), fresh()
    ev_a = torch.empty((T, N), dtype=torch.uint8).pin_memory()
    ev_b = torch.empty((T, N), dtype=torch.uint8).pin_memory()
    a.rollout_host(actions, ev_a, auto_reset=True)
    for k in range(T):
        b.step_host(actions[k], ev_b[k], auto_reset=True)
    assert bool((ev_a == ev_b).all()) and int((ev_a & 7).ne(0).sum()) > 100
    xa, xb = a.get_arrays(), b.get_arrays()
    for key in ('ships', 'n_bullets', 'tick', 'episode'):
        assert (xa[key] == xb[key]).all(), key
    assert a.stats() == b.stats()


def test_value_network_single_vs_batch_and_padding_neutral():
    """astro/test/test_rl.py:13-45 against the drop-in: single and batched evaluation agree, the
    -1 padding is output-neutral, and BatchedGames.observe() feeds the same network on the GPU."""
    import torch
    from astro_b200 import rl
    torch.manual_seed(1)
    z, meta = H.load_traj()
    g = 0
    nb = z['g%d_nb' % g]
    off = np.concatenate([[0], np.cumsum(nb)])
    states = [H.state_from_arrays(z['g%d_ships' % g][k], z['g%d_planets' % g][k], z['g%d_bullets' % g][off[k]:off[k + 1]], 0.0, 0.0)
              for k in (0, 20, 40, 60)]
    net = rl.ValueNetwork(solo=False, nout=6).cuda()
    single = torch.stack([net.evaluate(s) for s in states])
    batch = net.evaluate_batch(states)
    assert float((single - batch).abs().max()) < 1e-6
    assert float((batch - net.evaluate_batch(states[::-1]).flip(0)).abs().max()) < 1e-6
    games = _games(core.DEFAULT_CONFIG, len(states), bullet_cap=32, precision=64)
    games.set_states(states, ticks=np.zeros(len(states), dtype=np.int64))
    q = net.forward_torch(games.observe())       # [n, 2, 6]: 36 rows incl. all -1 padding rows
    assert float((q[:, 0] - batch).abs().max()) < 1e-6
    rolled = net.evaluate_batch([core.roll_ships(s, 1) for s in states])
    assert float((q[:, 1] - rolled).abs().max()) < 1e-6


# ------------------------------------------------------------------ full-size properties

def _events_digest(games, ticks, auto_reset=True):
    import torch
    acc = torch.zeros(games.n, dtype=torch.int64, device=games.device)
    for k in range(ticks):
        _, _, ev = games.step(None, auto_reset=auto_reset, want_reward=False)
        acc = acc * 31 + ev.to(torch.int64) + 1
    return acc


def test_full_size_properties_1M_games():
    """BASELINE config #4 size on one GPU (1,048,576 games): conservation laws of the device
    counters, determinism, and shard-independence (a game's trajectory depends only on its
    global id, not on which shard holds it)."""
    cfg, N, K, T = core.DEFAULT_CONFIG, 1 << 20, 32, 150
    pool = H.make_pool(cfg, 1024)

    def run(n, first):
        games = _games(cfg, n, bullet_cap=K, precision=32, seed=9, first_game=first)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        return games, _events_digest(games, T)

    games, dig = run(N, 0)
    st = games.stats()
    assert st['env_steps'] == N * T and st['skipped'] == 0
    assert st['episodes'] == st['wins0'] + st['wins1'] + st['both_lost'] + st['timeouts']
    assert st['episodes'] > N // 2
    arr_nb = (games.meta.cpu().numpy().view(np.uint32) & 1023).astype(np.int64)
    # every bullet written by one tick is read by the next (games that end write none)
    assert st['bullets_in'] == st['bullets_out'] - int(arr_nb.sum())
    assert st['overflow'] == 0
    _, dig2 = run(N, 0)
    assert bool((dig == dig2).all())
    half = N // 2
    _, lo = run(half, 0)
    _, hi = run(half, half)
    assert bool((dig[:half] == lo).all()) and bool((dig[half:] == hi).all())
    # the same 150 ticks through astro_tick_many (one launch): every game's event history and the
    # counters are those of 150 separate launches
    import torch
    fused = _games(cfg, N, bullet_cap=K, precision=32, seed=9, first_game=0)
    fused.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    fused.reset_all()
    ev = torch.empty((T, fused.n_pad), dtype=torch.uint8, device='cuda')
    fused.step_many(T, None, events=ev, auto_reset=True)
    acc = torch.zeros(N, dtype=torch.int64, device='cuda')
    for k in range(T):
        acc = acc * 31 + ev[k, :N].to(torch.int64) + 1
    assert bool((acc == dig).all())
    assert fused.stats() == st


# ------------------------------------------------------------------ drop-in API (reference tests)

class _Nothing(core.Bot):
    def __call__(self, state):
        return 2


def test_create_step_roll_like_reference():
    """astro/test/test_core.py:20-52 against the drop-in module."""
    import itertools as it
    for base in (core.DEFAULT_CONFIG, core.SOLO_CONFIG, core.SOLO_EASY_CONFIG):
        for config in it.islice(core.generate_configs(base), 4):
            state = core.create(config)
            nships = 1 if config.solo else 2
            assert state.ships.x.shape == (nships, 2) and state.ships.b.shape == (nships,)
            assert 1 <= state.planets.x.shape[0] <= config.max_planets
            assert state.planets.b is None and state.bullets.b is None
            nxt, reward = core.step(state, np.full(nships, 2), config)
            assert nxt is not None and (reward == 0).all() and reward.shape == (nships,)
            assert nxt.ships.x.shape == state.ships.x.shape and nxt.t == config.dt
            rolled = core.roll_ships(nxt, nships - 1)
            assert rolled.ships.x.shape == nxt.ships.x.shape
            assert core.roll_ships(None, 0) is None


def test_play_solo_easy_and_log_roundtrip(tmp_path):
    """astro/test/test_core.py:55-64: a passive ship always falls into the planet."""
    game = core.play(core.SOLO_EASY_CONFIG, [_Nothing()])
    assert game.winner is None and len(game.ticks) > 10
    path = str(tmp_path / 'log' / 'game.jsonl')
    core.save_log(path, game)
    back = core.load_log(path)
    assert back.config == game.config and back.winner == game.winner and len(back.ticks) == len(game.ticks)
    for a, b in zip(back.ticks, game.ticks):
        assert np.array_equal(a.state.ships.x, b.state.ships.x) and np.array_equal(a.reward, b.reward)


def test_abi_errors_are_reported_not_thrown():
    import ctypes as C
    L = nat.lib()
    cfg = nat.AstroConfig()
    h = C.c_void_p()
    assert L.astro_batch_create(C.byref(cfg), 33, 32, 32, 0, C.byref(h)) == -1
    assert b'multiple of 32' in L.astro_last_error()
    assert L.astro_batch_create(C.byref(cfg), 32, 32, 16, 0, C.byref(h)) == -1
    assert L.astro_batch_create(C.byref(cfg), 32, 32, 32, 0, C.byref(h)) == 0
    assert L.astro_tick(h, None, None, None, None, 0, None) == -3      # not bound
    assert b'bind' in L.astro_last_error()
    assert L.astro_batch_destroy(h) == 0


# ------------------------------------------------------------------ scripted bots on the device

def test_script_controls_replay_golden_games_f64():
    """BASELINE config #1 (script bot vs script bot) without the host in the loop: the reference's
    scripted games are replayed free-running in the float64 build with the controls chosen by the
    device ScriptBot kernel — every control equals the one the reference's bot chose and every
    state stays bit-identical, to the last tick."""
    z, meta = H.load_traj()
    checked = 0
    for m in meta:
        if m['kind'] not in ('duel_script', 'solo_script_timeout', 'duel_nothing_vs_script'):
            continue
        g, S = m['game'], m['nships']
        cfg = H.config_from(m['config'])
        games = _games(cfg, 1, bullet_cap=32, precision=64)
        games.set_states([H.state_from_arrays(z['g%d_ships' % g][0], z['g%d_planets' % g][0], np.zeros((0, 4)), 0.0, 0.0)])
        for k in range(m['nticks']):
            arr = games.get_arrays()
            assert H.same_bits(arr['ships'][0], z['g%d_ships' % g][k]), (g, k)
            ctl = games.script_controls()
            if m['kind'] == 'duel_nothing_vs_script':
                ctl[:, 0] = 2   # script.NothingBot (script.py:6-10) flies ship 0
            assert (ctl[0].cpu().numpy() == z['g%d_control' % g][k]).all(), (g, k)
            reward, done, _ = games.step(ctl)
            assert H.same_bits(reward[0].cpu().numpy(), z['g%d_reward' % g][k]), (g, k)
            checked += 1
        assert bool(done[0].item()) == (not m['truncated'])
    assert checked > 900


@pytest.mark.parametrize('precision', [32, 64])
def test_script_controls_match_oracle_on_batched_states(precision):
    """4,096 games under random play, sampled every 7 ticks (so that planets, bullets and resets are in
    every phase): the device bot's control of every ship == the oracle's on the same state."""
    cfg = core.DEFAULT_CONFIG
    N, K, S = 4096, 32, 2
    pool = H.make_pool(cfg, 512)
    games = _games(cfg, N, bullet_cap=K, precision=precision)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    seen = np.zeros(6, dtype=np.int64)
    for k in range(140):
        if k % 7 == 0:
            arr = games.get_arrays()
            ob, _ = H.oracle_batch_from(arr, S, K)
            want = ao.script_batch(cfg, ob)
            got = games.script_controls()[:N].cpu().numpy()
            assert (got == want).all(), (k, np.nonzero((got != want).any(axis=1))[0][:8])
            seen += np.bincount(got.ravel(), minlength=6)
        games.step(None, auto_reset=True)
    assert seen[0] > 0 and seen[2] > 0 and seen[3] > 0 and seen[4] > 0   # left / idle / forward / right all occur
    # scripted self-play on the device: bot kernel -> tick kernel, no host in the loop
    games.stats(clear=True)
    for k in range(300):
        games.step(games.script_controls(), auto_reset=True)
    st = games.stats()
    assert st['env_steps'] == N * 300 and st['episodes'] > 0 and st['bullets_spawned'] > 0
    # finished games get the no-op control
    g1 = _games(cfg, 64, bullet_cap=K, precision=precision)
    assert (g1.script_controls().cpu().numpy() == 2).all()


def test_script_controls_solo():
    cfg = core.SOLO_CONFIG
    pool = H.make_pool(cfg, 64)
    games = _games(cfg, 512, bullet_cap=4, precision=32)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    for k in range(60):
        arr = games.get_arrays()
        ob, _ = H.oracle_batch_from(arr, 1, 4)
        got = games.script_controls()[:512].cpu().numpy()
        assert (got == ao.script_batch(cfg, ob)).all(), k
        games.step(got, auto_reset=True)


# ------------------------------------------------------------------ core.create on the device

def _host_pool(cfg, seeds):
    S = 1 if cfg.solo else 2
    ships = np.zeros((len(seeds), S, 5)); planets = np.zeros((len(seeds), 4, 4)); npl = np.zeros(len(seeds), dtype=np.int32)
    for i, sd in enumerate(seeds):
        s = core.create(cfg._replace(seed=int(sd)))
        ships[i, :, 0:2], ships[i, :, 2:4], ships[i, :, 4] = s.ships.x, s.ships.dx, s.ships.b
        p = s.planets.x.shape[0]
        planets[i, :p, 0:2], planets[i, :p, 2:4] = s.planets.x, s.planets.dx
        npl[i] = p
    return ships, planets, npl


def test_create_on_device_matches_reference_golden():
    """core.create (core.py:86-135) on the device against the 48 create() outputs recorded from the
    reference: float64 build bit for bit (MT19937 draw order, float32 islands, float64 planet
    velocities); float32 build = the same values rounded to float32."""
    z = np.load(os.path.join(H.G, 'create.npz'))
    meta = json.load(open(os.path.join(H.G, 'create.json')))
    for m in meta:
        cfg = H.config_from(m['config'])
        for prec in (64, 32):
            games = _games(cfg, 32, bullet_cap=4, precision=prec)
            ships, planets, npl = (t.cpu().numpy() for t in games.create_on_device([cfg.seed]))
            cast = (lambda a: np.asarray(a, dtype=np.float64)) if prec == 64 else (lambda a: np.asarray(a, dtype=np.float32).astype(np.float64))
            P = z[m['key'] + '_planets_x'].shape[0]
            assert npl[0] == P, m['key']
            assert H.same_bits(ships[0, :, 0:2], cast(z[m['key'] + '_ships_x'])), m['key']
            assert H.same_bits(ships[0, :, 2:4], cast(z[m['key'] + '_ships_dx'])), m['key']
            assert H.same_bits(ships[0, :, 4], cast(z[m['key'] + '_ships_b'])), m['key']
            assert H.same_bits(planets[0, :P, 0:2], cast(z[m['key'] + '_planets_x'])), m['key']
            assert H.same_bits(planets[0, :P, 2:4], cast(z[m['key'] + '_planets_dx'])), m['key']
            assert (planets[0, P:] == 0).all()


@pytest.mark.parametrize('cfg', [core.DEFAULT_CONFIG, core.SOLO_CONFIG, core.SOLO_EASY_CONFIG,
                                 core.DEFAULT_CONFIG._replace(max_planets=3, seed=7),
                                 core.DEFAULT_CONFIG._replace(max_planets=2, seed=123, planet_orbit=0.4, gravity=0.08)])
def test_create_on_device_matches_host_create_over_the_config_stream(cfg):
    """2,048 seeds of core.generate_configs: the device pool == pool.make_pool (host core.create),
    every bit, incl. rejection sampling for max_planets = 3 and the no-draw case max_planets = 1;
    then a rollout re-created from the device pool behaves exactly like one from the host pool."""
    M = 2048
    seeds = rng.config_seeds(cfg.seed, M)
    import itertools as it
    assert [c.seed for c in it.islice(core.generate_configs(cfg), 8)] == [int(x) for x in seeds[:8]]
    assert (rng.config_seeds(cfg.seed, 8, skip=5) == seeds[5:13]).all()
    want = H.make_pool(cfg, M)
    for prec in (64, 32):
        games = _games(cfg, 256, bullet_cap=32, precision=prec)
        ships, planets, npl = (t.cpu().numpy().astype(np.float64) if t.dtype.is_floating_point else t.cpu().numpy()
                               for t in games.create_on_device(seeds))
        cast = (lambda a: a) if prec == 64 else (lambda a: a.astype(np.float32).astype(np.float64))
        assert (npl == want['np']).all()
        assert H.same_bits(ships, cast(want['ships'])) and H.same_bits(planets, cast(want['planets']))
    a = _games(cfg, 1024, bullet_cap=32, precision=32)
    a.set_reset_pool_on_device(M)
    b = _games(cfg, 1024, bullet_cap=32, precision=32)
    b.set_reset_pool_arrays(want['ships'], want['planets'], want['np'])
    for g in (a, b):
        g.reset_all()
        for _ in range(120):
            g.step(None, auto_reset=True)
    xa, xb = a.get_arrays(), b.get_arrays()
    for k in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (xa[k] == xb[k]).all(), k
    assert a.stats() == b.stats() and a.stats()['episodes'] > 0


# ------------------------------------------------------------------ one observation tensor for both ships

def test_observe_shared_and_forward_both():
    """observe(shared=True) is exactly perspective 0 of observe(); ValueNetwork.forward_both on it
    gives both ships' values (fp32 tolerance 1e-6 against forward() on the two-perspective batch:
    the same products summed in a different order inside the first layer)."""
    import torch
    from astro_b200 import rl
    cfg, N, K = core.DEFAULT_CONFIG, 4096, 32
    pool = H.make_pool(cfg, 256)
    games = _games(cfg, N, bullet_cap=K, precision=32, seed=3)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    for _ in range(80):
        games.step(None, auto_reset=True)
    games.step(None, auto_reset=False)
    full = games.observe()
    shared = games.observe(shared=True)
    assert shared.shape == (N, 36, 15)
    assert torch.equal(shared, full[:, 0])
    torch.manual_seed(0)
    net = rl.ValueNetwork(solo=False, nout=6).to(full.device)
    with torch.no_grad():
        q_full = net.forward_torch(full)     # [N, 2, 6]
        q_both = net.forward_both(shared)    # [N, 2, 6]
    assert q_both.shape == q_full.shape
    assert float((q_both - q_full).abs().max()) <= 1e-6
    live = (games.get_arrays()['finished'] == 0)
    a_full, a_both = q_full.argmax(-1).cpu().numpy()[live], q_both.argmax(-1).cpu().numpy()[live]
    assert (a_full == a_both).mean() > 0.999


# ------------------------------------------------------------------ JSONL logs of batched rollouts

def test_game_recorder_writes_reference_format_logs(tmp_path):
    """logs.GameRecorder over a batched float64 rollout: the recorded games equal core.play-style
    records — every Tick holds the pre-step state, replaying the logged controls through the
    oracle reproduces each next state bit for bit, the winner follows core.py:409 — and the files
    load back through load_log in the reference's JSONL format."""
    from astro_b200 import logs
    cfg = core.DEFAULT_CONFIG
    N, K = 256, 32
    pool = H.make_pool(cfg, 64)
    games = _games(cfg, N, bullet_cap=K, precision=64, seed=5)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    follow = [0, 37, 255]
    rec = logs.GameRecorder(games, follow, folder=str(tmp_path / 'logs'))
    for k in range(400):
        if k % 2:
            rec.step(None, auto_reset=True)                       # device counter-stream controls
        else:
            rec.step(games.script_controls(), auto_reset=True)    # device ScriptBot controls
    assert len(rec.finished) >= 3 and len(rec.paths) == len(rec.finished)
    for game, path in zip(rec.finished, rec.paths):
        assert game.ticks[0].state.t == 0.0 and game.ticks[0].state.bullets.x.shape == (0, 2)
        for a, b in zip(game.ticks[:-1], game.ticks[1:]):
            ob = ao.Batch(1, 2, K)
            P, B = a.state.planets.x.shape[0], a.state.bullets.x.shape[0]
            ob.ships[0, :, 0:2], ob.ships[0, :, 2:4], ob.ships[0, :, 4] = a.state.ships.x, a.state.ships.dx, a.state.ships.b
            ob.planets[0, :P, 0:2], ob.planets[0, :P, 2:4] = a.state.planets.x, a.state.planets.dx
            ob.bullets[0, :B, 0:2], ob.bullets[0, :B, 2:4] = a.state.bullets.x, a.state.bullets.dx
            ob.np_[0], ob.nb[0], ob.reload[0], ob.t[0] = P, B, a.state.reload, a.state.t
            o2, rew, done, ev = ao.step_batch(cfg, ob, a.control.reshape(1, 2))
            assert not done[0] and (rew[0] == a.reward).all()
            assert H.same_bits(o2.ships[0, :, 0:2], b.state.ships.x) and H.same_bits(o2.ships[0, :, 4], b.state.ships.b)
            assert o2.nb[0] == b.state.bullets.x.shape[0]
            assert H.same_bits(o2.bullets[0, :o2.nb[0], 0:2], b.state.bullets.x)
        last = game.ticks[-1]
        assert (last.reward != 0).any() or last.state.t + cfg.dt >= cfg.max_time
        assert game.winner == (None if last.reward.max() < 1 else int(last.reward.argmax()))
        back = core.load_log(path)
        assert back.winner == game.winner and len(back.ticks) == len(game.ticks)
        assert np.array_equal(back.ticks[3 % len(back.ticks)].state.ships.x, game.ticks[3 % len(game.ticks)].state.ships.x)
        head = json.loads(open(path).readline())
        assert head['config']['_type'] == 'astro.core:Config'


# ------------------------------------------------------------------ fused features + value network

@pytest.mark.parametrize('solo', [False, True])
def test_policy_kernel_matches_value_network(solo):
    """astro_policy_controls == ValueNetwork.forward(observe()) -> argmax, for every game and both
    perspectives: outputs within 2e-6 of the PyTorch fp32 network (same products, different
    summation order), controls identical wherever the top two outputs are further apart than that."""
    import torch
    from astro_b200 import rl
    cfg = core.SOLO_CONFIG if solo else core.DEFAULT_CONFIG
    S, N, K = (1 if solo else 2), 4096 + 32, 32
    pool = H.make_pool(cfg, 256)
    games = _games(cfg, N, bullet_cap=K, precision=32, seed=4)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    for _ in range(70):
        games.step(None, auto_reset=True)
    games.step(None, auto_reset=False)            # leaves a few finished games behind
    torch.manual_seed(2)
    net = rl.ValueNetwork(solo=solo, nout=6).to(games.device)
    with torch.no_grad():
        for prm in net.parameters():              # livelier than the default init: spread the outputs
            prm.mul_(3.0)
        want = net.forward_torch(games.observe())  # [N, S, 6]
    games.set_policy(net)
    q = torch.empty((games.n_pad, S, 6), dtype=torch.float32, device=games.device)
    act = games.policy_controls(q_out=q)
    fin = torch.from_numpy(games.get_arrays()['finished']).to(games.device)
    assert fin.any()
    live = ~fin
    err = (q[:N][live] - want[live]).abs().max().item()
    assert err <= 2e-6, err
    assert (q[:N][fin] == 0).all() and (act[:N][fin] == 2).all()
    top2 = want.topk(2, dim=-1).values
    clear = live.unsqueeze(-1) & ((top2[..., 0] - top2[..., 1]) > 1e-5)
    assert clear.float().mean() > 0.9
    assert (act[:N].long()[clear] == want.argmax(-1)[clear]).all()
    assert len(torch.unique(act[:N][live])) >= 3
    # ship_mask: only ship 0's column is written
    if not solo:
        out = torch.full((games.n_pad, 2), 9, dtype=torch.uint8, device=games.device)
        games.policy_controls(out=out, ships=[0])
        assert (out[:, 1] == 9).all() and (out[:N, 0] == act[:N, 0]).all()


@pytest.mark.parametrize('N,T', [(1024, 150), (16384, 1000)])
def test_policy_rollout_equals_torch_rollout(N, T):
    """A self-play rollout driven by the fused kernel ends in the same statistics as one driven by
    observe() -> ValueNetwork -> argmax — BASELINE config #5, at a reduced size and at its stated size
    (16,384 games x 1,000 ticks, observation extraction feeding the policy batch every tick)."""
    import torch
    from astro_b200 import rl
    cfg, K = core.DEFAULT_CONFIG, 32
    pool = H.make_pool(cfg, 256)
    torch.manual_seed(5)
    net = rl.ValueNetwork(solo=False, nout=6).cuda()
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(3.0)
    runs = []
    for fused in (False, True):
        games = _games(cfg, N, bullet_cap=K, precision=32, seed=9)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        games.set_policy(net)
        same = 0
        for k in range(T):
            with torch.no_grad():
                a_torch = net.forward_torch(games.observe()).argmax(-1).to(torch.uint8)
            a_fused = games.policy_controls()[:N]
            same += int((a_torch == a_fused).sum())
            games.step(a_fused if fused else a_torch, auto_reset=True)
        runs.append((games.stats(), same / (T * N * 2)))
    assert runs[0][1] > 0.9995 and runs[1][1] > 0.9995          # controls agree except at near-ties
    assert runs[0][0]['env_steps'] == N * T
    assert abs(runs[0][0]['episodes'] - runs[1][0]['episodes']) <= 0.05 * runs[0][0]['episodes'] + 5


# ------------------------------------------------------------------ whole game loops on the device

@pytest.mark.parametrize('bots', [('script', 'script'), ('policy', 'script'), ('nothing', 'script'), ('policy', 'policy'),
                                  ('stream', 'stream'), ('explore', 'script'), ('explore', 'explore')])
def test_rollout_device_equals_tick_by_tick_loop(bots):
    """astro_rollout_device == the same loop driven from Python one call at a time: identical final
    state and statistics (the bot kernels write the controls the tick consumes, nothing else differs)."""
    import torch
    from astro_b200 import rl
    cfg, N, K, T = core.DEFAULT_CONFIG, 2048, 32, 160
    pool = H.make_pool(cfg, 256)
    torch.manual_seed(11)
    net = rl.ValueNetwork(solo=False, nout=6).cuda()
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(3.0)
    out = []
    for fused_loop in (True, False):
        games = _games(cfg, N, bullet_cap=K, precision=32, seed=13)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        games.set_policy(net)
        xstate = games.set_exploration(1.0, 0.1, seed=5)
        if fused_loop:
            games.rollout_device(T, bots=bots)
        else:
            for k in range(T):
                if bots[0] == 'stream':
                    games.step(None, auto_reset=True)
                    continue
                a = games.script_controls() if 'script' in bots else torch.full((games.n_pad, 2), 2, dtype=torch.uint8, device='cuda')
                for s, b in enumerate(bots):
                    if b == 'nothing':
                        a[:, s] = 2
                ships = [s for s, b in enumerate(bots) if b in ('policy', 'explore')]
                if ships:
                    games.policy_controls(out=a, ships=ships)
                ships = [s for s, b in enumerate(bots) if b == 'explore']
                if ships:
                    games.explore_controls(a, xstate, 1.0, 0.1, seed=5, ships=ships)
                games.step(a, auto_reset=True)
        out.append((games.get_arrays(), games.stats()))
    (xa, sa), (xb, sb) = out
    assert sa == sb and sa['env_steps'] == N * T and sa['episodes'] > 0
    for k in ('ships', 'planets', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (xa[k] == xb[k]).all(), k
    live = np.arange(K)[None, :] < xa['n_bullets'][:, None]
    assert (xa['bullets'][live] == xb['bullets'][live]).all()
    if bots == ('nothing', 'script'):
        assert sa['wins1'] > sa['wins0']       # the scripted ship beats the idle one


def test_abi_errors_of_the_bot_and_create_entry_points():
    """Every new entry point reports misuse through its return code and astro_last_error()."""
    import ctypes as C
    import torch
    L = nat.lib()
    games = _games(core.DEFAULT_CONFIG, 64, bullet_cap=8, precision=32)
    h, st = games._h, games._stream()
    act = torch.zeros((64, 2), dtype=torch.uint8, device='cuda')
    assert L.astro_script_controls(h, 0.1, 0.45, None, st) == -1 and b'null' in L.astro_last_error()
    assert L.astro_policy_controls(h, act.data_ptr(), None, 3, st) == -3 and b'astro_policy_set_weights' in L.astro_last_error()
    w = np.zeros(10, dtype=np.float32)
    assert L.astro_policy_set_weights(h, w.ctypes.data_as(C.c_void_p), 10, 6) == -1 and b'expected 4934 floats' in L.astro_last_error()
    assert L.astro_policy_set_weights(h, w.ctypes.data_as(C.c_void_p), 10, 9) == -1
    assert L.astro_rollout_device(h, 4, 2, 1, 0.1, 0.45, act.data_ptr(), None, 0, st) == -3      # policy without weights
    assert L.astro_rollout_device(h, 4, 0, 1, 0.1, 0.45, act.data_ptr(), None, 0, st) == -1      # stream mixed with a bot
    assert L.astro_rollout_device(h, 4, 1, 1, 0.1, 0.45, None, None, 0, st) == -1                # bots need the scratch buffer
    assert L.astro_rollout_device(h, 4, 7, 1, 0.1, 0.45, act.data_ptr(), None, 0, st) == -1
    cc = nat.AstroCreateConfig(0.2, 0.9, 0.5, 5, 0)
    seeds = torch.zeros(4, dtype=torch.int32, device='cuda')
    buf = torch.zeros(4 * 2 * 5 + 4 * 16 + 4, dtype=torch.float32, device='cuda')
    assert L.astro_create_games(h, C.byref(cc), seeds.data_ptr(), 4, buf.data_ptr(), buf.data_ptr(), buf.data_ptr(), st) == -1
    assert b'max_planets' in L.astro_last_error()
    assert L.astro_observe_shared(h, None, 12, st) == -1
    big = nat.AstroConfig()
    hh = C.c_void_p()
    assert L.astro_batch_create(C.byref(big), 1 << 26, 64, 32, 0, C.byref(hh)) == -1 and b'2^31' in L.astro_last_error()
    # astro_tick_many / bullet buffer entry points
    assert L.astro_tick_many(h, None, None, None, None, -1, 0, st) == -1 and b'n_ticks' in L.astro_last_error()
    assert L.astro_tick_many(h, None, None, None, None, 3, nat.TICK_AUTO_RESET, st) == -3 and b'astro_set_reset_pool' in L.astro_last_error()
    assert L.astro_tick_many(h, None, None, None, None, 0, 0, st) == 0                    # zero ticks: nothing to do
    assert L.astro_bullet_buffer(h) == 0 and L.astro_set_bullet_buffer(h, 2) == -1
    assert L.astro_tick_many(h, None, None, None, None, 3, 0, st) == 0 and L.astro_bullet_buffer(h) == 1   # odd count: flipped
    assert L.astro_set_bullet_buffer(h, 0) == 0                                          # (all slots finished: the lists are empty)
    # a working call after the failures
    assert L.astro_script_controls(h, 0.1, 0.45, act.data_ptr(), st) == 0
    torch.cuda.synchronize()
    assert (act.cpu().numpy() == 2).all()      # every slot is still finished: no-op controls


def test_policy_kernel_float64_state():
    """The fused policy kernel on the float64 validation build: features are cast to float32 exactly
    as rl.py:62-70 casts them, so the outputs match the network on observe() of the same batch."""
    import torch
    from astro_b200 import rl
    cfg, N = core.DEFAULT_CONFIG, 512
    pool = H.make_pool(cfg, 64)
    games = _games(cfg, N, bullet_cap=32, precision=64, seed=8)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    for _ in range(60):
        games.step(None, auto_reset=True)
    torch.manual_seed(3)
    net = rl.ValueNetwork(solo=False, nout=6).cuda()
    games.set_policy(net)
    q = torch.empty((games.n_pad, 2, 6), dtype=torch.float32, device='cuda')
    games.policy_controls(q_out=q)
    with torch.no_grad():
        want = net.forward_torch(games.observe())
    assert float((q[:N] - want).abs().max()) <= 2e-6


def test_tick_many_solo_and_float64_fall_back_to_single_launches():
    """astro_tick_many on the builds without the fused kernel (float64 state: one launch per tick inside the call) and on
    solo games (S = 1 instantiation of the fused kernel): same outcome as separate ticks."""
    import torch
    for cfg, prec in ((core.DEFAULT_CONFIG, 64), (core.SOLO_CONFIG, 32)):
        pool = H.make_pool(cfg, 256)
        outs = []
        for fused in (False, True):
            g = _games(cfg, 1024, bullet_cap=32, precision=prec, seed=3)
            g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
            g.reset_all()
            ev = torch.zeros((40, g.n_pad), dtype=torch.uint8, device='cuda')
            if fused:
                g.step_many(40, None, events=ev, auto_reset=True)
            else:
                for k in range(40):
                    ev[k] = g.step(None, auto_reset=True)[2]
            outs.append((g.get_arrays(), ev.cpu().numpy(), g.stats()))
        (a0, e0, s0), (a1, e1, s1) = outs
        assert (e0 == e1).all() and s0 == s1 and s0['env_steps'] == 1024 * 40
        assert H.same_bits(a0['ships'], a1['ships']) and (a0['tick'] == a1['tick']).all() and (a0['n_bullets'] == a1['n_bullets']).all()


@pytest.mark.gpu
@pytest.mark.parametrize('with_actions', [False, True])
def test_tick_many_equals_tick_by_tick(with_actions):
    """astro_tick_many (ticks of a tile back to back inside one launch, state handed on through L2) against the
    same ticks as separate launches: every tick's events, rewards and done flags, the final state bit for bit and
    the episode statistics — over fire ticks, deaths, re-creations and a launch boundary (270 ticks > 256 per launch)."""
    import torch
    cfg, N, K, T = core.DEFAULT_CONFIG, 4096, 32, 270
    pool = H.make_pool(cfg, 512)
    runs = []
    for fused in (False, True):
        g = _games(cfg, N, bullet_cap=K, precision=32, seed=5)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        for _ in range(40):                      # bullets in the air before the comparison starts
            g.step(None, auto_reset=True)
        g.stats(clear=True)
        gen = torch.Generator(device='cpu').manual_seed(11)
        acts = torch.randint(0, 6, (T, g.n_pad, 2), dtype=torch.uint8, generator=gen).cuda() if with_actions else None
        ev = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
        rw = torch.zeros((T, g.n_pad, 2), dtype=torch.float32, device='cuda')
        dn = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
        if fused:
            g.step_many(T, acts, events=ev, reward=rw, done=dn, auto_reset=True)
        else:
            for k in range(T):
                r, d, e = g.step(None if acts is None else acts[k], auto_reset=True)
                ev[k], rw[k], dn[k] = e, r, d
        runs.append((g.get_arrays(), ev.cpu().numpy(), rw.cpu().numpy(), dn.cpu().numpy(), g.stats()))
    (a0, e0, r0, d0, s0), (a1, e1, r1, d1, s1) = runs
    assert (e0 == e1).all() and (r0 == r1).all() and (d0 == d1).all()
    assert s0 == s1 and s0['episodes'] > 1000 and s0['bullets_spawned'] > 10000
    for k in ('n_bullets', 'n_planets', 'tick', 'episode', 'finished'):
        assert (a0[k] == a1[k]).all(), k
    assert H.same_bits(a0['ships'], a1['ships'])
    pm = np.arange(4)[None, :] < a0['n_planets'][:, None]
    bm = np.arange(K)[None, :] < a0['n_bullets'][:, None]
    assert H.same_bits(a0['planets'][pm], a1['planets'][pm]) and H.same_bits(a0['bullets'][bm], a1['bullets'][bm])


@pytest.mark.parametrize('with_actions', [False, True])
def test_tick_many_without_auto_reset_freezes_games_like_separate_ticks(with_actions):
    """astro_tick_many with auto-reset OFF (replays, rollout_host(auto_reset=False)): a game that ends on a non-last
    tick of a launch must leave its finished word (and the ending tick's ships) in memory at once — the later ticks of
    the launch skip it.  A short max_time makes every game end mid-launch; compared with separate astro_tick calls on
    meta, ships, bullets, events, done — and the launch that follows must skip the frozen games, not resurrect them."""
    import torch
    cfg, N, K, T = core.DEFAULT_CONFIG._replace(max_time=0.9), 2048, 32, 48     # timeout on a game's 45th tick
    pool = H.make_pool(cfg, 256)
    runs = []
    for fused in (False, True):
        g = _games(cfg, N, bullet_cap=K, precision=32, seed=9)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        for _ in range(20):
            g.step(None, auto_reset=True)                 # games now sit at different ticks: they time out on ticks 25..45 of T
        g.stats(clear=True)
        gen = torch.Generator(device='cpu').manual_seed(3)
        acts = torch.randint(0, 6, (T + 8, g.n_pad, 2), dtype=torch.uint8, generator=gen).cuda() if with_actions else None
        ev = torch.zeros((T + 8, g.n_pad), dtype=torch.uint8, device='cuda')
        dn = torch.zeros((T + 8, g.n_pad), dtype=torch.uint8, device='cuda')
        if fused:
            g.step_many(T, None if acts is None else acts[:T].contiguous(), events=ev[:T], done=dn[:T], auto_reset=False)
        else:
            for k in range(T):
                _, d, e = g.step(None if acts is None else acts[k], auto_reset=False)
                ev[k], dn[k] = e, d
        mid = g.get_arrays()
        # the follow-up launch: frozen games are skipped (ASTRO_EV_SKIPPED), the others carry on
        if fused:
            g.step_many(8, None if acts is None else acts[T:].contiguous(), events=ev[T:], done=dn[T:], auto_reset=False)
        else:
            for k in range(T, T + 8):
                _, d, e = g.step(None if acts is None else acts[k], auto_reset=False)
                ev[k], dn[k] = e, d
        runs.append((mid, g.get_arrays(), ev.cpu().numpy(), dn.cpu().numpy(), g.stats(), g.observe().cpu().numpy()))
    (m0, a0, e0, d0, s0, o0), (m1, a1, e1, d1, s1, o1) = runs
    assert (e0 == e1).all() and (d0 == d1).all() and s0 == s1
    assert m0['finished'].sum() > N // 2 and s0['skipped'] > 0
    assert ((e0[T:] & nat.EV_SKIPPED) != 0).sum() >= m0['finished'].sum() * 8
    for a, b in ((m0, m1), (a0, a1)):
        for k in ('n_bullets', 'n_planets', 'tick', 'episode', 'finished'):
            assert (a[k] == b[k]).all(), k
        assert H.same_bits(a['ships'], b['ships'])        # finished games included: the ending tick's post-step ships
        live = ~a['finished']
        pm = (np.arange(4)[None, :] < a['n_planets'][:, None]) & live[:, None]
        bm = (np.arange(K)[None, :] < a['n_bullets'][:, None]) & live[:, None]
        assert H.same_bits(a['planets'][pm], b['planets'][pm]) and H.same_bits(a['bullets'][bm], b['bullets'][bm])
    assert H.same_bits(o0, o1)


def test_explore_controls_match_host_twin_and_the_reference_process():
    """astro_explore_controls (rl.EpsilonGreedy, rl.py:10-30, as rl.QBotTrainer lays it over the greedy control,
    rl.py:249-258): every ship's state and control equal the host twin (astro_b200/rng.py explore_step, same counter
    stream) tick by tick, through deaths and re-creations (dt < 0 on a new game's first call); and the process has
    the reference's statistics: stationary active fraction p_in / (p_in + p_out) with p = 1 - exp(-dt / t), random
    controls uniform on 0..4 (randint(0, 5) never draws 5)."""
    import torch
    cfg, N, T, seed = core.DEFAULT_CONFIG, 4096, 400, 7
    pool = H.make_pool(cfg, 256)
    g = _games(cfg, N, bullet_cap=32, precision=32, seed=2, first_game=1000)
    g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    g.reset_all()
    state = torch.zeros((g.n_pad, 2), dtype=torch.int32, device='cuda')
    host_state = np.zeros((N, 2), dtype=np.int32)
    ids = 1000 + np.arange(N)
    active = 0
    hist = np.zeros(6, dtype=np.int64)
    entered = left = idle_calls = active_calls = 0
    for k in range(T):
        acts = torch.full((g.n_pad, 2), 2, dtype=torch.uint8, device='cuda')
        arr_tick = (g.meta.cpu().numpy().view(np.uint32)[:N] >> 14).astype(np.int64)
        before = (host_state & 0xff) - 1
        ref = rng.explore_step(seed, ids, g.step_index, arr_tick, host_state, cfg.dt, 1.0, 0.1)
        g.explore_controls(acts, state, t_in=1.0, t_out=0.1, seed=seed)
        got = acts.cpu().numpy()[:N].astype(np.int64)
        assert (got == np.where(ref >= 0, ref, 2)).all(), k
        assert (state.cpu().numpy()[:N] == host_state).all(), k
        active += int((ref >= 0).sum())
        hist += np.bincount(ref[ref >= 0], minlength=6)
        same_game = (arr_tick[:, None] > 0) | (k == 0)
        idle_calls += int(((before < 0) & same_game).sum())
        entered += int(((before < 0) & (ref >= 0) & same_game).sum())
        active_calls += int(((before >= 0) & same_game).sum())
        left += int(((before >= 0) & (ref < 0) & same_game).sum())
        g.step(acts, auto_reset=True)
    p_in, p_out = 1 - np.exp(-cfg.dt / 1.0), 1 - np.exp(-cfg.dt / 0.1)
    assert abs(entered / idle_calls - p_in) < 0.1 * p_in and abs(left / active_calls - p_out) < 0.05 * p_out
    frac = active / (N * 2 * T)
    assert abs(frac - p_in / (p_in + p_out)) < 0.01, frac
    assert hist[5] == 0 and hist[:5].min() > 0.9 * hist[:5].mean()
    L = nat.lib()
    assert L.astro_explore_controls(g._h, 0.0, 0.1, 0, state.data_ptr(), state.data_ptr(), 3, g._stream()) == -1
    assert L.astro_explore_controls(g._h, 1.0, 0.1, 0, None, state.data_ptr(), 3, g._stream()) == -1


@pytest.mark.parametrize('N,K', [(45, 3), (32, 1023), (7, 0), (1, 32)])
def test_extreme_sizes_teacher_forced_and_fused(N, K):
    """Ragged and extreme shapes: a game count that is not a multiple of the 32-game tile (padding slots stay finished),
    one game, the largest bullet pool the meta word can count (K = 1023), no pool at all (K = 0: every newborn
    overflows) — the same teacher-forced check against the oracle, and astro_tick_many against separate launches."""
    import torch
    cfg = core.DEFAULT_CONFIG
    games, worst, n_done, n_fired = _teacher_forced(cfg, N, K, 90, 32, pool_size=64)
    assert n_fired > 0
    if K == 0:
        assert games.stats()['overflow'] > 0 and games.stats()['bullets_out'] == 0
    pool = H.make_pool(cfg, 64)
    outs = []
    for fused in (False, True):
        g = _games(cfg, N, bullet_cap=K, precision=32, seed=1)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        ev = torch.zeros((70, g.n_pad), dtype=torch.uint8, device='cuda')
        if fused:
            g.step_many(70, None, events=ev, auto_reset=True)
        else:
            for k in range(70):
                ev[k, :N] = g.step(None, auto_reset=True)[2]
        outs.append((g.get_arrays(), ev.cpu().numpy()[:, :N], g.stats()))
    (a0, e0, s0), (a1, e1, s1) = outs
    assert (e0 == e1).all() and s0 == s1 and s0['env_steps'] == N * 70
    for key in ('ships', 'n_bullets', 'n_planets', 'tick', 'episode'):
        assert (a0[key] == a1[key]).all(), key


def test_timeouts_inside_fused_launches():
    """A short max_time (timeout on a game's 50th tick; ticks are per game, so re-created games time out at different
    launch ticks): timeout terminal, its reward and the re-creation — against the oracle tick by tick, and the same
    through astro_tick_many."""
    import torch
    cfg = core.DEFAULT_CONFIG._replace(max_time=1.0)
    games, worst, n_done, n_fired = _teacher_forced(cfg, 256, 32, 130, 32, pool_size=64)
    assert games.stats()['timeouts'] > 100
    pool = H.make_pool(cfg, 64)
    outs = []
    for fused in (False, True):
        g = _games(cfg, 256, bullet_cap=32, precision=32, seed=1)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        ev = torch.zeros((130, g.n_pad), dtype=torch.uint8, device='cuda')
        rw = torch.zeros((130, g.n_pad, 2), dtype=torch.float32, device='cuda')
        if fused:
            g.step_many(130, None, events=ev, reward=rw, auto_reset=True)
        else:
            for k in range(130):
                r, _, e = g.step(None, auto_reset=True)
                ev[k], rw[k] = e, r
        outs.append((g.get_arrays(), ev.cpu().numpy(), rw.cpu().numpy(), g.stats()))
    (a0, e0, r0, s0), (a1, e1, r1, s1) = outs
    assert (e0 == e1).all() and (r0 == r1).all() and s0 == s1 and s0['timeouts'] > 100
    assert ((e0 & nat.EV_TIMEOUT) != 0).sum() == s0['timeouts']
    for key in ('ships', 'n_bullets', 'tick', 'episode'):
        assert (a0[key] == a1[key]).all(), key


def test_set_states_inside_live_tiles_keeps_the_other_games_lists():
    """Writing single games into tiles that hold other games' bullets (the tile list is unpacked, edited and packed
    again, batched.set_arrays): the other games are untouched, the written ones read back exactly, and the batch
    ticks on from there like a batch built from scratch with the same states."""
    cfg, N, K = core.DEFAULT_CONFIG, 96, 32
    pool = H.make_pool(cfg, 64)
    a = _games(cfg, N, bullet_cap=K, precision=32, seed=3)
    a.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    a.reset_all()
    for _ in range(60):
        a.step(None, auto_reset=True)
    before = a.get_arrays()
    assert before['n_bullets'].sum() > 100
    src, dst = [70, 71, 5], [3, 35, 36]
    donors = a.get_states(src)
    a.set_states(donors, index=dst)
    after = a.get_arrays()
    keep = np.ones(N, dtype=bool)
    keep[dst] = False
    live = np.arange(K)[None, :] < before['n_bullets'][:, None]
    for key in ('ships', 'planets', 'n_bullets', 'n_planets', 'tick'):
        assert (after[key][keep] == before[key][keep]).all(), key
    assert (after['bullets'][keep][live[keep]] == before['bullets'][keep][live[keep]]).all()
    for s, d in zip(src, dst):
        assert (after['ships'][d] == before['ships'][s]).all() and after['n_bullets'][d] == before['n_bullets'][s]
        nb = before['n_bullets'][s]
        assert (after['bullets'][d, :nb] == before['bullets'][s, :nb]).all()
        assert (after['planets'][d, :before['n_planets'][s]] == before['planets'][s, :before['n_planets'][s]]).all()
    # a twin built from scratch with the same states ticks identically
    b = _games(cfg, N, bullet_cap=K, precision=32, seed=3)
    b.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    b.set_arrays(after['ships'], after['planets'], after['n_planets'], after['bullets'], after['n_bullets'], after['tick'])
    b.set_stream(step=a.step_index)
    for _ in range(30):
        ea = a.step(None, auto_reset=False)[2].cpu().numpy()
        eb = b.step(None, auto_reset=False)[2].cpu().numpy()
        assert (ea == eb).all()
    xa, xb = a.get_arrays(), b.get_arrays()
    ok = ~xa['finished']
    assert (xa['finished'] == xb['finished']).all() and (xa['ships'][ok] == xb['ships'][ok]).all() and (xa['n_bullets'][ok] == xb['n_bullets'][ok]).all()


# ------------------------------------------------------------------ round 2: reference-pinned network, raw create(), guards

def _golden_states(z, e):
    g = e['game']
    nb = z['g%d_nb' % g]
    off = np.concatenate([[0], np.cumsum(nb)])
    return [H.state_from_arrays(z['g%d_ships' % g][k], z['g%d_planets' % g][k], z['g%d_bullets' % g][off[k]:off[k + 1]], 0.0, 0.0)
            for k in e['ticks']]


@pytest.mark.parametrize('precision', [64, 32])
def test_policy_kernel_matches_reference_network_outputs(precision):
    """The fused policy kernel (features + network, no observation tensor) against outputs of the UNMODIFIED
    reference: rl.ValueNetwork.evaluate_batch (rl.py:140-165) with seeded weights on states of the golden games,
    ship 0's perspective and ship 1's (core.roll_ships) — tests/golden/network.npz.  float64 state: q within 2e-6
    and the argmax equal off ties; float32 state (bearings rounded to float32 before norm_angle): within 2e-5."""
    import torch
    from astro_b200 import rl
    z, _ = H.load_traj()
    gold = np.load(os.path.join(H.G, 'network.npz'))
    fm = json.load(open(os.path.join(H.G, 'features.json')))
    tol = 2e-6 if precision == 64 else 2e-5
    for solo in (False, True):
        entries = [e for e in fm if (e['nships'] == 1) == solo]
        states, want0, want1 = [], [], []
        for e in entries:
            states += _golden_states(z, e)
            want0.append(gold['g%d_q0' % e['game']])
            if not solo:
                want1.append(gold['g%d_q1' % e['game']])
        want = np.concatenate(want0)[:, None, :] if solo else np.stack([np.concatenate(want0), np.concatenate(want1)], axis=1)
        net = rl.ValueNetwork(solo=solo, nout=6)
        pre = 'solo_' if solo else 'duel_'
        net.load_state_dict({k: torch.from_numpy(gold[pre + k.replace('.', '_')]) for k in net.state_dict()})
        cfg = core.SOLO_CONFIG if solo else core.DEFAULT_CONFIG
        cap = max(32, max(s.bullets.x.shape[0] for s in states))
        games = _games(cfg, len(states), bullet_cap=cap, precision=precision)
        games.set_states(states, ticks=np.zeros(len(states), dtype=np.int64))
        games.set_policy(net)
        S = 1 if solo else 2
        q = torch.empty((games.n_pad, S, 6), dtype=torch.float32, device='cuda')
        act = games.policy_controls(q_out=q).cpu().numpy()[:len(states)]
        got = q.cpu().numpy()[:len(states)]
        assert np.abs(got - want).max() <= tol, (solo, np.abs(got - want).max())
        top = np.sort(want, axis=-1)
        clear = (top[..., -1] - top[..., -2]) > 10 * tol
        assert clear.mean() > 0.8 and (act[clear] == want.argmax(-1)[clear]).all()
        # the PyTorch twin on the device's own observation: forward (both perspectives) and forward_both
        net = net.cuda()
        with torch.no_grad():
            obs = games.observe()
            assert float((net.forward_torch(obs)[:len(states)].cpu() - torch.from_numpy(want)).abs().max()) <= tol
            assert float((net(obs)[:len(states)].cpu() - torch.from_numpy(want)).abs().max()) <= tol      # the fused kernel (astro_value_forward)
            if not solo:
                both = net.forward_both(games.observe(shared=True))
                assert float((both[:len(states)].cpu() - torch.from_numpy(want)).abs().max()) <= tol


def test_two_batches_hold_two_networks():
    """The policy weights belong to the batch handle: two batches with different networks do not share the last one set."""
    import torch
    from astro_b200 import rl
    cfg = core.DEFAULT_CONFIG
    pool = H.make_pool(cfg, 64)
    outs = []
    batches = []
    for seed in (1, 2):
        g = _games(cfg, 256, bullet_cap=32, precision=32, seed=0)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        torch.manual_seed(seed)
        net = rl.ValueNetwork(solo=False, nout=6).cuda()
        g.set_policy(net)
        batches.append((g, net))
    for g, net in batches:      # both networks were loaded before either is used
        q = torch.empty((g.n_pad, 2, 6), dtype=torch.float32, device='cuda')
        g.policy_controls(q_out=q)
        with torch.no_grad():
            assert float((q[:256] - net.forward_torch(g.observe())).abs().max()) <= 2e-6
        outs.append(q)
    assert float((outs[0] - outs[1]).abs().max()) > 1e-3


def test_core_step_from_raw_create_matches_reference_play():
    """core.play's loop from core.create's RAW arrays (float32): the reference runs the first tick partly in float32
    (NEP 50), which astro_b200.core.step reproduces (ASTRO_TICK_ALL_CREATE_DTYPES) — every state of the reference's
    games, bit for bit, free-running from create() (tests/golden/traj_raw.npz), fire-on-the-first-tick included."""
    z = np.load(os.path.join(H.G, 'traj_raw.npz'))
    meta = json.load(open(os.path.join(H.G, 'traj_raw.json')))
    total = 0
    for m in meta:
        g = m['game']
        cfg = H.config_from(m['config'])
        ships, planets, nb, bullets = z['g%d_ships' % g], z['g%d_planets' % g], z['g%d_nb' % g], z['g%d_bullets' % g]
        off = np.concatenate([[0], np.cumsum(nb)])
        state = core.create(cfg)
        assert state.ships.x.dtype == np.float32
        n = min(m['nticks'], 60)
        for k in range(n):
            assert H.same_bits(np.concatenate([state.ships.x, state.ships.dx, np.asarray(state.ships.b)[:, None]], 1), ships[k]), (g, k)
            assert H.same_bits(np.concatenate([state.planets.x, state.planets.dx], 1), planets[k]), (g, k)
            assert H.same_bits(np.concatenate([state.bullets.x, state.bullets.dx], 1).reshape(-1, 4), bullets[off[k]:off[k + 1]]), (g, k)
            assert state.reload == z['g%d_reload' % g][k] and state.t == z['g%d_t' % g][k]
            state, reward = core.step(state, z['g%d_control' % g][k], cfg)
            assert (np.asarray(reward, dtype=np.float64) == z['g%d_reward' % g][k]).all()
            total += 1
            if state is None:
                assert k == m['nticks'] - 1 and not m['truncated']
                break
    assert total > 600


def test_batched_float64_create_dtypes_flag():
    """ASTRO_TICK_CREATE_DTYPES on a float64 batch: games on their tick 0 (as re-created from a create() pool) run the
    reference's first-tick arithmetic, every other game the float64 one — against the oracle's raw / plain modes."""
    cfg, N, K = core.DEFAULT_CONFIG, 512, 32
    pool = H.make_pool(cfg, 256)
    games = _games(cfg, N, bullet_cap=K, precision=64, seed=2)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    games.tick_flags = nat.TICK_CREATE_DTYPES
    ids = np.arange(N)
    n_raw = 0
    for k in range(150):
        arr = games.get_arrays()
        ctl = rng.actions(2, ids, k, 2)
        want = [ao.step_one(cfg, arr['ships'][g], arr['planets'][g, :arr['n_planets'][g]], arr['bullets'][g, :arr['n_bullets'][g]],
                            games.schedule.reload[arr['tick'][g]], games.schedule.t[arr['tick'][g]], ctl[g], bullet_cap=K,
                            raw=bool(arr['tick'][g] == 0)) for g in range(0, N, 4)]
        n_raw += int((arr['tick'][::4] == 0).sum())
        _, done, ev = games.step(None, auto_reset=True)
        done, new = done.cpu().numpy(), games.get_arrays()
        for w, g in zip(want, range(0, N, 4)):
            assert bool(done[g]) == w['done'], (k, g)
            if not w['done']:
                assert H.same_bits(new['ships'][g], w['ships']) and H.same_bits(new['planets'][g, :w['planets'].shape[0]], w['planets']), (k, g)
                assert new['n_bullets'][g] == w['bullets'].shape[0] and H.same_bits(new['bullets'][g, :w['bullets'].shape[0]], w['bullets'])
    assert n_raw > 200


def test_control_codes_above_5_are_flagged_and_flown_as_no_op():
    """Control codes outside the reference's table (core.py:220-227): the tick flags the game (ASTRO_EV_BAD_CONTROL,
    counted in stats) and flies the ship with control 2 — in every kernel form; core.step rejects them."""
    import torch
    cfg, N, K = core.DEFAULT_CONFIG, 1024, 32
    pool = H.make_pool(cfg, 128)
    gen = torch.Generator(device='cpu').manual_seed(5)
    T = 12
    acts = torch.randint(0, 6, (T, N, 2), dtype=torch.uint8, generator=gen)
    bad = acts.clone()
    where = torch.rand((T, N, 2), generator=gen) < 0.05
    bad[where] = torch.randint(6, 256, (int(where.sum()),), dtype=torch.int64, generator=gen).to(torch.uint8)
    clean = acts.clone()
    clean[where] = 2
    for prec, flags, fused in ((32, 0, False), (32, 0, True), (32, nat.TICK_GENERIC_KERNEL, False), (64, 0, False)):
        outs = []
        for a in (bad, clean):
            g = _games(cfg, N, bullet_cap=K, precision=prec, seed=1)
            g.tick_flags = flags
            g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
            g.reset_all()
            ev = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
            if fused:
                g.step_many(T, a.cuda(), events=ev, auto_reset=True)
            else:
                for k in range(T):
                    ev[k] = g.step(a[k].cuda(), auto_reset=True)[2]
            outs.append((g.get_arrays(), ev.cpu().numpy(), g.stats()))
        (a0, e0, s0), (a1, e1, s1) = outs
        flagged = where.any(-1).numpy()
        assert ((e0 & nat.EV_BAD_CONTROL) != 0)[flagged].all() and not ((e0 & nat.EV_BAD_CONTROL) != 0)[~flagged].any()
        assert ((e0 & (255 ^ nat.EV_BAD_CONTROL)) == e1).all() and s0['bad_controls'] == int(flagged.sum()) and s1['bad_controls'] == 0
        assert H.same_bits(a0['ships'], a1['ships']) and (a0['n_bullets'] == a1['n_bullets']).all()
    with pytest.raises(ValueError):
        core.step(core.create(cfg), np.array([6, 0]), cfg)
    g = _games(cfg, 64, bullet_cap=K, precision=32)
    with pytest.raises(ValueError):
        g.step(np.full((64, 2), 7))


def test_bearings_beyond_the_sincos_range_are_rejected():
    """util.direction is reproduced for |b| <= 71476 (numpy switches to another reduction beyond): a config whose
    bearings could get there is refused when the schedule is set, and so are states that already are."""
    cfg = core.DEFAULT_CONFIG._replace(ship_rspeed=4000.0, max_time=40.0)      # 2000 ticks x 80 rad
    with pytest.raises(nat.AstroError, match='util.direction'):
        _games(cfg, 32, bullet_cap=32, precision=32)
    g = _games(core.DEFAULT_CONFIG, 32, bullet_cap=32, precision=32)
    pool = H.make_pool(core.DEFAULT_CONFIG, 32)
    ships = pool['ships'].copy()
    ships[3, 1, 4] = 1.0e5
    with pytest.raises(ValueError, match='util.direction'):
        g.set_arrays(ships, pool['planets'], pool['np'])
    s = core.create(core.DEFAULT_CONFIG)
    s = s._replace(ships=s.ships._replace(b=np.array([0.0, -8.0e4])))
    with pytest.raises(nat.AstroError, match='util.direction'):
        core.step(s, np.array([2, 2]), core.DEFAULT_CONFIG)


def test_explore_process_matches_the_reference_statistics():
    """rl.EpsilonGreedy run by the reference itself (tests/golden/explore.json: 400k calls per setting) against the
    device process on another random stream: enter / leave rates, active fraction, control histogram (never 5)."""
    import torch
    gold = json.load(open(os.path.join(H.G, 'explore.json')))
    cfg, N, T = core.DEFAULT_CONFIG._replace(max_time=1000.0), 4096, 120
    pool = H.make_pool(cfg, 64)
    for e in gold:
        g = _games(cfg, N, bullet_cap=32, precision=32, seed=2)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        state = torch.zeros((g.n_pad, 2), dtype=torch.int32, device='cuda')
        idle = active = entered = left = 0
        hist = np.zeros(6, dtype=np.int64)
        prev = np.zeros((N, 2), dtype=np.int64)
        tick_prev = None
        for k in range(T):
            acts = torch.full((g.n_pad, 2), 2, dtype=torch.uint8, device='cuda')
            tick = (g.meta.cpu().numpy().view(np.uint32)[:N] >> 14).astype(np.int64)
            g.explore_controls(acts, state, t_in=e['t_in'], t_out=e['t_out'], seed=11)
            now = (state.cpu().numpy()[:N] & 0xff).astype(np.int64)
            same = (tick > 0)[:, None] if k else np.zeros((N, 1), dtype=bool)    # (a re-created game's first call never switches)
            idle += int(((prev == 0) & same).sum()); entered += int(((prev == 0) & (now > 0) & same).sum())
            active += int(((prev > 0) & same).sum()); left += int(((prev > 0) & (now == 0) & same).sum())
            hist += np.bincount((now[now > 0] - 1).ravel(), minlength=6)
            prev = now
            g.step(torch.full((g.n_pad, 2), 2, dtype=torch.uint8, device='cuda'), auto_reset=True)
        ref_in, ref_out = e['entered'] / e['idle_calls'], e['left'] / e['active_calls']
        assert abs(entered / idle - ref_in) < 0.08 * ref_in and abs(left / active - ref_out) < 0.05 * ref_out, (entered / idle, ref_in, left / active, ref_out)
        assert hist[5] == 0 and e['hist'][5] == 0
        ref_h = np.array(e['hist'][:5]) / sum(e['hist'])
        assert np.abs(hist[:5] / hist.sum() - ref_h).max() < 0.02


def test_packed_controls_and_event_planes_equal_the_byte_forms(monkeypatch):
    """One control byte per game (ship 0 bits 0-2, ship 1 bits 3-5) and three event bit planes per tick instead of
    2 + 1 bytes per game: astro_tick_many, astro_rollout_host and astro_tick_host (whole, and cut into slices of tiles
    whose copies overlap the other slices' kernels) give the same events and leave the same state, in both builds."""
    import torch
    cfg, N, K, T = core.DEFAULT_CONFIG, 4096 + 64, 32, 40
    pool = H.make_pool(cfg, 256)
    gen = torch.Generator(device='cpu').manual_seed(21)

    def fresh(prec):
        g = _games(cfg, N, bullet_cap=K, precision=prec, seed=4)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        for _ in range(30):
            g.step(None, auto_reset=True)
        g.stats(clear=True)
        return g

    for prec in (32, 64):
        base = fresh(prec)
        acts = torch.randint(0, 6, (T, base.n_pad, 2), dtype=torch.uint8, generator=gen)
        packed = base.pack_controls(acts)
        assert packed.shape == (T, base.n_pad) and packed.dtype == torch.uint8
        ev_ref = torch.zeros((T, base.n_pad), dtype=torch.uint8, device='cuda')
        base.step_many(T, acts.cuda(), events=ev_ref, auto_reset=True)
        want_ev = ev_ref.cpu().numpy()[:, :N] & 7
        want = (base.get_arrays(), base.stats())
        runs = {}
        # device buffers, several ticks per launch
        g = fresh(prec)
        planes = torch.zeros(g.planes_shape(T), dtype=torch.int32, device='cuda')
        g.step_many(T, packed.cuda(), events=planes, auto_reset=True, packed=True, planes=True)
        runs['tick_many'] = (g, g.unpack_event_planes(planes))
        # host buffers, pipelined
        g = fresh(prec)
        planes_h = torch.zeros(g.planes_shape(T), dtype=torch.int32).pin_memory()
        g.rollout_host(packed.pin_memory(), planes_h, auto_reset=True, packed=True, planes=True)
        runs['rollout_host'] = (g, g.unpack_event_planes(planes_h))
        # host buffers, tick by tick: unsliced and sliced
        for slices in (1, 3):
            monkeypatch.setenv('ASTRO_HOST_SLICES', str(slices))
            g = fresh(prec)
            out = np.zeros((T, N), dtype=np.uint8)
            pk, pl = packed.pin_memory(), torch.zeros(g.planes_shape(), dtype=torch.int32).pin_memory()
            for k in range(T):
                g.step_host(pk[k], pl, auto_reset=True, packed=True, planes=True)
                out[k] = g.unpack_event_planes(pl)
            runs['step_host/%d' % slices] = (g, out)
            # ... and the byte forms through the sliced path
            g = fresh(prec)
            out = np.zeros((T, N), dtype=np.uint8)
            ah, eh = acts.pin_memory(), torch.zeros(g.n_pad, dtype=torch.uint8).pin_memory()
            for k in range(T):
                g.step_host(ah[k], eh, auto_reset=True)
                out[k] = eh.numpy()[:N] & 7
            runs['step_host bytes/%d' % slices] = (g, out)
        monkeypatch.delenv('ASTRO_HOST_SLICES')
        # begin / end on a stream of its own
        g = fresh(prec)
        out = np.zeros((T, N), dtype=np.uint8)
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        pk, pl = packed.pin_memory(), torch.zeros(g.planes_shape(), dtype=torch.int32).pin_memory()
        for k in range(T):
            g.step_host_begin(pk[k], pl, auto_reset=True, packed=True, planes=True, stream=st)
            g.step_host_end()
            out[k] = g.unpack_event_planes(pl)
        st.synchronize()
        runs['begin/end'] = (g, out)
        with pytest.raises(nat.AstroError):
            g.step_host_end()
        for name, (g, ev) in runs.items():
            assert (ev == want_ev).all(), (prec, name)
            arr = g.get_arrays()
            assert g.stats() == want[1], (prec, name)
            for key in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'episode'):
                assert (arr[key] == want[0][key]).all(), (prec, name, key)
        assert want[1]['episodes'] > 300 and (want_ev == 4).sum() == 0 and ((want_ev & 3) != 0).sum() == want[1]['episodes']


# ------------------------------------------------------------------ fresh games without a pool

def _created_rows(cfg, seeds):
    """core.create for every seed as float32-rounded game-major rows (what a float32 batch holds after a re-creation)."""
    S = 1 if cfg.solo else 2
    ships = np.zeros((len(seeds), S, 5))
    planets = np.zeros((len(seeds), 4, 4))
    npl = np.zeros(len(seeds), dtype=np.int64)
    for i, sd in enumerate(seeds):
        s = core.create(cfg._replace(seed=int(sd)))
        ships[i, :, 0:2], ships[i, :, 2:4], ships[i, :, 4] = s.ships.x, s.ships.dx, s.ships.b
        p = s.planets.x.shape[0]
        planets[i, :p, 0:2], planets[i, :p, 2:4] = s.planets.x, s.planets.dx
        npl[i] = p
    return ships.astype(np.float32).astype(np.float64), planets.astype(np.float32).astype(np.float64), npl


@pytest.mark.parametrize('N,quota,skip', [(2048, 8, 0), (300, 1, 1000)])
def test_fresh_games_every_recreation_takes_the_next_unused_config(N, quota, skip):
    """Fresh-game mode, one launch per tick, teacher-forced against the oracle: every game that ends is re-created from a
    position of the generate_configs stream that no game has had before, the new state equals core.create(seed at that
    position) bit for bit (float32-rounded), and the books balance: positions handed out = ring + initial fill + records
    re-created.  A small quota makes tiles run dry between refills: those games wait (ASTRO_EV_AWAIT) and come back."""
    cfg, K, S = core.DEFAULT_CONFIG, 32, 2
    games = _games(cfg, N, bullet_cap=K, precision=32, seed=3)
    games.enable_fresh_games(quota=quota, skip=skip)
    games.reset_all()
    n_tiles = games.n_tiles
    seeds_of = lambda pos: rng.config_seeds(cfg.seed, int(pos.max()) + 1 - skip, skip)[pos - skip]
    pos, used, cursor = games.fresh_positions()
    assert cursor == skip + n_tiles * quota + games.n_pad and (used == 0).all()
    assert (np.sort(pos) == skip + n_tiles * quota + np.arange(N)).all()
    arr = games.get_arrays()
    ships, planets, npl = _created_rows(cfg, seeds_of(pos))
    assert (arr['ships'] == ships).all() and (arr['n_planets'] == npl).all() and (arr['planets'] == planets).all()
    seen = set(pos.tolist())
    ids = np.arange(N)
    T, n_recreated, n_await = 260, 0, 0
    for k in range(T):
        ob, alive = H.oracle_batch_from(arr, S, K)
        ob.reload[:] = games.schedule.reload[np.minimum(arr['tick'], games.schedule.n_ticks - 1)]
        ob.t[:] = games.schedule.t[np.minimum(arr['tick'], games.schedule.n_ticks - 1)]
        o2, rew, done, ev = ao.step_batch(cfg, ob, rng.actions(3, ids, k, S), alive)
        _, d_gpu, e_gpu = games.step(None, auto_reset=True)
        e_gpu = e_gpu.cpu().numpy()
        waiting = arr['finished']                                   # games that were waiting for a record before this tick
        assert ((e_gpu & 15) == (ev & 15))[~waiting].all(), k
        new = games.get_arrays()
        new_pos, used, cursor = games.fresh_positions()
        ended = (done != 0) & ~waiting
        took = new_pos != pos                                          # games that got a fresh record this tick
        await_now = (e_gpu & nat.EV_AWAIT) != 0
        assert (took | await_now)[ended].all() and not (took & ~(ended | waiting)).any(), k
        assert (new['finished'] == ((ended | waiting) & ~took)).all(), k
        if took.any():
            fresh = new_pos[took]
            assert len(set(fresh.tolist())) == fresh.size and not (set(fresh.tolist()) & seen), k
            seen |= set(fresh.tolist())
            ships, planets, npl = _created_rows(cfg, seeds_of(fresh))
            assert (new['ships'][took] == ships).all() and (new['planets'][took] == planets).all(), k
            assert (new['n_planets'][took] == npl).all() and (new['n_bullets'][took] == 0).all() and (new['tick'][took] == 0).all()
        live = ~(ended | waiting)
        assert (new['n_bullets'][live] == o2.nb[live]).all() and _close(new['ships'][live], o2.ships[live]).all(), k
        n_recreated += int(took.sum())
        n_await += int(await_now.sum())
        arr, pos = new, new_pos
    st = games.stats()
    assert st['awaiting'] == n_await and st['episodes'] == n_recreated + int(arr['finished'].sum())
    # the books: every position handed out is either in a ring (unused), or was taken by exactly one game
    assert cursor - skip == n_tiles * quota + games.n_pad + n_recreated - int(used.sum())
    assert len(seen) == N + n_recreated and max(seen) < cursor
    if quota == 1:
        assert n_await > 0          # tiles did run dry — and every waiting game came back or is still waiting, never re-used
    assert n_recreated > N // 2


def test_fresh_games_fused_launches_1M_no_repeats():
    """BASELINE-size check (1,048,576 games x 600 ticks, 20 ticks per launch, quota 48): no two live games ever share a
    stream position, positions only grow, and positions handed out = ring + initial fill + games re-created (+ records
    re-created but not yet used) — every re-creation consumed a config of the generate_configs stream exactly once."""
    import torch
    cfg, N, quota = core.DEFAULT_CONFIG, 1 << 20, 48
    games = _games(cfg, N, bullet_cap=32, precision=32, seed=0)
    games.enable_fresh_games(quota=quota)
    games.reset_all()
    pos0, _, cur0 = games.fresh_positions()
    prev = pos0
    taken = np.zeros(40 * N, dtype=bool)                                  # stream positions some game has had
    taken[pos0] = True
    for launch in range(30):
        games.step_many(20, None, auto_reset=True)
        pos, used, cursor = games.fresh_positions()
        assert np.unique(pos).size == N                                   # no two live games share a start state
        changed = pos != prev
        assert not taken[pos[changed]].any()                              # ... nor does a game get one that was had before
        taken[pos[changed]] = True
        prev = pos
    st = games.stats()
    assert st['awaiting'] == 0 and st['env_steps'] == N * 600
    # positions handed out: the ring, the initial fill, and one per record re-created; records re-created = records used
    # up to the last refill = episodes - records used since
    assert cursor == games.n_tiles * quota + N + st['episodes'] - int(used.sum())
    assert st['episodes'] > 5 * N
    # spot-check: the current state of games still on their tick 0 equals core.create of their position's seed
    arr = games.get_arrays(np.arange(0, N, 4099))
    p_s = pos[::4099]
    fresh = arr['tick'] == 0
    if fresh.any():
        seeds = rng.config_seeds(cfg.seed, int(p_s.max()) + 1, 0)[p_s[fresh]]
        ships, planets, npl = _created_rows(cfg, seeds)
        assert (arr['ships'][fresh] == ships).all() and (arr['n_planets'][fresh] == npl).all()


@pytest.mark.parametrize('window', [964, 50, 7, 1])
def test_nstep_experiences_match_the_reference_ingestion(window):
    """astro_nstep_experiences against rl.QBotTrainer.reward run by the reference itself (tests/golden/nstep.json: one bot
    slot per ship over ten recorded games back to back): every Experience the reference appended — which tick's state,
    the discounted reward, the discount, the new state's tick or None — comes out once, whatever the window the log is
    cut into (pairs still held at a window's end are carried into the next)."""
    import torch
    gold = json.load(open(os.path.join(H.G, 'nstep.json')))
    ticks = gold['ticks']
    T = len(ticks)
    ev = np.full((T, 32), nat.EV_SKIPPED, dtype=np.uint8)
    for t, (action, reward, terminal) in enumerate(ticks):
        e = 0
        if terminal:
            e = (1 if reward[0] < 0 else 0) | (2 if reward[1] < 0 else 0)
            e = e or nat.EV_TIMEOUT
        ev[t, 0] = e
    games = _games(core.DEFAULT_CONFIG, 32, bullet_cap=32, precision=32)
    ev_dev = torch.from_numpy(ev).cuda()
    for setting in gold['settings']:
        n_steps, discount = setting['n_steps'], setting['discount']
        got = [dict(), dict()]
        carry = None
        for t0 in range(0, T, window):
            chunk = ev_dev[t0:t0 + window].contiguous()
            rew, dis, nxt, carry = games.nstep_experiences(chunk, carry, n_steps=n_steps, discount=discount)
            rew, dis, nxt = rew.cpu().numpy()[:, 0], dis.cpu().numpy()[:, 0], nxt.cpu().numpy()[:, 0]
            for row in range(nxt.shape[0]):
                for me in range(2):
                    if nxt[row, me] >= -1:
                        tick = t0 + row - n_steps
                        assert tick >= 0 and tick not in got[me]
                        got[me][tick] = (float(rew[row, me]), float(dis[row, me]), -1 if nxt[row, me] < 0 else t0 + int(nxt[row, me]))
            assert (carry.cpu().numpy()[1:] == 0).all()
        for me in range(2):
            want = setting['experiences'][me]
            assert want[-1][0] == 'held' and int(carry[0, me]) == want[-1][1]
            assert len(got[me]) == len(want) - 1
            for tick, action, reward, disc, new in want[:-1]:
                r, d, n = got[me][tick]
                assert n == new and abs(r - reward) <= 1e-6 * max(1.0, abs(reward)) and abs(d - disc) <= 1e-6 * disc, (n_steps, tick)
                assert action == ticks[tick][0][me]


# ------------------------------------------------------------------ the statistics reduction over peer memory

def test_stats_allreduce_single_rank_equals_stats():
    """astro_stats_allreduce with a world of one rank (the exchange buffer is the rank's own): the kernel's local
    gather, row store, wait and sum give exactly astro_stats, with and without clearing."""
    import ctypes as C
    import torch
    cfg, N = core.DEFAULT_CONFIG, 2048
    games = _games(cfg, N, bullet_cap=32, precision=32, seed=2)
    games.set_reset_pool_on_device(128)
    games.reset_all()
    L = nat.lib()
    handle = (C.c_uint8 * 64)()
    out = torch.zeros(nat.N_STATS, dtype=torch.int64, device='cuda')
    assert L.astro_stats_allreduce(games._h, out.data_ptr(), 0, None) == -3          # before create / open: state error
    assert L.astro_stats_peer_open(games._h, bytes(64)) == -3
    assert L.astro_stats_peer_create(games._h, 3, 2, handle) == -1                   # rank out of range
    nat.check(L.astro_stats_peer_create(games._h, 0, 1, handle))
    assert L.astro_stats_peer_create(games._h, 0, 1, handle) == -3                   # twice
    nat.check(L.astro_stats_peer_open(games._h, bytes(handle)))
    for k in range(3):
        games.step_many(24, None, auto_reset=True)
        games.step(None, auto_reset=True)                                            # (slot rows: folded on the way)
        want = games.stats_tensor(clear=False).clone()
        nat.check(L.astro_stats_allreduce(games._h, out.data_ptr(), int(k == 1), None))
        assert (out == want).all() and int(want[nat.STAT_NAMES.index('env_steps')]) > 0
        if k == 1:
            assert games.stats()['env_steps'] == 0


def test_stats_allreduce_over_peer_memory_equals_nccl(tmp_path):
    """Two ranks (two GPUs of one box) through torch.distributed.run: astro_stats_allreduce == the NCCL all-reduce of the
    same counters, six rounds with the ranks arriving at different times, alternating clear."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'peer_worker.py')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2', '--master-addr', '127.0.0.1',
                        '--master-port', '29655', script], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600,
                       env=dict(os.environ, ASTRO_PEER_OUT=str(tmp_path)))
    assert r.returncode == 0, r.stdout[-3000:]
    res = [json.load(open(os.path.join(str(tmp_path), 'rank%d.json' % k))) for k in range(2)]
    for x in res:
        assert x['ok'], x
        assert len(x['rounds']) == 7 and all(x['rounds']), x


# ------------------------------------------------------------------ the network on a feature batch (astro_value_forward)

@pytest.mark.parametrize('solo', [False, True])
def test_value_forward_kernel_matches_the_torch_network(solo):
    """rl.ValueNetwork.forward on cuda float32 feature batches under no_grad = value_forward_kernel: within 2e-6 of the
    layer-by-layer PyTorch forward (the reference's, rl.py:140-165) on real observations (both perspectives, -1 padding),
    on ragged shapes (item counts off the 16-item groups, row counts off the 8-row chunks), on batches whose masked rows
    hold arbitrary values or that have no live row at all (masked_max's x - 1e9 * pad arithmetic, rl.py:115-128), and
    with autograd on it falls back to PyTorch (gradients flow)."""
    import torch
    from astro_b200 import rl
    cfg = core.SOLO_CONFIG if solo else core.DEFAULT_CONFIG
    S, D = (1, 10) if solo else (2, 15)
    torch.manual_seed(3)
    net = rl.ValueNetwork(solo=solo, nout=6).cuda()
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(2.0)
    games = _games(cfg, 4096, bullet_cap=32, precision=32, seed=4)
    games.set_reset_pool_on_device(256)
    games.reset_all()
    games.step_many(200, None, auto_reset=True)
    obs = games.observe()                                     # [n, S, 36, D]
    with torch.no_grad():
        want = net.forward_torch(obs)
        got = net(obs)
        assert got.shape == want.shape and float((got - want).abs().max()) <= 2e-6
        # ragged: 37 items (two groups and a bit), 13 rows; a single item; rows < 8
        for n_items, rows in ((37, 13), (1, 36), (16, 5), (33, 8)):
            x = obs[:n_items, 0, :rows].contiguous()
            assert float((net(x) - net.forward_torch(x)).abs().max()) <= 2e-6, (n_items, rows)
        # masked rows with arbitrary contents, live rows anywhere (not a prefix), items without a live row
        g = torch.Generator(device='cuda').manual_seed(5)
        x = torch.randn((101, 19, D), device='cuda', generator=g)
        x[..., 0] = (torch.rand((101, 19), device='cuda', generator=g) < 0.4).float() * 2 - 1     # flag +1 live / -1 masked
        x[7, :, 0] = -1.0
        x[64, :, 0] = -1.0
        w, gt = net.forward_torch(x), net(x)
        assert float((gt - w).abs().max()) <= 2e-6
        # the parameters change: the next call uploads them again
        for prm in net.parameters():
            prm.mul_(0.5)
        assert float((net(obs) - net.forward_torch(obs)).abs().max()) <= 2e-6
    # with autograd the PyTorch path runs
    q = net(obs[:8])
    q.sum().backward()
    assert net.f0.weight.grad is not None and float(net.f0.weight.grad.abs().sum()) > 0


def test_value_forward_abi_errors():
    import torch
    games = _games(core.DEFAULT_CONFIG, 64, bullet_cap=32, precision=32)
    L = nat.lib()
    x = torch.zeros((4, 8, 15), device='cuda')
    q = torch.zeros((4, 6), device='cuda')
    assert L.astro_value_forward(games._h, x.data_ptr(), 4, 8, q.data_ptr(), None) == -3      # no weights yet
    from astro_b200 import rl
    games.set_policy(rl.ValueNetwork(solo=False, nout=6))
    assert L.astro_value_forward(games._h, None, 4, 8, q.data_ptr(), None) == -1
    assert L.astro_value_forward(games._h, x.data_ptr(), 4, 0, q.data_ptr(), None) == -1
    assert L.astro_value_forward(games._h, x.data_ptr(), 0, 8, q.data_ptr(), None) == 0
    with pytest.raises(ValueError):
        games.value_forward(torch.zeros((4, 8, 10), device='cuda'))
