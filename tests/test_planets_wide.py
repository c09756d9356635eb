"""Games of up to eight planets: the 8-slot batch layout (AstroConfig.planet_slots = 8) from the kernels to core.step.

The reference plays any number of planets (core.py:86-135 draws 1..max_planets, _gravity / _collisions / _update_bodies
are written for any count); its recorded games (tests/golden) all have at most four, so they pin the 8-slot kernels
through replays in an 8-slot batch, and games of five to eight planets are checked against the oracle's per-game
entry points, which take the planet count as an argument."""
import json
import os

import numpy as np
import pytest

from astro_b200 import core, rng
from astro_b200 import _native as nat
from astro_b200 import batched
from astro_b200.pool import make_pool
from oracle import astro_oracle as ao
from tests import helpers as H

TOL = 1e-5
WIDE = nat.MAX_PLANETS_WIDE
CFG8 = core.DEFAULT_CONFIG._replace(max_planets=8, seed=3)


def _games(*a, **k):
    return batched.BatchedGames(*a, **k)


def _close(got, ref):
    return np.abs(got - ref) <= TOL * np.maximum(1.0, np.abs(ref))


# ------------------------------------------------------------------ without a GPU

def test_planet_slots_follow_max_planets_and_name_the_limit():
    assert batched.planet_slots_for(core.DEFAULT_CONFIG) == 4
    assert batched.planet_slots_for(core.DEFAULT_CONFIG._replace(max_planets=1)) == 4
    for mp in (5, 6, 7, 8):
        assert batched.planet_slots_for(core.DEFAULT_CONFIG._replace(max_planets=mp)) == 8
    with pytest.raises(ValueError, match='at most 8 planets'):
        batched.planet_slots_for(core.DEFAULT_CONFIG._replace(max_planets=9))
    assert make_pool(core.DEFAULT_CONFIG, 3)['planets'].shape == (3, 4, 4)
    assert make_pool(CFG8, 3)['planets'].shape == (3, 8, 4)


def test_abi5_structs():
    import ctypes as C
    assert nat.ABI_VERSION == 5 and nat.MAX_PLANETS == 4 and nat.MAX_PLANETS_WIDE == 8
    assert [f[0] for f in nat.AstroConfig._fields_][-1] == 'planet_slots'
    assert nat.AstroSingleGame.planets.offset == 80 and C.sizeof(nat.AstroSingleGame) == 80 + 8 * 32 + 16 + 4 + 4 + 64 + 32


# ------------------------------------------------------------------ 1. the golden replays in an 8-slot batch

@pytest.mark.gpu
def test_golden_trajectories_f64_in_wide_batch():
    """The reference's recorded games replayed free-running in an 8-slot float64 batch: every state bit for bit."""
    import collections
    z, meta = H.load_traj()
    groups = collections.defaultdict(list)
    for m in meta:
        groups[tuple(sorted((k, v) for k, v in m['config'].items() if k != 'seed'))].append(m)
    checked = 0
    for _, ms in groups.items():
        cfg = H.config_from(ms[0]['config'])
        S, n = ms[0]['nships'], len(ms)
        games = _games(cfg, n, bullet_cap=32, precision=64, planet_slots=WIDE)
        assert tuple(games.planets.shape[1:]) == (WIDE, 32, 4)
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
                assert games.schedule.t[arr['tick'][i]] == z['g%d_t' % g][k]
                ctl[i] = z['g%d_control' % g][k]
                checked += 1
            reward, done, _ = games.step(ctl)
            reward, done = reward.cpu().numpy(), done.cpu().numpy()
            for i, m in enumerate(ms):
                if k < m['nticks']:
                    assert H.same_bits(reward[i], z['g%d_reward' % m['game']][k]), (m['game'], k)
                    assert bool(done[i]) == (k == m['nticks'] - 1 and not m['truncated']), (m['game'], k)
    assert checked > 6000


@pytest.mark.gpu
def test_golden_trajectories_f32_in_wide_batch_teacher_forced():
    """The same games in an 8-slot float32 batch, teacher-forced from the golden state every tick: discrete outcomes
    exact, continuous state within the float32 tolerance."""
    z, meta = H.load_traj()
    checked = 0
    for m in meta:
        g, cfg = m['game'], H.config_from(m['config'])
        S = m['nships']
        games = _games(cfg, 1, bullet_cap=32, precision=32, planet_slots=WIDE)
        off = np.concatenate([[0], np.cumsum(z['g%d_nb' % g])])
        for k in range(0, m['nticks'] - 1, 3):
            bl = z['g%d_bullets' % g][off[k]:off[k + 1]]
            st = H.state_from_arrays(z['g%d_ships' % g][k], z['g%d_planets' % g][k], bl, z['g%d_reload' % g][k], z['g%d_t' % g][k])
            games.set_schedule_origin(st.reload, st.t)
            games.set_states([st], ticks=[0])
            reward, done, _ = games.step(np.asarray(z['g%d_control' % g][k], dtype=np.uint8).reshape(1, S))
            assert not bool(done[0].item()) and (reward[0].cpu().numpy() == z['g%d_reward' % g][k]).all(), (g, k)
            arr = games.get_arrays()
            B, P = int(z['g%d_nb' % g][k + 1]), m['nplanets']
            assert arr['n_bullets'][0] == B, (g, k)
            assert _close(arr['ships'][0], z['g%d_ships' % g][k + 1]).all(), (g, k)
            assert _close(arr['planets'][0, :P], z['g%d_planets' % g][k + 1]).all(), (g, k)
            assert _close(arr['bullets'][0, :B], z['g%d_bullets' % g][off[k + 1]:off[k + 2]]).all(), (g, k)
            checked += 1
    assert checked > 1500


def _force_wide(monkeypatch):
    orig = core._single_game
    monkeypatch.setattr(core, '_single_game', lambda config, n_bullets, n_planets: orig(config, n_bullets, WIDE))


@pytest.mark.gpu
def test_golden_edges_and_raw_create_through_core_step_in_wide_handle(monkeypatch):
    """core.step through an 8-slot single-game handle: the 70 knife-edge cases and the reference's games played from
    create()'s raw float32 arrays, bit for bit."""
    _force_wide(monkeypatch)
    z = np.load(os.path.join(H.G, 'edges.npz'))
    for c in json.load(open(os.path.join(H.G, 'edges.json'))):
        i, cfg = c['case'], H.config_from(c['config'])
        state = H.state_from_arrays(z['c%d_ships' % i], z['c%d_planets' % i], z['c%d_bullets' % i], c['reload'], c['t'])
        nxt, reward = core.step(state, np.array(c['control']), cfg)
        assert (nxt is None) == c['done'] and H.same_bits(reward, c['reward']), c['name']
        if nxt is not None:
            o = z['c%d_o_planets' % i]
            assert H.same_bits(nxt.planets.x, o[:, 0:2]) and H.same_bits(nxt.planets.dx, o[:, 2:4]), c['name']
            o = z['c%d_o_bullets' % i].reshape(-1, 4)
            assert H.same_bits(nxt.bullets.x, o[:, 0:2]) and H.same_bits(nxt.bullets.dx, o[:, 2:4]), c['name']
            o = z['c%d_o_ships' % i]
            assert H.same_bits(nxt.ships.x, o[:, 0:2]) and H.same_bits(nxt.ships.b, o[:, 4]), c['name']
    z = np.load(os.path.join(H.G, 'traj_raw.npz'))
    total = 0
    for m in json.load(open(os.path.join(H.G, 'traj_raw.json'))):
        g, cfg = m['game'], H.config_from(m['config'])
        ships, planets = z['g%d_ships' % g], z['g%d_planets' % g]
        state = core.create(cfg)
        for k in range(min(m['nticks'], 60)):
            assert H.same_bits(np.concatenate([state.ships.x, state.ships.dx, np.asarray(state.ships.b)[:, None]], 1), ships[k]), (g, k)
            assert H.same_bits(np.concatenate([state.planets.x, state.planets.dx], 1), planets[k]), (g, k)
            state, reward = core.step(state, z['g%d_control' % g][k], cfg)
            assert (np.asarray(reward, dtype=np.float64) == z['g%d_reward' % g][k]).all()
            total += 1
            if state is None:
                break
    assert total > 600


# ------------------------------------------------------------------ 2. five to eight planets against the oracle

def _wide_batch(N, K, precision, pool_size=512, seed=0, cfg=CFG8):
    games = _games(cfg, N, bullet_cap=K, precision=precision, seed=seed)
    assert games.PL == WIDE
    games.set_reset_pool_on_device(pool_size)
    games.reset_all()
    return games


def _oracle_step_all(cfg, games, arr, ctl):
    """oracle.step_one for every live game of get_arrays() `arr` -> list of result dicts (None for finished games)."""
    out = []
    for i in range(arr['ships'].shape[0]):
        if arr['finished'][i]:
            out.append(None)
            continue
        P, B, tk = int(arr['n_planets'][i]), int(arr['n_bullets'][i]), int(arr['tick'][i])
        out.append(ao.step_one(cfg, arr['ships'][i], arr['planets'][i, :P], arr['bullets'][i, :B],
                               games.schedule.reload[tk], games.schedule.t[tk], ctl[i], bullet_cap=games.K))
    return out


def _teacher_forced_wide(precision, N, K, ticks, start=None, seed=0):
    cfg = CFG8
    games = _wide_batch(N, K, precision, seed=seed)
    if start is not None:
        start(games)
    S = 2
    ids = np.arange(N)
    arr = games.get_arrays()
    assert arr['n_planets'].max() == 8 and arr['n_planets'].min() == 1
    n_done = 0
    for k in range(ticks):
        ctl = rng.actions(seed, ids, k, S)
        ref = _oracle_step_all(cfg, games, arr, ctl)
        r_gpu, d_gpu, e_gpu = (t.cpu().numpy() for t in games.step(None, auto_reset=True))
        new = games.get_arrays()
        for i, o in enumerate(ref):
            assert o is not None
            assert int(e_gpu[i]) == o['events'] and bool(d_gpu[i]) == o['done'], (k, i)
            assert (r_gpu[i].astype(np.float64) == o['reward']).all(), (k, i)
            if o['done']:
                n_done += 1
                assert new['tick'][i] == 0 and new['n_bullets'][i] == 0 and new['episode'][i] == arr['episode'][i] + 1
                continue
            P, B = int(arr['n_planets'][i]), o['bullets'].shape[0]
            assert new['n_bullets'][i] == B and new['n_planets'][i] == P and new['tick'][i] == arr['tick'][i] + 1, (k, i)
            for got, want in ((new['ships'][i], o['ships']), (new['planets'][i, :P], o['planets']), (new['bullets'][i, :B], o['bullets'])):
                if precision == 64:
                    assert H.same_bits(got, want), (k, i)
                else:
                    assert _close(got, want).all(), (k, i, float(np.abs(got - want).max()))
        arr = new
    return games, n_done


@pytest.mark.gpu
@pytest.mark.parametrize('precision', [64, 32])
def test_five_to_eight_planets_teacher_forced_against_oracle(precision):
    """2,048 games of 1..8 planets, random controls, 200 ticks, auto-reset from a device-created pool; the oracle
    re-fed the device's state every tick: float64 bit for bit, float32 discrete outcomes exact and state within 1e-5."""
    games, n_done = _teacher_forced_wide(precision, 2048, 32, 200)
    st = games.stats()
    assert n_done > 1000 and st['episodes'] == n_done and st['planets_live'] > 3.5 * st['env_steps']


def _band_fill(K, seed):
    """Bullets parked at the collision radius (within a few ulp) of planet slots 4-7 of games with more than four
    planets, the rest random: the float32 band test and its float64 fallback run on the new slots."""
    def fill(games):
        r = np.random.RandomState(seed)
        arr = games.get_arrays()
        n = games.n
        bl = np.concatenate([r.uniform(-1.1, 1.1, (n, K, 2)), r.uniform(-1.0, 1.0, (n, K, 2))], axis=2)
        rp = games.config.planet_radius
        for i in range(n):
            P = int(arr['n_planets'][i])
            for j in range(K // 2):
                p = 4 + j % max(1, P - 4) if P > 4 else j % P
                ang = r.uniform(0, 2 * np.pi)
                rad = rp * (1.0 + r.choice([-1, 0, 1]) * r.randint(0, 4) * 2.0 ** -52)
                bl[i, j, 0:2] = arr['planets'][i, p, 0:2] + rad * np.array([np.sin(ang), np.cos(ang)])
                bl[i, j, 2:4] = 0.0
        nb = np.full(n, K)
        games.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], bl, nb, r.randint(0, 40, n))
    return fill


@pytest.mark.gpu
@pytest.mark.parametrize('precision', [64, 32])
def test_bullets_at_the_radius_of_planet_slots_4_to_7(precision):
    _teacher_forced_wide(precision, 512, 64, 3, start=_band_fill(64, 7))


# ------------------------------------------------------------------ 3. fused ticks == separate ticks

@pytest.mark.gpu
@pytest.mark.parametrize('per_launch', [1, 20, 64])
def test_fused_ticks_equal_separate_ticks_wide(per_launch):
    """astro_tick_many in an 8-slot batch against one launch per tick: events, rewards, the final state and the
    statistics bit for bit, through deaths and re-creations from the 256-byte pool records; the first launch starts
    from a fill with more than 224 bullets in some tiles (a second staging round)."""
    import torch
    N, K, T = 4096, 32, 128
    runs = []
    for fused in (False, True):
        g = _wide_batch(N, K, 32, seed=5)
        r = np.random.RandomState(3)
        arr = g.get_arrays()
        bl = np.concatenate([r.uniform(-0.9, 0.9, (N, K, 2)), r.uniform(-0.5, 0.5, (N, K, 2))], axis=2)
        nb = r.randint(0, 8, N)
        nb[:32] = K                     # tile 0: 1,024 bullets
        nb[32:64] = 9                   # tile 1: 288
        g.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], bl, nb, arr['tick'])
        g.stats(clear=True)
        gen = torch.Generator(device='cpu').manual_seed(11)
        acts = torch.randint(0, 6, (T, g.n_pad, 2), dtype=torch.uint8, generator=gen).cuda()
        ev = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
        rw = torch.zeros((T, g.n_pad, 2), dtype=torch.float32, device='cuda')
        if fused:
            for k0 in range(0, T, per_launch):
                n = min(per_launch, T - k0)
                g.step_many(n, acts[k0:k0 + n], events=ev[k0:k0 + n], reward=rw[k0:k0 + n], auto_reset=True)
        else:
            for k in range(T):
                r_, _, e_ = g.step(acts[k], auto_reset=True)
                ev[k], rw[k] = e_, r_
        runs.append((g.get_arrays(), ev.cpu().numpy(), rw.cpu().numpy(), g.stats()))
    (a0, e0, r0, s0), (a1, e1, r1, s1) = runs
    assert (e0 == e1).all() and (r0 == r1).all() and s0 == s1
    assert s0['episodes'] > 1000 and (a0['episode'] > 0).any()
    for k in ('n_bullets', 'n_planets', 'tick', 'episode', 'finished'):
        assert (a0[k] == a1[k]).all(), k
    pm = np.arange(WIDE)[None, :] < a0['n_planets'][:, None]
    bm = np.arange(K)[None, :] < a0['n_bullets'][:, None]
    assert H.same_bits(a0['ships'], a1['ships'])
    assert H.same_bits(a0['planets'][pm], a1['planets'][pm]) and H.same_bits(a0['bullets'][bm], a1['bullets'][bm])


# ------------------------------------------------------------------ 4. the drop-in core.play

@pytest.mark.gpu
def test_core_play_with_eight_planets_equals_oracle_loop():
    """core.step from raw create() arrays with max_planets = 8: a loop of oracle.step_one (raw on the first tick) bit
    for bit, with the reference's reward dtypes."""
    played = 0
    for seed in range(40):
        cfg = CFG8._replace(seed=seed)
        state = core.create(cfg)
        P = state.planets.x.shape[0]
        ref = dict(ships=np.concatenate([state.ships.x, state.ships.dx, state.ships.b[:, None]], 1).astype(np.float64),
                   planets=np.concatenate([state.planets.x, state.planets.dx], 1).astype(np.float64),
                   bullets=np.zeros((0, 4)), reload=state.reload, t=state.t)
        r = np.random.RandomState(seed)
        for k in range(120):
            ctl = r.randint(0, 6, 2)
            o = ao.step_one(cfg, ref['ships'], ref['planets'], ref['bullets'], ref['reload'], ref['t'], ctl, raw=(k == 0))
            state, reward = core.step(state, ctl, cfg)
            assert (state is None) == o['done'] and (np.asarray(reward, dtype=np.float64) == o['reward']).all(), (seed, k)
            if state is None:
                assert reward.dtype in (np.int64, np.float32)
                break
            assert reward.dtype == np.float32 and state.planets.x.shape[0] == P
            got = np.concatenate([state.ships.x, state.ships.dx, state.ships.b[:, None]], 1)
            assert H.same_bits(got, o['ships']) and H.same_bits(np.concatenate([state.planets.x, state.planets.dx], 1), o['planets'])
            assert H.same_bits(np.concatenate([state.bullets.x, state.bullets.dx], 1).reshape(-1, 4), o['bullets'])
            assert state.reload == o['reload'] and state.t == o['t']
            ref = o
            played += 1
    assert played > 1000
    game = core.play(CFG8._replace(seed=7, max_time=2.0), [_Idle(), _Idle()])   # (seed 7: eight planets)
    assert game.ticks and game.ticks[0].state.planets.x.shape[0] > 4


class _Idle(core.Bot):
    def __call__(self, state):
        return 2


# ------------------------------------------------------------------ 5. creation on the device

@pytest.mark.gpu
@pytest.mark.parametrize('max_planets', [5, 6, 7, 8])
def test_create_on_device_five_to_eight_planets(max_planets):
    cfg = core.DEFAULT_CONFIG._replace(max_planets=max_planets, seed=max_planets)
    M = 4096
    seeds = rng.config_seeds(cfg.seed, M)
    want = make_pool(cfg, M)
    assert want['np'].max() == max_planets
    for prec in (64, 32):
        games = _games(cfg, 64, bullet_cap=32, precision=prec)
        ships, planets, npl = (t.cpu().numpy().astype(np.float64) if t.dtype.is_floating_point else t.cpu().numpy()
                               for t in games.create_on_device(seeds))
        cast = (lambda a: a) if prec == 64 else (lambda a: a.astype(np.float32).astype(np.float64))
        assert (npl == want['np']).all()
        assert H.same_bits(ships, cast(want['ships'])) and H.same_bits(planets, cast(want['planets']))


# ------------------------------------------------------------------ 6. the other kernels on 8-planet states

def _played_wide(precision, N=2048, ticks=60, seed=1):
    games = _wide_batch(N, 32, precision, seed=seed)
    for _ in range(ticks):
        games.step(None, auto_reset=True)
    games.step(None, auto_reset=False)        # leaves a few finished games behind
    return games


@pytest.mark.gpu
@pytest.mark.parametrize('precision', [32, 64])
def test_observe_script_and_export_import_on_eight_planet_states(precision):
    games = _played_wide(precision)
    arr = games.get_arrays()
    assert arr['finished'].any() and (arr['n_planets'] > 4).mean() > 0.3
    obs = games.observe().cpu().numpy()
    shared = games.observe(shared=True).cpu().numpy()
    n_rows = obs.shape[2]
    assert n_rows >= WIDE + games.K
    ctl = games.script_controls()[:games.n].cpu().numpy()
    for g in range(games.n):
        if arr['finished'][g]:
            assert (obs[g] == -1).all() and (ctl[g] == 2).all()
            continue
        P, B = arr['n_planets'][g], arr['n_bullets'][g]
        for me in range(2):
            ref = ao.features(2, arr['ships'][g], arr['planets'][g, :P], arr['bullets'][g, :B], me, n_rows)
            assert (obs[g, me].view(np.uint32) == ref.view(np.uint32)).all(), (g, me)
            rolled = np.roll(arr['ships'][g], -me, 0)
            assert ctl[g, me] == ao.script_control(games.config, rolled, arr['planets'][g, :P], 0), (g, me)
        assert (shared[g].view(np.uint32) == obs[g, 0].view(np.uint32)).all(), g
    # export -> import round trip, into a second batch and back into scrambled slots of the same one
    other = _games(CFG8, games.n, bullet_cap=32, precision=precision, planet_slots=WIDE)
    t = games.export_arrays()
    other.set_arrays(*(t[k].cpu().numpy() for k in ('ships', 'planets', 'n_planets', 'bullets', 'n_bullets', 'tick')),
                     finished=t['finished'].cpu().numpy(), episode=t['episode'].cpu().numpy().view(np.uint32))
    b = other.get_arrays()
    for k in ('ships', 'planets', 'bullets', 'n_bullets', 'n_planets', 'tick', 'finished', 'episode'):
        assert (b[k] == arr[k]).all(), k
    perm = np.random.RandomState(2).permutation(games.n)
    live = ~arr['finished']
    games.set_arrays(arr['ships'][perm], arr['planets'][perm], arr['n_planets'][perm], arr['bullets'][perm],
                     np.where(live[perm], arr['n_bullets'][perm], 0), arr['tick'][perm])
    c = games.get_arrays()
    assert (c['n_planets'] == arr['n_planets'][perm]).all() and H.same_bits(c['planets'], arr['planets'][perm])


@pytest.mark.gpu
def test_policy_kernels_on_eight_planet_states():
    import torch
    from astro_b200 import rl
    games = _played_wide(32, N=4096 + 32, ticks=70, seed=4)
    torch.manual_seed(2)
    net = rl.ValueNetwork(solo=False, nout=6).to(games.device)
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(3.0)
        want = net.forward_torch(games.observe())
    games.set_policy(net)
    q = torch.empty((games.n_pad, 2, 6), dtype=torch.float32, device=games.device)
    act = games.policy_controls(q_out=q)
    fin = torch.from_numpy(games.get_arrays()['finished']).to(games.device)
    live = ~fin
    N = games.n
    assert fin.any()
    err = (q[:N][live] - want[live]).abs().max().item()
    assert err <= 2e-6, err
    top2 = want.topk(2, dim=-1).values
    clear = live.unsqueeze(-1) & ((top2[..., 0] - top2[..., 1]) > 1e-5)
    assert (act[:N].long()[clear] == want.argmax(-1)[clear]).all()


@pytest.mark.gpu
def test_rollout_device_script_bots_in_wide_batch_take_the_bot_kernel_loop():
    """astro_rollout_device with ScriptBots on an 8-slot batch: the bot-kernel -> tick loop, equal to stepping with
    script_controls() by hand."""
    runs = []
    for by_hand in (False, True):
        g = _wide_batch(1024, 32, 32, seed=9)
        if by_hand:
            for _ in range(40):
                g.step(g.script_controls(), auto_reset=True)
        else:
            g.rollout_device(40, bots=('script', 'script'), auto_reset=True)
        runs.append((g.get_arrays(), g.stats()))
    (a, sa), (b, sb) = runs
    assert sa == sb and H.same_bits(a['ships'], b['ships']) and (a['n_bullets'] == b['n_bullets']).all()


# ------------------------------------------------------------------ 7. the limits

@pytest.mark.gpu
def test_limits_are_reported():
    import ctypes as C
    with pytest.raises(ValueError, match='at most 8 planets'):
        _games(core.DEFAULT_CONFIG._replace(max_planets=9), 32)
    with pytest.raises(ValueError, match='1..8 planets'):
        core.step(core.State(ships=core.Bodies(np.zeros((2, 2)), np.zeros((2, 2)), np.zeros(2)),
                             planets=core.Bodies(np.zeros((9, 2)), np.zeros((9, 2)), None),
                             bullets=core.Bodies(np.zeros((0, 2)), np.zeros((0, 2)), None), reload=0.0, t=0.0),
                  np.array([2, 2]), core.DEFAULT_CONFIG)
    g = _games(CFG8, 64)
    with pytest.raises(nat.AstroError, match='fresh-game mode'):
        g.enable_fresh_games()
    L = nat.lib()
    cfg = nat.AstroConfig()
    cfg.planet_slots = 6
    h = C.c_void_p()
    assert L.astro_batch_create(C.byref(cfg), 32, 4, 32, 0, C.byref(h)) == -1 and b'planet_slots' in L.astro_last_error()
    with pytest.raises(ValueError, match='needs planet_slots=8'):
        _games(CFG8, 64, planet_slots=4)
