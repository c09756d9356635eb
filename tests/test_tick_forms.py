"""Every tick kernel instantiation the launchers can pick, each checked against the oracle or against its twin.

launch_tick_f32 / launch_tick_f32_wide / launch_tick (astro_b200.cu) choose the instantiation from the batch layout
and the call's options.  LEDGER below lists all 40 of them and the tests that launch each one; a CPU test holds the
ledger to the symbols of the built library, and every GPU test asserts, through torch.profiler, that it launched
exactly the tick forms it is about.

- The production forms, tick_f32_kernel<2, *, *, false, true> (FIX: packed controls, event planes, auto-reset from the
  pool), teacher-forced against the oracle one tick per launch, with every episode counter recomputed on the host; the
  fused form with its resident bullet pool against one launch per tick on bullets that sit in the float32 uncertainty
  band on every tick of a launch.
- Every statistics-off form against its statistics-on twin.
- Solo games with bullets in flight and parked around the ship."""
import os
import re

import numpy as np
import pytest

from astro_b200 import core, rng
from astro_b200 import _native as nat
from oracle import astro_oracle as ao
from tests import helpers as H

TOL = 1e-5
STAGE_ITEMS = 224                 # a tile's staging buffer in the launch of several ticks: the resident pool's limit
SOLO_BULLETS = core.SOLO_CONFIG._replace(reload_time=0.3)
WIDE_DUEL = core.DEFAULT_CONFIG._replace(max_planets=8, seed=3)
WIDE_SOLO = SOLO_BULLETS._replace(max_planets=8, seed=3)
# one volley every 100 ticks: the parked bullets and the bullets in flight fit a tile's staging buffer together
KNIFE_CFG = core.DEFAULT_CONFIG._replace(reload_time=2.0)


# ------------------------------------------------------------------ kernel names and the ledger

_FORM = re.compile(r'\b(tick_f32_wide_kernel|tick_f32_kernel|tick_kernel)<([^<>]*)>')


def form_of(name):
    """A tick kernel's name, as CUPTI writes it (`tick_f32_kernel<2, true, false, false, true>`) or as cu++filt does
    (`tick_f32_kernel<(int)2, (bool)1, ...>`), as a tuple: ('tick_f32_kernel', 2, 1, 0, 0, 1); tick_kernel keeps its
    element type: ('tick_kernel', 'float', 2, 1, 4).  None for any other kernel."""
    m = _FORM.search(name)
    if m is None:
        return None
    out = [m.group(1)]
    for a in m.group(2).split(','):
        a = re.sub(r'^\((?:int|bool)\)', '', a.strip())
        out.append({'true': 1, 'false': 0}.get(a, int(a) if a.isdigit() else a))
    return tuple(out)


def f32(S, stats, many, bot=0, fix=0):
    return ('tick_f32_kernel', S, stats, many, bot, fix)


def wide(S, stats, many):
    return ('tick_f32_wide_kernel', S, stats, many)


def generic(r, S, stats, PL):
    return ('tick_kernel', r, S, stats, PL)


def _ledger():
    led = {}

    def add(test, *forms):
        for f in forms:
            led.setdefault(f, []).append(test)
    twins = 'test_statistics_off_equals_statistics_on'
    for st in (0, 1):
        for S in (1, 2):
            add(twins, f32(S, st, 0), f32(S, st, 1), f32(S, st, 1, 1), wide(S, st, 0), wide(S, st, 1))
            for PL in (4, 8):
                add(twins, generic('float', S, st, PL), generic('double', S, st, PL))
        add(twins, f32(2, st, 0, 0, 1), f32(2, st, 1, 0, 1))
        add('test_fix_one_tick_teacher_forced', f32(2, st, 0, 0, 1))
        add('test_solo_one_tick_teacher_forced_with_bullets', f32(1, st, 0))
    add('test_golden_edges_through_the_one_tick_forms', f32(2, 1, 0, 0, 1), f32(1, 1, 0))
    for test in ('test_resident_pool_on_persistent_knife_edges', 'test_resident_pool_over_staging_rounds_and_back'):
        add(test, f32(2, 1, 1, 0, 1), f32(2, 1, 0, 0, 1))
    add('test_solo_forms_with_bullets_equal_one_launch_per_tick', f32(1, 1, 0), f32(1, 1, 1), f32(1, 1, 1, 1),
        wide(1, 1, 0), wide(1, 1, 1))
    return {f: tuple(t) for f, t in led.items()}


LEDGER = _ledger()


def _tick_forms_of_library():
    forms = [form_of(n) for n in H.library_kernel_names()]
    return [f for f in forms if f is not None]


def test_kernel_names_parse_in_both_spellings():
    assert form_of('void (anonymous namespace)::tick_f32_kernel<2, true, false, false, true>((anonymous namespace)::TickParams)') \
        == ('tick_f32_kernel', 2, 1, 0, 0, 1)
    assert form_of('void <unnamed>::tick_f32_kernel<(int)2, (bool)1, (bool)0, (bool)0, (bool)1>(<unnamed>::TickParams)') \
        == ('tick_f32_kernel', 2, 1, 0, 0, 1)
    assert form_of('void <unnamed>::tick_kernel<double, (int)1, (bool)0, (int)8>(<unnamed>::TickParams)') \
        == ('tick_kernel', 'double', 1, 0, 8)
    assert form_of('void (anonymous namespace)::tick_f32_wide_kernel<1, false, true>((anonymous namespace)::TickParams)') \
        == ('tick_f32_wide_kernel', 1, 0, 1)
    assert form_of('void (anonymous namespace)::observe_kernel<float, 2, 4>(int)') is None


def test_library_tick_forms_equal_the_ledger():
    """The built library's tick instantiations are exactly the ledger's keys, and every test the ledger names exists
    here: a form added to the library without a test that launches it fails here, with no GPU needed."""
    forms = _tick_forms_of_library()
    assert len(forms) == len(set(forms)) == 40
    assert set(forms) == set(LEDGER), (sorted(set(forms) - set(LEDGER)), sorted(set(LEDGER) - set(forms)))
    for form, tests in LEDGER.items():
        assert tests, form
        for t in tests:
            assert callable(globals().get(t)) and t.startswith('test_'), (form, t)


def _launched(fn):
    """Runs fn() under torch.profiler with CUDA activity; returns its result and the tick forms launched."""
    return H.launched(fn, form_of)


def _expect(forms, fn):
    """fn() must launch exactly the tick forms `forms`, each at least once, and each must be in the ledger under the
    calling test."""
    import inspect
    test = next(f.function for f in inspect.stack(0) if f.function.startswith('test_'))
    for f in forms:
        assert test in LEDGER[f], (test, f)
    result, got = _launched(fn)
    assert got == set(forms), (sorted(set(forms) - got), sorted(got - set(forms)))
    return result


# ------------------------------------------------------------------ batches, controls, the oracle checker

def _batch(cfg, N, K, seed=0, first_game=0, pool_size=256, precision=32, planet_slots=None, reset=True):
    from astro_b200.batched import BatchedGames
    g = BatchedGames(cfg, N, bullet_cap=K, precision=precision, seed=seed, first_game=first_game, planet_slots=planet_slots)
    pool = H.make_pool(cfg, pool_size, planet_slots)
    g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    if reset:
        g.reset_all()
    return g, pool


def _controls(n_pad, S, seed, bad=0.0, no_thrust=False):
    """controls(k) -> (what the tick is handed: packed bytes [n_pad] for duel games, else [n_pad, S] bytes; the codes
    the oracle flies [n_pad, S]; which games were handed a bad code [n_pad]).  `bad`: share of packed bytes with a
    3-bit field of 6 or 7, or with bits 6-7 set (ship 1's code 8 or more); the tick flies those ships with control 2."""
    r = np.random.RandomState(seed)

    def controls(k):
        c = 2 * r.randint(0, 3, (n_pad, S)) if no_thrust else r.randint(0, 6, (n_pad, S))
        if S == 1:
            return c.astype(np.uint8), c, np.zeros(n_pad, dtype=bool)
        byte = (c[:, 0] | (c[:, 1] << 3)).astype(np.int64)
        if bad:
            sel, kind, code = r.rand(n_pad) < bad, r.randint(0, 3, n_pad), r.randint(6, 8, n_pad)
            byte = np.where(sel & (kind == 0), (byte & 0xf8) | code, byte)
            byte = np.where(sel & (kind == 1), (byte & 0xc7) | (code << 3), byte)
            byte = np.where(sel & (kind == 2), byte | (r.randint(1, 4, n_pad) << 6), byte)
        c0, c1 = byte & 7, byte >> 3
        flown = np.stack([np.where(c0 > 5, 2, c0), np.where(c1 > 5, 2, c1)], axis=1)
        return byte.astype(np.uint8), flown, (c0 > 5) | (c1 > 5)
    return controls


def _expected_stats(S, arr, alive, ev, done, o2, bad, n_pad):
    """The 14 counters of one tick (warp_totals, astro_b200.cu) from the oracle's outputs."""
    a = alive
    h0, h1 = a & ((ev & nat.EV_HIT0) != 0), a & ((ev & nat.EV_HIT1) != 0)
    coll, ended = h0 | h1, a & (done != 0)
    v = dict.fromkeys(nat.STAT_NAMES, 0)
    v['episodes'] = int(ended.sum())
    if S == 2:
        v['wins0'], v['wins1'] = int((coll & ~h0).sum()), int((coll & ~h1).sum())
    v['both_lost'] = int((coll & ((h0 & h1) if S == 2 else coll)).sum())
    v['timeouts'] = int((a & ((ev & nat.EV_TIMEOUT) != 0)).sum())
    v['env_steps'] = int(a.sum())
    v['bullets_spawned'] = S * int((a & ((ev & nat.EV_FIRED) != 0)).sum())
    v['overflow'] = int((a & ((ev & nat.EV_OVERFLOW) != 0)).sum())
    v['planets_live'] = int(arr['n_planets'][a].sum())
    v['bullets_in'] = int(arr['n_bullets'][a].sum())
    v['bullets_out'] = int(o2.nb[a & ~ended].sum())
    v['skipped'] = int(n_pad - a.sum())
    v['bad_controls'] = int((a & bad).sum())
    return v


def _teacher_forced(games, pool, ticks, controls, stats=True):
    """The float32 tick against the oracle, the oracle re-fed the tick's input state every tick, auto-reset on.  Duel
    games tick through astro_tick_many(1 tick, packed controls, event planes): the FIX instantiation; solo games through
    astro_tick with byte controls.  Each tick: the event planes (or event bytes and rewards), bullet counts exactly and
    every list in order, ships / planets / bullets within TOL, re-created games against the pool pick of the tick's
    stream step, and all 14 counters (all zero with stats=False).  Returns totals of what happened."""
    import torch
    cfg, S, K, N, n_pad = games.config, games.S, games.K, games.n, games.n_pad
    M = pool['ships'].shape[0]
    rpool = {k: (v.astype(np.float32).astype(np.float64) if v.dtype != np.int32 else v) for k, v in pool.items()}
    ids = games.first_game + np.arange(N)
    arr = games.get_arrays()
    games.stats(clear=True)
    tot = dict(done=0, hits=0, fired=0, bad=0, overflow=0, worst=0.0)
    for k in range(ticks):
        byte, flown, bad = controls(k)
        alive = ~arr['finished']
        ob, _ = H.oracle_batch_from(arr, S, K)
        ob.reload[:] = games.schedule.reload[arr['tick']]
        ob.t[:] = games.schedule.t[arr['tick']]
        o2, rew, done, ev = ao.step_batch(cfg, ob, flown[:N], alive.astype(np.uint8))
        step = games.step_index
        if S == 2:
            planes = torch.zeros(games.planes_shape(1), dtype=torch.int32, device='cuda')
            games.step_many(1, torch.from_numpy(byte[None]).cuda(), events=planes, auto_reset=True, stats=stats,
                            packed=True, planes=True)
            pl = planes[0].cpu().numpy().view(np.uint32)
            g = np.arange(n_pad)
            got = (pl[:, g // 32] >> (g % 32).astype(np.uint32)) & 1
            want = np.zeros((3, n_pad), dtype=np.uint32)
            want[0, :N], want[1, :N], want[2, :N] = alive & (done != 0), alive & ((ev & 1) != 0), alive & ((ev & 2) != 0)
            assert (got == want).all(), (k, np.nonzero((got != want).any(0))[0][:8])
        else:
            r_gpu, d_gpu, e_gpu = games.step(torch.from_numpy(byte).cuda(), auto_reset=True, stats=stats)
            r_gpu, d_gpu, e_gpu = r_gpu.cpu().numpy(), d_gpu.cpu().numpy(), e_gpu.cpu().numpy()
            want = np.where(alive, ev | np.where(bad[:N], nat.EV_BAD_CONTROL, 0), nat.EV_SKIPPED)
            assert (e_gpu == want).all(), (k, np.nonzero(e_gpu != want)[0][:8], e_gpu[e_gpu != want][:8], want[e_gpu != want][:8])
            assert (d_gpu[alive] == done[alive]).all(), k
            assert (r_gpu[alive].astype(np.float64) == rew[alive]).all(), k
        new = games.get_arrays()
        live, dead = alive & (done == 0), alive & (done != 0)
        assert (new['finished'] == ~alive).all(), k
        assert (new['n_bullets'][live] == o2.nb[live]).all(), k
        assert (new['tick'][live] == arr['tick'][live] + 1).all(), k
        assert (new['n_planets'][live] == arr['n_planets'][live]).all(), k
        assert (new['episode'][live] == arr['episode'][live]).all(), k
        pm = (np.arange(nat.MAX_PLANETS)[None, :] < o2.np_[:, None])[live]
        bm = (np.arange(K)[None, :] < o2.nb[:, None])[live]
        for name, got, ref, mask in (('ships', new['ships'][live], o2.ships[live], None),
                                     ('planets', new['planets'][live], o2.planets[live], pm),
                                     ('bullets', new['bullets'][live], o2.bullets[live], bm)):
            if mask is not None:
                got, ref = got[mask], ref[mask]
            err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
            if err.size:
                tot['worst'] = max(tot['worst'], float(err.max()))
            assert (err <= TOL).all(), (k, name, float(err.max()))
        if dead.any():
            pick = rng.pool_pick(games.seed, ids[dead], np.full(int(dead.sum()), step + 1, dtype=np.uint32), M)
            assert (new['episode'][dead] == arr['episode'][dead] + 1).all(), k
            assert (new['ships'][dead] == rpool['ships'][pick]).all(), k
            assert (new['n_planets'][dead] == rpool['np'][pick]).all(), k
            assert (new['n_bullets'][dead] == 0).all() and (new['tick'][dead] == 0).all(), k
            for j, p in zip(np.nonzero(dead)[0], pick):
                P = rpool['np'][p]
                assert (new['planets'][j, :P] == rpool['planets'][p, :P]).all(), k
        want_st = _expected_stats(S, arr, alive, ev, done, o2, bad[:N], n_pad)
        st = games.stats(clear=True)
        assert st == (want_st if stats else dict.fromkeys(nat.STAT_NAMES, 0)), (k, st, want_st)
        tot['done'] += want_st['episodes']
        tot['hits'] += int((alive & ((ev & 3) != 0)).sum())
        tot['fired'] += int((alive & ((ev & nat.EV_FIRED) != 0)).sum())
        tot['bad'] += want_st['bad_controls']
        tot['overflow'] += want_st['overflow']
        arr = new
    return tot


# ------------------------------------------------------------------ 2. the one-tick FIX form against the oracle

FIX_CASES = {
    'random play': dict(N=4096 + 64, K=32, T=200),
    'random play, statistics off': dict(N=4096 + 64, K=32, T=200, stats=False),
    'stress fill': dict(N=8192, K=32, T=6, start=H.stress_fill(32, 3)),
    'K=0': dict(N=256, K=0, T=90),
    'K=1': dict(N=256, K=1, T=90, stats=False),
    'K=4': dict(N=512, K=4, T=90),
    'K=1023': dict(N=64, K=1023, T=4, start=H.stress_fill(1023, 5)),
    'N=1': dict(N=1, K=32, T=90),
    'N=45': dict(N=45, K=32, T=90, stats=False),
    'seed and first_game': dict(N=1000, K=32, T=60, seed=7, first_game=123457),
    'bad packed codes': dict(N=1024, K=32, T=40, bad=0.05),
}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(FIX_CASES))
def test_fix_one_tick_teacher_forced(case):
    """The production one-tick form, tick_f32_kernel<2, STATS, false, false, true>, teacher-forced against the oracle with
    host-generated packed controls, over the shapes and fills where a tile's list handling can go wrong."""
    c = dict(seed=0, first_game=0, stats=True, start=None, bad=0.0)
    c.update(FIX_CASES[case])
    games, pool = _batch(core.DEFAULT_CONFIG, c['N'], c['K'], seed=c['seed'], first_game=c['first_game'])
    if c['start'] is not None:
        c['start'](games)
    ctl = _controls(games.n_pad, 2, 11, bad=c['bad'])
    tot = _expect([f32(2, int(c['stats']), 0, 0, 1)], lambda: _teacher_forced(games, pool, c['T'], ctl, stats=c['stats']))
    assert tot['fired'] > 0, tot
    if c['T'] >= 60 and c['N'] >= 256:
        assert tot['done'] > 0 and tot['hits'] > 0, tot
    if c['K'] <= 4 or case == 'stress fill':
        assert tot['overflow'] > 0, tot
    if c['bad']:
        assert tot['bad'] > 0.05 * c['N'] * c['T'] * 0.8, tot


@pytest.mark.gpu
def test_golden_edges_through_the_one_tick_forms():
    """The 70 single-step knife-edge and precedence cases of tests/golden/edges.npz (inputs rounded to float32), grouped by
    (config, reload, t): the cases of a group share a batch, spread over the lanes of two tiles whose other slots are
    finished.  Duel cases tick through the FIX one-tick form, solo cases through the generic one."""
    import json
    z = np.load(os.path.join(H.G, 'edges.npz'))
    meta = json.load(open(os.path.join(H.G, 'edges.json')))
    groups = {}
    for c in meta:
        groups.setdefault((json.dumps(c['config'], sort_keys=True), c['reload'], c['t']), []).append(c)
    rnd = lambda a: np.asarray(a, dtype=np.float32).astype(np.float64)

    def run():
        n_cases = n_done = 0
        for (_, reload_, t), cases in groups.items():
            cfg = H.config_from(cases[0]['config'])
            S = 1 if cfg.solo else 2
            games, pool = _batch(cfg, 64, 32, seed=3, pool_size=64, reset=False)
            games.set_schedule_origin(reload_, t)
            index = (5 + 13 * np.arange(len(cases))) % 64
            states = [H.state_from_arrays(rnd(z['c%d_ships' % c['case']]), rnd(z['c%d_planets' % c['case']]),
                                          rnd(z['c%d_bullets' % c['case']]), reload_, t) for c in cases]
            games.set_states(states, index=index, ticks=np.zeros(len(cases), dtype=np.int64))
            flown = np.full((games.n_pad, S), 2)
            flown[index] = [np.asarray(c['control']).reshape(S) for c in cases]
            byte = (flown[:, 0] | (flown[:, 1] << 3)).astype(np.uint8) if S == 2 else flown.astype(np.uint8)
            tot = _teacher_forced(games, pool, 1, lambda k: (byte, flown, np.zeros(games.n_pad, dtype=bool)))
            n_cases += len(cases)
            n_done += tot['done']
        return n_cases, n_done
    n_cases, n_done = _expect([f32(2, 1, 0, 0, 1), f32(1, 1, 0)], run)
    assert n_cases == 70 and n_done > 10


# ------------------------------------------------------------------ 3. the fused resident form on persistent knife edges

def _knife_edges(n, K, seed):
    """One-planet games, the planet at rest at a lane-dependent position (a lone planet feels no gravity), both ships on
    opposite sides of a circular orbit around it, and bullets at rest: two at a few float32 ulps either side of
    planet_radius from the planet, two near the arena corner with min(|x|, |y|) within 4e-6 of 1.  The bullets that
    survive the first tick sit in the float32 uncertainty band on every tick after it.  Returns set_arrays() inputs."""
    cfg = KNIFE_CFG
    r = np.random.RandomState(seed)
    lane, tile = np.arange(n) % 32, np.arange(n) // 32
    f = lambda a: np.asarray(a, dtype=np.float32).astype(np.float64)
    px, py = f(-0.6 + 0.04 * lane), f(-0.45 + 0.3 * ((7 * lane + tile) % 4))
    planets = np.zeros((n, 4, 4))
    planets[:, 0, 0], planets[:, 0, 1] = px, py
    ships = np.zeros((n, 2, 5))
    R = 0.35
    v = np.sqrt(cfg.gravity * cfg.planet_mass / R)
    phase = r.uniform(0, 2 * np.pi, n)
    for s in range(2):
        a = phase + np.pi * s
        ships[:, s, 0], ships[:, s, 1] = px + R * np.cos(a), py + R * np.sin(a)
        ships[:, s, 2], ships[:, s, 3] = -v * np.sin(a), v * np.cos(a)
        ships[:, s, 4] = r.uniform(-np.pi, np.pi, n)
    bl = np.zeros((n, K, 4))
    # planet: bullet 0 is one that the float64 comparison keeps and the float32 one alone would cull, where a game's 512
    # candidates hold one (the float32 threshold lies below the float64 one: a narrow sliver); bullet 1 is random
    C = 512
    th = r.uniform(0, 2 * np.pi, (n, C))
    d = cfg.planet_radius + r.uniform(-1e-8, 1e-8, (n, C))
    d[:, 1] = cfg.planet_radius + r.uniform(-4e-8, 4e-8, n)
    cx, cy = f(px[:, None] + d * np.cos(th)), f(py[:, None] + d * np.sin(th))
    _, keep64, keep32 = _planet_decisions(px[:, None], py[:, None], cx, cy)
    want = keep64 & ~keep32
    want[:, 1] = False
    first = np.where(want.any(axis=1), want.argmax(axis=1), 0)
    bl[:, 0, 0], bl[:, 0, 1] = cx[np.arange(n), first], cy[np.arange(n), first]
    bl[:, 1, 0], bl[:, 1, 1] = cx[:, 1], cy[:, 1]
    # corner: one coordinate just inside the bound, the other just outside (kept: |x| <= 1 or |y| <= 1)
    sx, sy = np.where(r.rand(n, 2) < 0.5, -1.0, 1.0), np.where(r.rand(n, 2) < 0.5, -1.0, 1.0)
    inside, outside = 1.0 - r.uniform(0, 3.5e-6, (n, 2)), 1.0 + r.uniform(0, 3.5e-6, (n, 2))
    x_in = r.rand(n, 2) < 0.5
    bl[:, 2:4, 0] = sx * np.where(x_in, inside, outside)
    bl[:, 2:4, 1] = sy * np.where(x_in, outside, inside)
    bl = f(bl)
    nb = np.full(n, 4)
    ticks = r.randint(0, 100, n)
    return ships, planets, np.ones(n, dtype=np.int64), bl, nb, ticks


def _planet_decisions(px, py, bx, by):
    """A bullet at (bx, by) against a planet at (px, py), float32 values: inside the float32 band of bullet_step_t
    (|d2 - R2| <= 1e-6 R2, d2 = fma(dy, dy, dx * dx) in float32), kept by the float64 comparison (collide_exact), kept by
    the float32 comparison alone."""
    c = KNIFE_CFG
    r2 = (0.0 + c.planet_radius) * (0.0 + c.planet_radius)
    r2f = np.float32(r2)
    dx, dy = np.float32(px) - np.float32(bx), np.float32(py) - np.float32(by)
    p = (dx * dx).astype(np.float64)                                      # a float32 product, then one rounding of dy^2 + p
    d2 = (dy.astype(np.float64) * dy.astype(np.float64) + p).astype(np.float32)
    e0, e1 = np.float64(bx) - np.float64(px), np.float64(by) - np.float64(py)
    return np.abs(d2 - r2f) <= r2f * np.float32(1e-6), ~(e0 * e0 + e1 * e1 < r2), d2 >= r2f


def _band(planets, bullets, nb):
    """Per parked bullet (velocity 0) of one-planet games: inside the planet band, inside the arena band (min(|x|, |y|)
    within 4e-6 of 1), and the planet decisions of _planet_decisions."""
    live = (np.arange(bullets.shape[1])[None, :] < nb[:, None]) & (bullets[..., 2] == 0) & (bullets[..., 3] == 0)
    band, keep64, keep32 = _planet_decisions(planets[:, 0, 0][:, None], planets[:, 0, 1][:, None], bullets[..., 0], bullets[..., 1])
    mn = np.minimum(np.abs(bullets[..., 0]), np.abs(bullets[..., 1])).astype(np.float32)
    in_arena = live & (np.abs(mn - np.float32(1.0)) <= np.float32(4e-6))
    return live & band, in_arena, keep64, keep32


def _knife_batch(N, seed):
    games, pool = _batch(KNIFE_CFG, N, 32, seed=seed)
    games.set_arrays(*_knife_edges(N, 32, seed))
    games.stats(clear=True)
    return games, pool


def _packed(games, T, seed):
    import torch
    ctl = _controls(games.n_pad, 2, seed, no_thrust=True)
    return torch.from_numpy(np.stack([ctl(k)[0] for k in range(T)])).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize('per_launch', [2, 64, 256])
def test_resident_pool_on_persistent_knife_edges(per_launch):
    """On ticks 2..n of a fused launch the tile's bullets stay in shared memory and a bullet in the band is decided by
    the float64 path from its tag.  Bullets parked at rest on the knife edges stay in the band on every tick: the one-tick
    FIX form equals the oracle on them, and launches of `per_launch` ticks equal one launch per tick for 256 ticks
    (state, list order, event planes, statistics)."""
    N, T = 1024, 256
    ships, planets, npl, bl, nb, ticks = _knife_edges(N, 32, 1)
    in_planet, in_arena, keep64, keep32 = _band(planets, bl, nb)
    # the planet does not move, and the band holds bullets the float32 comparison alone would get wrong
    ob = ao.Batch(N, 2, 32)
    ob.ships[:], ob.planets[:], ob.np_[:], ob.bullets[:], ob.nb[:] = ships, planets, npl, bl, nb
    o2, _, done, _ = ao.step_batch(KNIFE_CFG, ob, np.full((N, 2), 2))
    assert (o2.planets[done == 0] == planets[done == 0]).all()
    assert in_planet.sum() > N // 2 and in_arena.sum() > N // 2
    assert (in_planet & keep64 & ~keep32).sum() > N // 8 and (in_planet & keep64 & keep32).sum() > N // 8
    if per_launch == 64:
        games, pool = _knife_batch(N, 1)
        _expect([f32(2, 1, 0, 0, 1)], lambda: _teacher_forced(games, pool, 40, _controls(games.n_pad, 2, 5, no_thrust=True)))
    fused, _ = _knife_batch(N, 1)
    single, _ = _knife_batch(N, 1)
    packed = _packed(fused, T, 7)
    totals = []
    ev_single = _expect([f32(2, 1, 0, 0, 1)], lambda: H.run_launches(single, packed, [1] * T, tile_totals=totals))
    ev_fused = _expect([f32(2, 1, 1, 0, 1)], lambda: H.run_launches(fused, packed, [per_launch] * (T // per_launch)))
    H.check_same(fused, single, ev_fused, ev_single)
    totals = np.array(totals)
    assert (totals <= STAGE_ITEMS).mean() > 0.9 and ev_single[:, 0].any()       # resident ticks; games that ended
    # knife-edge bullets are still there after 256 ticks
    arr = single.get_arrays()
    in_planet, in_arena, _, _ = _band(arr['planets'], arr['bullets'], arr['n_bullets'])
    assert in_planet.sum() > N // 8 and in_arena.sum() > N // 4


@pytest.mark.gpu
def test_resident_pool_over_staging_rounds_and_back():
    """Tiles that start above 448 items (three or more staging rounds) and drop to 224 or fewer inside one 160-tick launch,
    so the tile turns resident again: fused == one launch per tick."""
    N, T = 2048, 160
    fill = H.stress_fill(32, 9)

    def batch():
        games, _ = _batch(KNIFE_CFG, N, 32, seed=4)
        fill(games)
        games.stats(clear=True)
        return games
    fused, single = batch(), batch()
    packed = _packed(fused, T, 3)
    start = H.tile_sums(single.get_arrays()['n_bullets'])
    totals = []
    ev_single = _expect([f32(2, 1, 0, 0, 1)], lambda: H.run_launches(single, packed, [1] * T, tile_totals=totals))
    ev_fused = _expect([f32(2, 1, 1, 0, 1)], lambda: H.run_launches(fused, packed, [T]))
    H.check_same(fused, single, ev_fused, ev_single)
    totals = np.array(totals)
    back = (start > 2 * STAGE_ITEMS) & (totals[:-8] <= STAGE_ITEMS).any(axis=0)
    assert back.sum() >= 8, (start.max(), totals.min(axis=0).max())


# ------------------------------------------------------------------ 4. every statistics-off form against its twin

TWINS = ([('generic single', S, 4) for S in (1, 2)] + [('generic fused', S, 4) for S in (1, 2)] +
         [('fix single', 2, 4), ('fix fused', 2, 4)] + [('bot', S, 4) for S in (1, 2)] +
         [('wide single', S, 8) for S in (1, 2)] + [('wide fused', S, 8) for S in (1, 2)] +
         [(r, S, PL) for r in ('float', 'double') for S in (1, 2) for PL in (4, 8)])


def _twin_forms(kind, S, PL, st):
    return {'generic single': [f32(S, st, 0)], 'generic fused': [f32(S, st, 1)], 'fix single': [f32(2, st, 0, 0, 1)],
            'fix fused': [f32(2, st, 1, 0, 1)], 'bot': [f32(S, st, 1, 1)], 'wide single': [wide(S, st, 0)],
            'wide fused': [wide(S, st, 1)], 'float': [generic('float', S, st, PL)],
            'double': [generic('double', S, st, PL)]}[kind]


@pytest.mark.gpu
@pytest.mark.parametrize('kind,S,PL', TWINS, ids=['%s S=%d PL=%d' % t for t in TWINS])
def test_statistics_off_equals_statistics_on(kind, S, PL):
    """Each of the 20 ASTRO_TICK_NO_STATS instantiations, run on the same inputs as its statistics-on twin: identical
    state (every bullet list in order), events, rewards and done flags; the twin's counters count every env-step, and
    the statistics-off run's stay zero."""
    import torch
    cfg = (WIDE_SOLO if S == 1 else WIDE_DUEL) if PL == 8 else (SOLO_BULLETS if S == 1 else core.DEFAULT_CONFIG)
    N, K, T = 1000, 32, 40
    precision = 64 if kind == 'double' else 32
    runs = []
    for stats in (True, False):
        g, _ = _batch(cfg, N, K, seed=6, precision=precision, planet_slots=PL)
        if kind == 'float':
            g.tick_flags = nat.TICK_GENERIC_KERNEL
        for _ in range(30):
            g.step(None, auto_reset=True)
        g.stats(clear=True)
        gen = torch.Generator(device='cpu').manual_seed(17)
        acts = torch.randint(0, 6, (T, g.n_pad, S), dtype=torch.uint8, generator=gen).cuda()
        packed = g.pack_controls(acts).contiguous() if S == 2 else None
        ev = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
        rw = torch.zeros((T, g.n_pad, S), dtype=torch.float32, device='cuda')
        dn = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')
        planes = torch.zeros(g.planes_shape(T), dtype=torch.int32, device='cuda')

        def run():
            if kind in ('generic single', 'wide single', 'float', 'double'):
                for k in range(T):
                    r, d, e = g.step(acts[k], auto_reset=True, stats=stats)
                    rw[k, :N], dn[k, :N], ev[k, :N] = r, d, e
            elif kind in ('generic fused', 'wide fused'):
                g.step_many(T, acts, events=ev, reward=rw, done=dn, auto_reset=True, stats=stats)
            elif kind == 'fix single':
                for k in range(T):
                    g.step_many(1, packed[k:k + 1], events=planes[k:k + 1], auto_reset=True, stats=stats, packed=True, planes=True)
            elif kind == 'fix fused':
                g.step_many(T, packed, events=planes, auto_reset=True, stats=stats, packed=True, planes=True)
            else:
                g.rollout_device(T, bots='script', stats=stats)
                ev[0] = g._events
        _expect(_twin_forms(kind, S, PL, int(stats)), run)
        runs.append((g.get_arrays(), ev.cpu().numpy(), rw.cpu().numpy(), dn.cpu().numpy(), planes.cpu().numpy(),
                     g.stats(clear=True), g.stats()))
    (a0, *out0, st0, _), (a1, *out1, st1, after) = runs
    for key in a0:
        if key != 'bullets':
            assert np.array_equal(a0[key], a1[key]), key
    live = np.arange(K)[None, :] < a0['n_bullets'][:, None]
    assert np.array_equal(a0['bullets'][live], a1['bullets'][live])
    for x, y in zip(out0, out1):
        assert np.array_equal(x, y)
    assert st0['env_steps'] == N * T and st0['episodes'] > 0 and st0['bullets_spawned'] > 0, st0
    assert st1 == after == dict.fromkeys(nat.STAT_NAMES, 0), st1


# ------------------------------------------------------------------ 5. solo games with bullets

def _park_near_ships_and_planets(seed):
    """A start(games) that parks bullets at rest around every solo game's ship (some inside ship_radius: a hit on the
    first tick; some within a few float32 ulps of it) and at planet_radius from its first planet."""
    def park(games):
        r = np.random.RandomState(seed)
        cfg = games.config
        arr = games.get_arrays()
        n, K = games.n, games.K
        bl = np.zeros((n, 12, 4))
        th = r.uniform(0, 2 * np.pi, (n, 12))
        rad = np.concatenate([cfg.ship_radius * r.uniform(0.5, 3.0, (n, 6)),
                              cfg.ship_radius + r.uniform(-4e-8, 4e-8, (n, 2))], axis=1)
        bl[:, :8, 0] = arr['ships'][:, 0, 0:1] + rad * np.cos(th[:, :8])
        bl[:, :8, 1] = arr['ships'][:, 0, 1:2] + rad * np.sin(th[:, :8])
        pr = cfg.planet_radius + r.uniform(-4e-8, 4e-8, (n, 4))
        bl[:, 8:, 0] = arr['planets'][:, 0, 0:1] + pr * np.cos(th[:, 8:])
        bl[:, 8:, 1] = arr['planets'][:, 0, 1:2] + pr * np.sin(th[:, 8:])
        nb = r.randint(4, 13, n)
        ticks = r.randint(0, 30, n)
        games.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], bl[:, :K], np.minimum(nb, K), ticks)
    return park


@pytest.mark.gpu
@pytest.mark.parametrize('stats', [True, False])
def test_solo_one_tick_teacher_forced_with_bullets(stats):
    """Solo games that fire (reload_time 0.3) with bullets parked around the ship and at the planets' radius: the one-tick
    S = 1 form against the oracle.  Its frame mirrors ship 0 into the second half; a bullet's hit on the only ship sets
    HIT0 alone."""
    games, pool = _batch(SOLO_BULLETS, 2048 + 32, 32, seed=2, pool_size=128)
    _park_near_ships_and_planets(4)(games)
    ctl = _controls(games.n_pad, 1, 8)
    tot = _expect([f32(1, int(stats), 0)], lambda: _teacher_forced(games, pool, 60, ctl, stats=stats))
    assert tot['fired'] > 1000 and tot['hits'] > 200 and tot['done'] >= tot['hits'], tot


@pytest.mark.gpu
@pytest.mark.parametrize('form', ['fused', 'bot', 'wide'])
def test_solo_forms_with_bullets_equal_one_launch_per_tick(form):
    """The S = 1 forms that run several ticks per launch, or 8 planet slots, against one launch per tick of the generic
    form that the oracle checks above: fused (counter stream and given controls), BOT (ScriptBot inside the tick) and
    the 8-slot kernels, on solo games with bullets in flight and parked around the ship."""
    import torch
    cfg = WIDE_SOLO if form == 'wide' else SOLO_BULLETS
    N, K, T = 2000, 32, 90
    outs = []
    for many in (True, False):
        g, _ = _batch(cfg, N, K, seed=3, pool_size=128)
        _park_near_ships_and_planets(6)(g)
        g.stats(clear=True)
        gen = torch.Generator(device='cpu').manual_seed(5)
        acts = torch.randint(0, 6, (T, g.n_pad, 1), dtype=torch.uint8, generator=gen).cuda()
        ev = torch.zeros((T, g.n_pad), dtype=torch.uint8, device='cuda')

        def run():
            if form == 'bot':
                if many:
                    g.rollout_device(T, bots='script')
                else:
                    for k in range(T):
                        g.step(g.script_controls(), auto_reset=True)
                return
            if many:
                g.step_many(T // 2, acts[:T // 2].contiguous(), events=ev[:T // 2], auto_reset=True)
                g.step_many(T - T // 2, None, events=ev[T // 2:], auto_reset=True)
            else:
                for k in range(T):
                    ev[k, :N] = g.step(acts[k] if k < T // 2 else None, auto_reset=True)[2]
        forms = {'fused': [f32(1, 1, int(many))], 'bot': [f32(1, 1, 1, 1) if many else f32(1, 1, 0)],
                 'wide': [wide(1, 1, int(many))]}[form]
        _expect(forms, run)
        outs.append((g.get_arrays(), ev.cpu().numpy()[:, :N], g.stats()))
    (a0, e0, s0), (a1, e1, s1) = outs
    assert np.array_equal(e0, e1) and s0 == s1
    for key in a0:
        if key != 'bullets':
            assert np.array_equal(a0[key], a1[key]), key
    live = np.arange(K)[None, :] < a0['n_bullets'][:, None]
    assert np.array_equal(a0['bullets'][live], a1['bullets'][live])
    assert s0['env_steps'] == N * T and s0['both_lost'] > 100 and s0['bullets_spawned'] > 1000, s0
