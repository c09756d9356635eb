"""Generate the committed golden vectors by running the UNMODIFIED reference.

Run once in the build container (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py

It imports /root/reference/astro (core.py, util.py, script.py, rl.py) with stub
modules for flask / lru / tensorboardX (tests/golden/_refstubs.py) and writes, next to
this file:

  kat.json        known-answer vectors restated from the reference's own tests
                  (astro/test/test_core.py:6-17, astro/test/test_util.py:59-93),
                  evaluated by the reference functions themselves
  sincos.npz      numpy float32 sin/cos bit patterns (util.direction, util.py:87-92)
  create.npz      core.create() outputs (core.py:86-135) for seeded configs
  traj.npz/.json  full trajectories of core.step (core.py:215-303), inputs
                  canonicalised to float64 (SURVEY.md §8c), random / scripted controls
  edges.npz/.json hand-built knife-edge and terminal-precedence cases through core.step
  schedule.json   spawn ticks / timeout tick observed by running core.step itself
  features.npz    rl.ValueNetwork.get_features / get_features_batch (rl.py:43-112)
  traj_raw.npz/.json  trajectories from core.create's RAW float32 arrays (the first tick's float32 arithmetic)
  network.npz     rl.ValueNetwork (rl.py:115-165) with seeded weights: evaluate / evaluate_batch outputs + state_dict
  explore.json    rl.EpsilonGreedy (rl.py:10-30): empirical transition rates and control histogram
  nstep.json      rl.QBotTrainer.reward (rl.py:303-328): the Experiences the reference's n-step ingestion appends

Everything downstream (oracle/, tests/) reads only these files.
"""
import itertools as it
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import _refstubs  # noqa: E402
_refstubs.install()

from astro import core, util, script, rl  # noqa: E402  (the reference)
from astro_b200 import rng  # noqa: E402  (shared counter-based control stream)


def savez_lzma(path, arrays):
    """np.savez with LZMA members instead of deflate: traj.npz stays under 1 MB (np.load reads either)."""
    import io
    import zipfile
    with zipfile.ZipFile(path, 'w', compression=zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            buf = io.BytesIO()
            np.save(buf, np.asanyarray(a), allow_pickle=False)
            z.writestr(name + '.npy', buf.getvalue())


def f64_state(s):
    """Canonicalise a reference State to float64 arrays (oracle definition)."""
    def b(x):
        return None if x is None else np.asarray(x, dtype=np.float64)
    return core.State(
        ships=core.Bodies(b(s.ships.x), b(s.ships.dx), b(s.ships.b)),
        planets=core.Bodies(b(s.planets.x), b(s.planets.dx), None),
        bullets=core.Bodies(b(s.bullets.x).reshape(-1, 2), b(s.bullets.dx).reshape(-1, 2), None),
        reload=float(s.reload), t=float(s.t))


def cfg_dict(c):
    d = c._asdict()
    d['seed'] = int(d['seed'])
    return d


def pack_ships(s):
    return np.concatenate([s.ships.x, s.ships.dx, s.ships.b[:, None]], axis=1)


def pack_planets(s):
    return np.concatenate([s.planets.x, s.planets.dx], axis=1)


def pack_bullets(s):
    return np.concatenate([s.bullets.x, s.bullets.dx], axis=1).reshape(-1, 4)


# --------------------------------------------------------------------------- KAT

def make_kat():
    kat = {}
    x = [[0, 0], [1.9, 1.9], [3.8, 1.9], [3.8, 0.0]]
    r = [1, 1, 2, 0]
    kat['collisions'] = dict(
        x=x, r=r, hit=[bool(v) for v in core._collisions(np.array(x), np.array(r))])
    bearings = np.arange(0, 2 * np.pi + 1e-3, np.pi / 2)
    kat['direction'] = dict(
        bearing=bearings.tolist(),
        expected=[[0, 1], [1, 0], [0, -1], [-1, 0], [0, 1]],
        value=util.direction(bearings).astype(np.float64).tolist(), atol=1e-6)
    wrap_in = [[1.01, -0.95], [0.95, -1.01], [1.0, -1.0], [3.5, -3.5], [0.0, 0.999]]
    kat['wrap_unit_square'] = dict(
        x=wrap_in, value=util.wrap_unit_square(np.array(wrap_in)).tolist(),
        expected_first2=[[-0.99, -0.95], [0.95, 0.99]], atol=1e-6)
    na_in = [2 * np.pi + 0.5, -4 * np.pi - 0.5, 0.0, np.pi, -np.pi, 240.0, -240.0]
    kat['norm_angle'] = dict(
        b=na_in, value=[float(util.norm_angle(v)) for v in na_in],
        expected_first2=[0.5, -0.5], atol=1e-6)
    kat['generate_configs_seeds'] = [
        int(c.seed) for c in it.islice(core.generate_configs(core.DEFAULT_CONFIG), 8)]
    with open(os.path.join(HERE, 'kat.json'), 'w') as f:
        json.dump(kat, f, indent=1)


def make_sincos():
    r = np.random.RandomState(7)
    x = np.concatenate([
        r.uniform(-260, 260, 20000), r.uniform(-7, 7, 20000),
        r.uniform(-1e-3, 1e-3, 2000), np.arange(0, 2 * np.pi + 1e-3, np.pi / 2),
        np.array([0.0, -0.0, 1e-30, 2.80125, 0.62816095]),
    ]).astype(np.float32)
    # through the reference helper, float64 inputs included (util.py:90-91 casts)
    d32 = util.direction(x)
    d64 = util.direction(x.astype(np.float64))
    assert (d32.view(np.uint32) == d64.view(np.uint32)).all()
    np.savez_compressed(os.path.join(HERE, 'sincos.npz'), x=x,
                        sin_bits=d32[:, 0].view(np.uint32), cos_bits=d32[:, 1].view(np.uint32))


# ------------------------------------------------------------------------ create

def make_create():
    out = {}
    meta = []
    for name, base in (('default', core.DEFAULT_CONFIG), ('solo', core.SOLO_CONFIG),
                       ('solo_easy', core.SOLO_EASY_CONFIG)):
        for k, c in enumerate(it.chain([base], it.islice(core.generate_configs(base), 15))):
            s = core.create(c)
            key = '%s_%d' % (name, k)
            meta.append(dict(key=key, config=cfg_dict(c),
                             dtypes=dict(ships_x=str(s.ships.x.dtype), ships_dx=str(s.ships.dx.dtype),
                                         ships_b=str(s.ships.b.dtype), planets_x=str(s.planets.x.dtype),
                                         planets_dx=str(s.planets.dx.dtype))))
            out[key + '_ships_x'] = s.ships.x
            out[key + '_ships_dx'] = s.ships.dx
            out[key + '_ships_b'] = s.ships.b
            out[key + '_planets_x'] = s.planets.x
            out[key + '_planets_dx'] = s.planets.dx
    np.savez_compressed(os.path.join(HERE, 'create.npz'), **out)
    with open(os.path.join(HERE, 'create.json'), 'w') as f:
        json.dump(meta, f, indent=1)


# ------------------------------------------------------------------ trajectories

def run_game(config, control_fn, state0=None, max_ticks=None, raw=False):
    """Teacher = the reference.  Returns dict of per-tick arrays (pre-step states).
    raw=True: the game starts from core.create's own arrays (float32 positions), NOT canonicalised:
    the reference's first tick then runs partly in float32 (recorded values are exact in float64)."""
    state = core.create(config) if raw else f64_state(core.create(config) if state0 is None else state0)
    ships, planets, nb, bullets, reload_, t_, ctrl, rew = [], [], [], [], [], [], [], []
    k = 0
    while True:
        c = np.asarray(control_fn(state, k), dtype=np.int64)
        ships.append(pack_ships(state))
        planets.append(pack_planets(state))
        bl = pack_bullets(state)
        nb.append(bl.shape[0])
        bullets.append(bl)
        reload_.append(state.reload)
        t_.append(state.t)
        ctrl.append(c)
        nxt, reward = core.step(state, c, config)
        rew.append(np.asarray(reward, dtype=np.float64))
        k += 1
        if nxt is None:
            truncated = False
            break
        assert nxt.ships.x.dtype == np.float64 and (raw or nxt.planets.x.dtype == np.float64)
        state = nxt
        if max_ticks is not None and k >= max_ticks:
            truncated = True
            # record the final (post-step) state as one more pre-step entry w/o step
            break
    out = dict(ships=np.stack(ships), planets=np.stack(planets), nb=np.array(nb, dtype=np.int32),
               bullets=np.concatenate(bullets, axis=0) if bullets else np.zeros((0, 4)),
               reload=np.array(reload_), t=np.array(t_), control=np.stack(ctrl),
               reward=np.stack(rew))
    if truncated:
        out['final_ships'] = pack_ships(state)
        out['final_planets'] = pack_planets(state)
        out['final_bullets'] = pack_bullets(state)
        out['final_reload_t'] = np.array([state.reload, state.t])
    return out, truncated


def make_traj():
    arrays, meta = {}, []

    def add(kind, config, control_fn, **kw):
        g = len(meta)
        data, truncated = run_game(config, control_fn, **kw)
        for k, v in data.items():
            arrays['g%d_%s' % (g, k)] = v
        meta.append(dict(game=g, kind=kind, config=cfg_dict(config), nships=int(data['ships'].shape[1]),
                         nplanets=int(data['planets'].shape[1]), nticks=int(data['ships'].shape[0]),
                         truncated=bool(truncated), max_bullets=int(data['nb'].max())))
        print(kind, meta[-1]['nticks'], 'ticks, P =', meta[-1]['nplanets'],
              'max nb =', meta[-1]['max_bullets'], 'final reward', data['reward'][-1])

    # (1) duel, uniform random controls from the shared counter stream (seed 0, game id = g)
    for g, c in enumerate(it.islice(core.generate_configs(core.DEFAULT_CONFIG), 24)):
        add('duel_random', c,
            lambda s, k, g=g: rng.actions(0, np.array([g]), k, 2)[0])
    # (2) config #1 of BASELINE.json: script bot vs script bot, default map
    for c in it.islice(core.generate_configs(core.DEFAULT_CONFIG), 3):
        bots = [script.ScriptBot.create(c), script.ScriptBot.create(c)]
        add('duel_script', c, lambda s, k, bots=bots: core.Bots.control(bots, s), max_ticks=700)
    # (3) nothing vs script (test_core.py:94-98): bullets hitting ships
    for c in it.islice(core.generate_configs(core.DEFAULT_CONFIG._replace(max_time=20)), 3):
        bots = [script.NothingBot(), script.ScriptBot.create(c)]
        add('duel_nothing_vs_script', c, lambda s, k, bots=bots: core.Bots.control(bots, s))
    # (4) duel, nobody steers: long games, timeout path at max_time=6 (tick 299)
    for c in it.islice(core.generate_configs(core.DEFAULT_CONFIG._replace(max_time=6)), 3):
        add('duel_idle_short_timeout', c, lambda s, k: np.array([2, 2]))
    # (5) solo games (test_core.py:55-75,88-92)
    for c in it.islice(core.generate_configs(core.SOLO_EASY_CONFIG), 2):
        add('solo_easy_nothing', c, lambda s, k: np.array([2]))
    for c in it.islice(core.generate_configs(core.SOLO_CONFIG), 2):
        add('solo_nothing', c, lambda s, k: np.array([2]), max_ticks=600)
    for c in it.islice(core.generate_configs(core.SOLO_CONFIG._replace(max_time=8)), 2):
        bot = script.ScriptBot.create(c)
        add('solo_script_timeout', c, lambda s, k, bot=bot: np.array([bot(s)]))
    savez_lzma(os.path.join(HERE, 'traj.npz'), arrays)
    with open(os.path.join(HERE, 'traj.json'), 'w') as f:
        json.dump(meta, f, indent=1)


def make_traj_raw():
    """Games played by the reference from core.create's RAW output (float32 ships / planet positions): pins the
    float32 arithmetic of the first tick (core.py:138-153, :200-212 on float32 arrays) and everything after it."""
    arrays, meta = {}, []

    def add(kind, config, control_fn, **kw):
        g = len(meta)
        data, truncated = run_game(config, control_fn, raw=True, **kw)
        for k, v in data.items():
            arrays['g%d_%s' % (g, k)] = v
        meta.append(dict(game=g, kind=kind, config=cfg_dict(config), nships=int(data['ships'].shape[1]),
                         nplanets=int(data['planets'].shape[1]), nticks=int(data['ships'].shape[0]),
                         truncated=bool(truncated), max_bullets=int(data['nb'].max())))
        print('raw', kind, meta[-1]['nticks'], 'ticks, P =', meta[-1]['nplanets'])

    for g, c in enumerate(it.islice(core.generate_configs(core.DEFAULT_CONFIG._replace(seed=7)), 12)):
        add('duel_random_raw', c, lambda s, k, g=g: rng.actions(3, np.array([g]), k, 2)[0], max_ticks=120)
    # ships fire on the very first tick (reload_time <= dt): the newborn are float32 throughout
    for g, c in enumerate(it.islice(core.generate_configs(core.DEFAULT_CONFIG._replace(seed=8, reload_time=0.02)), 4)):
        add('duel_fire_every_tick_raw', c, lambda s, k, g=g: rng.actions(4, np.array([g]), k, 2)[0], max_ticks=40)
    for c in it.islice(core.generate_configs(core.SOLO_CONFIG._replace(seed=9)), 3):
        add('solo_nothing_raw', c, lambda s, k: np.array([3]), max_ticks=80)
    np.savez_compressed(os.path.join(HERE, 'traj_raw.npz'), **arrays)
    with open(os.path.join(HERE, 'traj_raw.json'), 'w') as f:
        json.dump(meta, f, indent=1)


# -------------------------------------------------------------------- edge cases

def make_edges():
    """Single core.step calls on hand-built states: predicate knife edges, terminal
    precedence, bullet cull quirk (SURVEY.md §8c item 5-6)."""
    cfg = core.DEFAULT_CONFIG
    cases = []

    def state(ships, planets, bullets, reload=0.0, t=0.0):
        ships = np.asarray(ships, dtype=np.float64).reshape(-1, 5)
        planets = np.asarray(planets, dtype=np.float64).reshape(-1, 4)
        bullets = np.asarray(bullets, dtype=np.float64).reshape(-1, 4)
        return core.State(
            ships=core.Bodies(ships[:, 0:2].copy(), ships[:, 2:4].copy(), ships[:, 4].copy()),
            planets=core.Bodies(planets[:, 0:2].copy(), planets[:, 2:4].copy(), None),
            bullets=core.Bodies(bullets[:, 0:2].copy(), bullets[:, 2:4].copy(), None),
            reload=reload, t=t)

    def add(name, s, control, config=cfg):
        control = np.asarray(control, dtype=np.int64)
        nxt, reward = core.step(s, control, config)
        c = dict(name=name, config=cfg_dict(config), control=control.tolist(),
                 done=nxt is None, reward=np.asarray(reward, dtype=np.float64).tolist(),
                 reload=s.reload, t=s.t)
        arr = dict(ships=pack_ships(s), planets=pack_planets(s), bullets=pack_bullets(s))
        if nxt is not None:
            arr.update(o_ships=pack_ships(nxt), o_planets=pack_planets(nxt), o_bullets=pack_bullets(nxt))
            c['o_reload'], c['o_t'] = nxt.reload, nxt.t
        cases.append((c, arr))

    far_planet = [[0.0, 0.0, 0.0, 0.0]]
    quiet = [[-0.7, -0.7, 0, 0, 0.3], [0.7, 0.7, 0, 0, -2.0]]
    f32 = np.float32

    # bullet cull quirk: kept while EITHER coordinate is inside [-1, 1] (core.py:195)
    add('cull_any_axis', state(quiet, far_planet, [
        [1.5, 0.0, 0, 0], [1.5, 1.5, 0, 0], [-1.0, 1.0, 0, 0], [0.5, -1.7, 0, 0],
        [-3.0, 2.0, 0, 0], [1.0, 1.0, 0, 0]]), [2, 2])
    # cull knife edge: x' lands within 1 ulp(f64) / 1 ulp(f32) of +-1
    edge = []
    for x0 in (1.0, np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0), float(np.nextafter(f32(1.0), f32(2.0))),
               float(np.nextafter(f32(1.0), f32(0.0))), -1.0, float(np.nextafter(f32(-1.0), f32(-2.0)))):
        edge.append([x0, 2.0, 0.0, 0.0])           # y out: kept iff x in
        edge.append([2.0, x0, 0.0, 0.0])
    for v in (0.5, 1.5, -1.5, 0.25):
        x0 = float(f32(1.0 - 0.02 * v))            # float32 start (what the fp32 build stores)
        edge.append([x0, 3.0, v, 0.0])
        edge.append([-x0, -3.0, -v, 0.0])
    add('cull_knife_edge', state(quiet, far_planet, edge), [2, 2])

    # collision knife edges: |d|^2 vs (r_i+r_j)^2 strict '<' (core.py:210-212)
    rs, rp = cfg.ship_radius, cfg.planet_radius
    for name, R, other in (('ship_planet', rs + rp, 'planet'), ('ship_ship', rs + rs, 'ship'),
                           ('ship_bullet', rs, 'bullet'), ('planet_bullet', rp, 'bullet_p')):
        for k, delta in enumerate((0.0, 1.0, -1.0)):
            d = R
            for _ in range(int(abs(delta))):
                d = np.nextafter(d, 10.0 if delta > 0 else 0.0)
            ships = [[-0.5, -0.5, 0, 0, 0.3], [0.7, 0.7, 0, 0, -2.0]]
            planets = [[0.0, 0.5, 0.0, 0.0]]
            bullets = []
            if other == 'planet':
                ships[0][0:2] = [0.0 + d, 0.5]
            elif other == 'ship':
                ships[1][0:2] = [-0.5, -0.5 + d]
            elif other == 'bullet':
                bullets = [[-0.5 - d, -0.5, 0.1, 0.1], [0.3, 0.3, 0.2, -0.1]]
            else:
                bullets = [[0.3, 0.3, 0.2, -0.1], [0.0, 0.5 - d, 0.1, 0.1], [-0.3, -0.3, 0.2, -0.1]]
            add('knife_%s_%d' % (name, k), state(ships, planets, bullets), [2, 3])
    # float32-stored near-contact (the production layout stores f32)
    for k, eps in enumerate((0, 1, -1, 2, -2)):
        d = f32(rs + rp)
        for _ in range(abs(eps)):
            d = np.nextafter(d, f32(10.0 if eps > 0 else 0.0))
        add('knife_f32_ship_planet_%d' % k,
            state([[float(d), 0.5, 0, 0, 0.3], [0.7, 0.7, 0, 0, -2.0]], [[0.0, 0.5, 0, 0]], []), [2, 2])

    # terminal precedence and reward conventions (core.py:253-260)
    t_last = 59.98000000000378     # value of t on step-call 2999 of the default config
    add('collision_and_timeout_same_tick', state(
        [[0.1, 0.5, 0, 0, 0.3], [0.7, 0.7, 0, 0, -2.0]], [[0.0, 0.5, 0, 0]], [], t=t_last), [2, 2])
    add('timeout_only', state(quiet, far_planet, [[0.2, 0.9, 0.1, 0.0]], t=t_last), [2, 2])
    add('timeout_not_yet', state(quiet, far_planet, [], t=59.95), [2, 2])
    add('bullet_hits_ship0', state(quiet, far_planet, [[-0.71, -0.70, 0, 0], [0.3, 0.3, 0, 0]]), [2, 2])
    add('bullet_hits_ship1', state(quiet, far_planet, [[0.3, 0.3, 0, 0], [0.71, 0.71, 0, 0]]), [2, 2])
    add('ship_ship', state([[0.5, 0.5, 0, 0, 0.3], [0.52, 0.53, 0, 0, -2.0]], far_planet, []), [2, 2])
    add('both_into_planet', state([[0.1, 0.0, 0, 0, 0.3], [-0.1, 0.05, 0, 0, -2.0]], far_planet, []), [2, 2])
    add('bullet_in_planet_removed', state(quiet, far_planet, [
        [0.3, 0.3, 0.1, 0], [0.05, 0.1, 0.1, 0], [-0.3, 0.4, 0, 0.1], [0.19, 0.0, 0, 0]]), [1, 4])
    solo = core.SOLO_CONFIG
    add('solo_timeout', state([quiet[0]], far_planet, [], t=t_last), [2], config=solo)
    add('solo_crash', state([[0.1, 0.0, 0, 0, 0.3]], far_planet, []), [3], config=solo)
    # firing: both ships fire together, old ship state used, order [survivors, ship0, ship1]
    add('fire_tick', state(
        [[-0.7, -0.7, 0.3, -0.2, 0.3], [0.7, 0.7, -0.1, 0.4, -2.0]], far_planet,
        [[0.3, 0.3, 0.1, 0], [0.05, 0.1, 0.1, 0], [-0.3, 0.4, 0, 0.1]], reload=0.28), [5, 0])
    add('fire_tick_exact_threshold', state(quiet, far_planet, [], reload=0.3 - 0.02), [2, 2])
    add('fire_newborn_culled', state(
        [[0.9995, 0.9995, 1.0, 1.0, np.pi / 4], [-0.7, 0.7, 0, 0, 0.1]], far_planet, [], reload=0.29), [2, 2])
    # wrap of ships / large bearings / controls
    add('ship_wraps', state(
        [[0.9999, -0.9999, 2.0, -3.0, 200.5], [-0.99999, 0.7, -1.0, 0, -240.0]], far_planet, []), [1, 5])
    for ctl in it.product(range(6), range(6)):
        add('controls_%d%d' % ctl, state(
            [[-0.6, -0.5, 0.1, 0.2, 1.3], [0.6, 0.55, -0.1, 0.05, -4.0]],
            [[0.0, 0.5, 0.2, 0.0], [0.0, -0.5, -0.2, 0.0]], [[0.1, 0.1, 1.0, 1.0]], reload=0.1, t=1.0), ctl)
    # 4 planets, planet-planet gravity incl. the clamped self term
    add('four_planets', state(
        quiet, [[0.5, 0, 0, 0.27], [0, 0.5, -0.27, 0], [-0.5, 0, 0, -0.27], [0, -0.5, 0.27, 0]], []), [3, 3])

    arrays, meta = {}, []
    for i, (c, arr) in enumerate(cases):
        c['case'] = i
        meta.append(c)
        for k, v in arr.items():
            arrays['c%d_%s' % (i, k)] = v
    np.savez_compressed(os.path.join(HERE, 'edges.npz'), **arrays)
    with open(os.path.join(HERE, 'edges.json'), 'w') as f:
        json.dump(meta, f, indent=1)
    print(len(cases), 'edge cases;', sum(c['done'] for c, _ in cases), 'terminal')


# ---------------------------------------------------------------------- schedule

def make_schedule():
    """Observe spawn ticks and the timeout tick by running core.step itself on a world
    where nothing ever collides (gravity 0, everything at rest, ships aim outwards)."""
    out = {}
    for name, c in (('default', core.DEFAULT_CONFIG),
                    ('max_time_20', core.DEFAULT_CONFIG._replace(max_time=20)),
                    ('reload_0p25', core.DEFAULT_CONFIG._replace(reload_time=0.25, max_time=30)),
                    ('dt_0p03', core.DEFAULT_CONFIG._replace(dt=0.03, max_time=45, reload_time=0.31)),
                    ('solo', core.SOLO_CONFIG)):
        cq = c._replace(gravity=0.0)
        S = 1 if c.solo else 2
        ships = np.array([[-0.9, -0.9, 0, 0, -3 * np.pi / 4], [0.9, 0.9, 0, 0, np.pi / 4]])[:S]
        s = core.State(
            ships=core.Bodies(ships[:, 0:2].copy(), ships[:, 2:4].copy(), ships[:, 4].copy()),
            planets=core.Bodies(np.array([[0.0, 0.0]]), np.array([[0.0, 0.0]]), None),
            bullets=core.Bodies(np.zeros((0, 2)), np.zeros((0, 2)), None), reload=0.0, t=0.0)
        spawn, k = [], 0
        control = np.full(S, 2)
        reloads, ts = [], []
        while True:
            before = s.bullets.x.shape[0]
            reloads.append(s.reload)
            ts.append(s.t)
            nxt, reward = core.step(s, control, cq)
            if nxt is None:
                assert not (np.asarray(reward) < 0).any()
                timeout_tick = k
                break
            # newborn bullets leave the arena only after many ticks; a count increase = a spawn
            if nxt.reload < s.reload:
                spawn.append(k)
            s = nxt
            k += 1
        out[name] = dict(config=cfg_dict(c), spawn_ticks=spawn, timeout_tick=timeout_tick,
                         reload_hex=[float(v).hex() for v in reloads], t_hex=[float(v).hex() for v in ts])
        print(name, 'spawns', len(spawn), spawn[:4], 'timeout tick', timeout_tick)
    with open(os.path.join(HERE, 'schedule.json'), 'w') as f:
        json.dump(out, f)


# ---------------------------------------------------------------------- features

def make_features():
    """rl.ValueNetwork.get_features / get_features_batch on states sampled from traj.npz."""
    z = np.load(os.path.join(HERE, 'traj.npz'))
    meta = json.load(open(os.path.join(HERE, 'traj.json')))
    arrays, fmeta = {}, []
    for m in meta:
        g = m['game']
        if m['kind'] not in ('duel_random', 'duel_script', 'solo_nothing', 'duel_nothing_vs_script'):
            continue
        nb = z['g%d_nb' % g]
        off = np.concatenate([[0], np.cumsum(nb)])
        ticks = sorted(set([0, m['nticks'] // 3, m['nticks'] // 2, m['nticks'] - 1, int(np.argmax(nb))]))
        states = []
        for k in ticks:
            sh = z['g%d_ships' % g][k]
            pl = z['g%d_planets' % g][k]
            bl = z['g%d_bullets' % g][off[k]:off[k + 1]]
            states.append(core.State(
                ships=core.Bodies(sh[:, 0:2], sh[:, 2:4], sh[:, 4]),
                planets=core.Bodies(pl[:, 0:2], pl[:, 2:4], None),
                bullets=core.Bodies(bl[:, 0:2], bl[:, 2:4], None),
                reload=float(z['g%d_reload' % g][k]), t=float(z['g%d_t' % g][k])))
        for k, s in zip(ticks, states):
            arrays['g%d_t%d_f0' % (g, k)] = rl.ValueNetwork.get_features(s)
            if m['nships'] == 2:
                arrays['g%d_t%d_f1' % (g, k)] = rl.ValueNetwork.get_features(core.roll_ships(s, 1))
        arrays['g%d_batch' % g] = rl.ValueNetwork.get_features_batch(states)
        fmeta.append(dict(game=g, ticks=ticks, nships=m['nships']))
    np.savez_compressed(os.path.join(HERE, 'features.npz'), **arrays)
    with open(os.path.join(HERE, 'features.json'), 'w') as f:
        json.dump(fmeta, f)
    print(len(arrays), 'feature arrays')


def make_network():
    """The reference's ValueNetwork (rl.py:32-165) with seeded weights on the states of features.npz:
    evaluate / evaluate_batch outputs for ship 0's perspective and (duel) the rolled perspective of ship 1,
    plus the flattened state_dict — pins forward, forward_both and the fused policy kernel."""
    import torch
    z = np.load(os.path.join(HERE, 'traj.npz'))
    fmeta = json.load(open(os.path.join(HERE, 'features.json')))
    arrays = {}
    nets = {}
    for solo in (False, True):
        torch.manual_seed(1234 + int(solo))
        net = rl.ValueNetwork(solo=solo, nout=6)
        with torch.no_grad():                 # (default init is small: widen it so that the outputs spread over (-1, 1))
            for p_ in net.parameters():
                p_.mul_(3.0)
        nets[solo] = net
        for name, v in net.state_dict().items():
            arrays['%s_%s' % ('solo' if solo else 'duel', name.replace('.', '_'))] = v.numpy().copy()
    for m in fmeta:
        g, solo = m['game'], m['nships'] == 1
        nb = z['g%d_nb' % g]
        off = np.concatenate([[0], np.cumsum(nb)])
        states = []
        for k in m['ticks']:
            sh, pl, bl = z['g%d_ships' % g][k], z['g%d_planets' % g][k], z['g%d_bullets' % g][off[k]:off[k + 1]]
            states.append(core.State(ships=core.Bodies(sh[:, 0:2], sh[:, 2:4], sh[:, 4]),
                                     planets=core.Bodies(pl[:, 0:2], pl[:, 2:4], None),
                                     bullets=core.Bodies(bl[:, 0:2], bl[:, 2:4], None),
                                     reload=float(z['g%d_reload' % g][k]), t=float(z['g%d_t' % g][k])))
        net = nets[solo]
        with torch.no_grad():
            arrays['g%d_q0' % g] = net.evaluate_batch(states).numpy()
            arrays['g%d_q0_single' % g] = np.stack([net.evaluate(s).numpy() for s in states])
            if not solo:
                arrays['g%d_q1' % g] = net.evaluate_batch([core.roll_ships(s, 1) for s in states]).numpy()
    np.savez_compressed(os.path.join(HERE, 'network.npz'), **arrays)
    print(len(arrays), 'network arrays; torch', torch.__version__)


def make_explore():
    """rl.EpsilonGreedy (rl.py:10-30) run by the reference itself over many calls at the game's dt: the empirical
    enter / leave rates, the active fraction and the histogram of its random controls — what the device-side
    process (another random stream) has to reproduce statistically."""
    State = core.State
    out = []
    for t_in, t_out in ((1.0, 0.1), (0.5, 0.5)):
        eg = rl.EpsilonGreedy(t_in, t_out, seed=5)
        dt, n = 0.02, 400000
        idle_calls = active_calls = entered = left = 0
        hist = [0] * 6
        t = 0.0
        for k in range(n):
            was = eg._policy
            now = eg(State(None, None, None, 0.0, t))
            t += dt
            if was is None:
                idle_calls += 1
                entered += now is not None
            else:
                active_calls += 1
                left += now is None
            if now is not None:
                hist[int(now)] += 1
        out.append(dict(t_in=t_in, t_out=t_out, dt=dt, calls=n, idle_calls=idle_calls, active_calls=active_calls,
                        entered=int(entered), left=int(left), hist=hist))
    with open(os.path.join(HERE, 'explore.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print('explore', out)


def make_nstep():
    """rl.QBotTrainer.reward (rl.py:303-328) — the n-step replay ingestion — run by the reference itself on the logged
    ticks of the recorded duel games played back to back by one bot slot per ship (the bot object persists across games,
    like rl.train's): per (n_steps, discount) setting the Experiences it appended, each identified by the global tick of
    its state: (tick, action, reward, discount, tick of the new state or -1)."""
    z = np.load(os.path.join(HERE, 'traj.npz'))
    meta = json.load(open(os.path.join(HERE, 'traj.json')))
    games = [m for m in meta if m['kind'] == 'duel_random' and not m['truncated']][:10]
    ticks = []                                   # (action pair, reward pair, terminal)
    for m in games:
        g = m['game']
        for k in range(m['nticks']):
            ticks.append((z['g%d_control' % g][k].tolist(), z['g%d_reward' % g][k].tolist(), k == m['nticks'] - 1))

    class Q:
        @staticmethod
        def get_features(state):
            return state                         # (a state stands for itself: its global tick)

    class Trainer:
        q = Q()
    out = dict(ticks=ticks, settings=[])
    for n_steps, discount in ((100, 0.995), (7, 0.9), (1, 0.5)):
        per_ship = []
        for me in range(2):
            bot = rl.QBotTrainer(Trainer(), seed=1)
            bot.n_steps, bot.discount = n_steps, discount
            bot._step = lambda: None             # (the optimisation step is not part of the ingestion)
            for t, (action, reward, terminal) in enumerate(ticks):
                bot._nstep_buffer.append((t, int(action[me])))          # what __call__ appends (rl.py:254): (features, action)
                bot.reward(None if terminal else t + 1, reward[me])
            per_ship.append([[int(x.state_f), int(x.action), float(x.reward), float(x.discount),
                              -1 if x.new_state_f is None else int(x.new_state_f)] for x in bot._replay_buffer]
                            + [['held', len(bot._nstep_buffer)]])
        out['settings'].append(dict(n_steps=n_steps, discount=discount, experiences=per_ship))
    with open(os.path.join(HERE, 'nstep.json'), 'w') as f:
        json.dump(out, f)
    print('nstep', [len(s['experiences'][0]) for s in out['settings']], 'experiences over', len(ticks), 'ticks')


if __name__ == '__main__':
    if len(sys.argv) > 1:          # python make_golden.py make_network make_explore ...: only the named parts
        for name in sys.argv[1:]:
            globals()[name]()
        sys.exit(0)
    make_kat()
    make_sincos()
    make_create()
    make_traj()
    make_edges()
    make_schedule()
    make_features()
    make_traj_raw()
    make_network()
    make_explore()
    make_nstep()
    print('numpy', np.__version__)
