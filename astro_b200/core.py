"""Drop-in surface of `astro.core` (reference: astro/core.py) over the CUDA tick.

Same names, argument meaning and results as the reference so that `astro.script`, `astro.rl`
and `astro.server` style code can drive it unchanged:

    Bodies / State / Config / Tick / Game, DEFAULT_CONFIG / SOLO_CONFIG / SOLO_EASY_CONFIG
    generate_configs, create, step, roll_ships, Bot, Bots, play, save_log, load_log

`step` runs the game tick on the GPU (float64 validation arithmetic: results are bit-identical
to the reference — on float64 states, and on the float32 arrays `create` returns, whose first tick
the reference evaluates partly in float32); there is no CPU implementation of the tick in this package.
For throughput use `astro_b200.batched.BatchedGames`, which steps N games per launch.
"""
import collections
import json
import os

import numpy as np

# ---- types (core.py:11-49) ---------------------------------------------------------------
Bodies = collections.namedtuple('Bodies', ('x', 'dx', 'b'))
State = collections.namedtuple('State', ('ships', 'planets', 'bullets', 'reload', 't'))
Config = collections.namedtuple('Config', (
    'gravity', 'dt', 'max_time', 'reload_time', 'bullet_speed', 'ship_thrust', 'ship_rspeed', 'ship_radius',
    'seed', 'solo', 'outer_ship_position', 'inner_ship_position', 'max_planets', 'planet_orbit',
    'planet_mass', 'planet_radius'))
Tick = collections.namedtuple('Tick', ('state', 'control', 'reward', 'bot_data'))
Game = collections.namedtuple('Game', ('config', 'winner', 'ticks'))

# ---- presets (core.py:52-74) ---------------------------------------------------------------
DEFAULT_CONFIG = Config(
    gravity=0.05, dt=0.02, max_time=60, reload_time=0.3, bullet_speed=1.5, ship_thrust=1.0,
    ship_rspeed=4.0, ship_radius=0.025, seed=42, solo=False, outer_ship_position=0.9,
    inner_ship_position=0.2, max_planets=4, planet_orbit=0.5, planet_mass=1.0, planet_radius=0.2)
SOLO_CONFIG = DEFAULT_CONFIG._replace(solo=True, reload_time=1000)
SOLO_EASY_CONFIG = SOLO_CONFIG._replace(max_planets=1)


def direction(bearing):
    """Unit vector (sin b, cos b) in float32 (util.direction, util.py:87-92)."""
    bearing = np.asarray(bearing)
    return np.stack((np.sin(bearing, dtype=np.float32), np.cos(bearing, dtype=np.float32)), axis=-1)


def generate_configs(config):
    """Infinite stream of re-seeded configs (core.py:77-83): MT19937 seeded with config.seed,
    one randint(2**30) per config."""
    stream = np.random.RandomState(config.seed)
    while True:
        yield config._replace(seed=stream.randint(1 << 30))


def create(config):
    """Random initial State, deterministic in config.seed (core.py:86-135).

    Draw order on RandomState(seed): planet count; 2 corner signs; inner-ship bearing; [placement
    coin when there is more than one planet]; one bearing per ship; [planet ring phase and
    direction].  Array dtypes follow the reference under numpy >= 2 (float32 except planets.dx).
    """
    draw = np.random.RandomState(config.seed)
    n_planets = draw.randint(1, config.max_planets + 1)
    corner = config.outer_ship_position * np.sign(draw.rand(2).astype(np.float32) - 0.5)
    near = config.inner_ship_position * direction(2 * np.pi * draw.rand())
    if n_planets == 1:
        ship_x = corner[None] if config.solo else np.stack((corner, -corner))
    elif config.solo:
        ship_x = (corner if draw.rand() < 0.5 else near)[None]
    else:
        ship_x = np.stack((corner, near) if draw.rand() < 0.5 else (near, corner))
    ship_b = 2 * np.pi * draw.rand(ship_x.shape[0]).astype(np.float32)
    if n_planets == 1:
        planet_x = np.zeros((1, 2), dtype=np.float32)
        planet_dx = np.zeros((1, 2), dtype=np.float32)
    else:
        phase = 2 * np.pi * draw.rand() + np.linspace(0, 2 * np.pi, num=n_planets, endpoint=False)
        spin = draw.choice((-1, 1))
        planet_x = config.planet_orbit * direction(phase)
        ring_speed = np.sqrt(config.gravity * config.planet_mass * (n_planets - 1) / 2)
        planet_dx = ring_speed * direction(phase + spin * np.pi / 2)
    empty = np.zeros((0, 2), dtype=np.float32)
    return State(
        ships=Bodies(x=ship_x, dx=np.zeros_like(ship_x), b=ship_b),
        planets=Bodies(x=planet_x, dx=planet_dx, b=None),
        bullets=Bodies(x=empty, dx=empty.copy(), b=None),
        reload=0.0, t=0.0)


# ---- the tick ------------------------------------------------------------------------------
_SINGLE = {}


def _world_key(config):
    return (float(config.gravity), float(config.dt), float(config.max_time), float(config.reload_time),
            float(config.bullet_speed), float(config.ship_thrust), float(config.ship_rspeed),
            float(config.ship_radius), float(config.planet_mass), float(config.planet_radius), bool(config.solo))


def _native():
    from . import _native as nat
    return nat


class _SingleGame:
    """One game on the GPU for `step`: a one-tile float64 batch driven through astro_step_single_host — one pinned
    record in, import -> tick -> export on the stream, one pinned record out.  No tensor indexing, no schedule
    rebuild: reload / t stay Python floats on the host (as in the reference, core.py:257-280,302) and the device is
    told the outcome of their two predicates through a fixed four-entry schedule
    (entry 0, 1: nothing fires; 2: the ships fire; 3: the game times out)."""
    PLAIN, FIRE, TIMEOUT = 1, 2, 3

    def __init__(self, config, cap, planet_slots):
        import ctypes as C
        import torch
        from . import _native as nat
        from .batched import BatchedGames
        self.nat, self.C = nat, C
        self.S = 1 if config.solo else 2
        self.cap = cap
        # (the handle's slots follow the state being stepped, not config.max_planets)
        self.games = BatchedGames(config._replace(max_planets=planet_slots), nat.TILE, bullet_cap=cap, precision=64,
                                  planet_slots=planet_slots)
        fire = np.array([1 << self.FIRE], dtype=np.uint32)
        nat.check(nat.lib().astro_set_schedule(self.games._h, fire.ctypes.data_as(C.c_void_p), 4, self.TIMEOUT))
        self.games.schedule = None       # (the batch's own reload / t tables do not apply to this handle)
        nbytes = int(nat.lib().astro_single_game_bytes(cap))
        self._pin = [torch.zeros(nbytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        pl, wide = nat.AstroSingleGame.planets.offset, nat.MAX_PLANETS_WIDE
        views = []
        for buf in self._pin:
            raw = buf.numpy()
            rec = nat.AstroSingleGame.from_address(buf.data_ptr())
            head = C.sizeof(nat.AstroSingleGame)
            views.append(dict(rec=rec, ptr=C.c_void_p(buf.data_ptr()),
                              ships=raw[0:80].view(np.float64).reshape(2, 5),
                              planets=raw[pl:pl + 32 * wide].view(np.float64).reshape(wide, 4),
                              bullets=raw[head:].view(np.float64).reshape(cap, 4)))
        self.inp, self.out = views

    def step(self, state, control, code, flags=0):
        a, o, S = self.inp, self.out, self.S
        a['ships'][:S, 0:2], a['ships'][:S, 2:4], a['ships'][:S, 4] = state.ships.x, state.ships.dx, state.ships.b
        p, nb = np.shape(state.planets.x)[0], np.shape(state.bullets.x)[0]
        a['planets'][:p, 0:2], a['planets'][:p, 2:4] = state.planets.x, state.planets.dx
        if nb:
            a['bullets'][:nb, 0:2], a['bullets'][:nb, 2:4] = state.bullets.x, state.bullets.dx
        rec = a['rec']
        rec.n_planets, rec.n_bullets, rec.tick = p, nb, code
        for s in range(S):
            rec.control[s] = int(control[s])
        g = self.games
        self.nat.check(self.nat.lib().astro_step_single_host(g._h, a['ptr'], o['ptr'], flags, g._stream()))
        out = o['rec']
        return int(out.events[0]), out.n_bullets, o


def _single_game(config, n_bullets, n_planets):
    nships = 1 if config.solo else 2
    cap = max(32, -(-(n_bullets + nships) // 32) * 32)
    # a game of <= 4 planets always runs in a 4-slot batch: the layout and kernels it has always run in
    slots = 4 if n_planets <= 4 else 8
    key = _world_key(config) + (cap, slots)
    single = _SINGLE.get(key)
    if single is None:
        single = _SINGLE[key] = _SingleGame(config, cap, slots)
    return single


def step(state, control, config):
    """Advance one game by one tick on the GPU (core.py:215-303).

    state -- State; control -- int array [nships] with codes 0..5 (core.py:220-227);
    returns (State or None, reward array [nships]) exactly like the reference: None when the
    game ended; reward is int64 (1 - 2*hit) after a collision and float32 otherwise.
    """
    control = np.asarray(control)
    nships = np.shape(state.ships.x)[0]
    if nships != (1 if config.solo else 2):
        raise ValueError('state has %d ships but config.solo=%r' % (nships, config.solo))
    if control.shape != (nships,) or control.min() < 0 or control.max() > 5:
        raise ValueError('control must hold %d codes 0..5 (core.py:220-227), got %r' % (nships, control))
    npl = np.shape(state.planets.x)[0]
    if not 1 <= npl <= 8:
        raise ValueError('a state needs 1..8 planets, got %d' % npl)
    # reload / t: Python floats, the reference's operations (core.py:257, 263, 267, 280, 302)
    timeout = config.max_time <= state.t + config.dt
    next_reload = state.reload + config.dt
    fire = config.reload_time <= next_reload
    if fire:
        next_reload -= config.reload_time
    single = _single_game(config, np.shape(state.bullets.x)[0], npl)
    code = _SingleGame.TIMEOUT if timeout else (_SingleGame.FIRE if fire else _SingleGame.PLAIN)
    # A state straight from create() holds float32 arrays: the reference's first tick then runs partly in float32
    # (NEP 50 promotion) — reproduced by the kernel's ASTRO_TICK_ALL_CREATE_DTYPES arithmetic.
    raw = (np.shape(state.bullets.x)[0] == 0 and np.asarray(state.ships.x).dtype == np.float32
           and np.asarray(state.planets.x).dtype == np.float32)
    ev, nb, o = single.step(state, control, code, _native().TICK_ALL_CREATE_DTYPES if raw else 0)
    if ev & 3:      # collision: 1 - 2 * hit (core.py:255), int64
        hit = np.array([(ev >> s) & 1 for s in range(nships)], dtype=np.int64)
        return None, 1 - 2 * hit
    if ev & 4:      # timeout (core.py:260)
        return None, np.full(nships, 1 if config.solo else 0, dtype=np.float32)
    sh, pl, bl = o['ships'], o['planets'], o['bullets']
    new = State(ships=Bodies(x=sh[:nships, 0:2].copy(), dx=sh[:nships, 2:4].copy(), b=sh[:nships, 4].copy()),
                planets=Bodies(x=pl[:npl, 0:2].copy(), dx=pl[:npl, 2:4].copy(), b=None),
                bullets=Bodies(x=bl[:nb, 0:2].copy(), dx=bl[:nb, 2:4].copy(), b=None),
                reload=next_reload, t=state.t + config.dt)
    return new, np.zeros(nships, dtype=np.float32)


def roll_ships(state, index):
    """Rotate the ships so that ship `index` comes first (core.py:306-327)."""
    if state is None:
        return None
    s = state.ships
    return State(
        ships=Bodies(x=np.roll(s.x, -index, 0), dx=np.roll(s.dx, -index, 0), b=np.roll(s.b, -index, 0)),
        planets=state.planets, bullets=state.bullets, reload=state.reload, t=state.t)


class Bot:
    """Bot protocol (core.py:330-356)."""

    def __call__(self, state):
        raise NotImplementedError

    def reward(self, state, reward):
        pass

    @property
    def data(self):
        pass


class Bots:
    """Helpers applying a list of bots to a game (core.py:359-374)."""

    @staticmethod
    def control(bots, state):
        return np.array([bot(roll_ships(state, i)) for i, bot in enumerate(bots)])

    @staticmethod
    def reward(bots, state, reward):
        for i, bot in enumerate(bots):
            if hasattr(bot, 'reward'):
                bot.reward(roll_ships(state, i), reward[i])

    @staticmethod
    def data(bots):
        return [bot.data if hasattr(bot, 'data') else None for bot in bots]


def play(config, bots):
    """Play one game to the end (core.py:377-410); every Tick records the pre-step state."""
    ticks = []
    state = create(config)
    while True:
        control = Bots.control(bots, state)
        before = state
        state, reward = step(state, control, config)
        Bots.reward(bots, state, reward)
        ticks.append(Tick(state=before, control=control, reward=reward, bot_data=Bots.data(bots)))
        if state is None:
            winner = None if np.max(reward) < 1 else int(np.argmax(reward))
            return Game(config=config, winner=winner, ticks=ticks)


# ---- JSONL game logs (core.py:413-443, util.py:13-64) -----------------------------------------
_TYPES = {'Bodies': Bodies, 'State': State, 'Config': Config, 'Tick': Tick, 'Game': Game}


def _to_jsonable(obj, module='astro.core'):
    if isinstance(obj, tuple) and hasattr(obj, '_fields'):
        d = {'_type': '%s:%s' % (module, type(obj).__name__)}
        d.update((k, _to_jsonable(getattr(obj, k), module)) for k in obj._fields)
        return d
    if isinstance(obj, np.ndarray):
        return {'_values': obj.tolist(), '_shape': list(obj.shape)}   # nested, as util.to_jsonable (util.py:24-26): astro.js indexes x[i][0]
    if isinstance(obj, dict):
        return {k: _to_jsonable(v, module) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [_to_jsonable(v, module) for v in obj]
    if isinstance(obj, np.generic):
        return obj.item()
    return obj


def _from_jsonable(obj):
    if isinstance(obj, dict):
        if '_type' in obj:
            cls = _TYPES[obj['_type'].split(':')[-1]]
            return cls(**{k: _from_jsonable(v) for k, v in obj.items() if k != '_type'})
        if '_values' in obj:
            return np.array(obj['_values']).reshape(obj['_shape'])
        return {k: _from_jsonable(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_from_jsonable(v) for v in obj]
    return obj


def save_log(path, game):
    """Write a Game as JSON lines in the reference's log format (core.py:413-427): a header
    line {config, winner}, then one Tick per line; arrays as {_values, _shape}, namedtuples
    tagged `_type: astro.core:<Name>` so the reference's UI/loader can replay them."""
    folder = os.path.dirname(path)
    if folder and not os.path.isdir(folder):
        os.makedirs(folder)
    with open(path, 'w') as f:
        f.write(json.dumps(_to_jsonable(dict(config=game.config, winner=game.winner))) + '\n')
        for tick in game.ticks:
            f.write(json.dumps(_to_jsonable(tick)) + '\n')


def load_log(path):
    """Read a game log written by save_log or by the reference (core.py:430-443)."""
    with open(path) as f:
        header = _from_jsonable(json.loads(next(f)))
        ticks = [_from_jsonable(json.loads(line)) for line in f]
    return Game(config=header['config'], winner=header['winner'], ticks=ticks)
