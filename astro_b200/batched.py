"""BatchedGames — N independent Astro games resident in HBM, advanced by one CUDA launch per tick.

Host side of the C ABI in include/astro_b200.h.  PyTorch owns the device memory and the stream;
all arithmetic of the tick / observation path runs in csrc/astro_b200.cu.  There is no CPU
implementation behind this class.

Reference semantics: one `step()` here == `astro.core.step` (astro/core.py:215-303) applied to
every game; `observe()` == `ValueNetwork.get_features_batch` (astro/rl.py:43-112) for every game
and both ship perspectives (`core.roll_ships`, core.py:306-327).
"""
import ctypes as C

import numpy as np

from . import _native as nat
from . import core
from .schedule import Schedule


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('astro_b200 needs a CUDA device: there is no CPU path for the game tick')
    return torch


def planet_slots_for(config):
    """Planet slots per game of a batch playing `config`: 4 for max_planets <= 4 (the batch is laid out exactly as
    before 8-slot batches existed), 8 for max_planets 5..8."""
    mp = int(config.max_planets)
    if mp > nat.MAX_PLANETS_WIDE:
        raise ValueError('config.max_planets=%d: games of at most %d planets are supported' % (mp, nat.MAX_PLANETS_WIDE))
    return nat.MAX_PLANETS if mp <= nat.MAX_PLANETS else nat.MAX_PLANETS_WIDE


class BatchedGames:
    def __init__(self, config, n_games, bullet_cap=32, precision=32, device=None, seed=0, first_game=0, planet_slots=None):
        """planet_slots: planet rows per game, 4 or 8; by default planet_slots_for(config).  8 slots hold games of up to
        eight planets (the `planets` tensor is [tiles, 8, 32, 4], game-major arrays [m, 8, 4])."""
        torch = _torch()
        if precision not in (32, 64):
            raise ValueError('precision must be 32 or 64')
        if not 0 <= bullet_cap <= nat.MAX_BULLET_CAP:
            raise ValueError('bullet_cap out of range')
        default_pl = planet_slots_for(config)
        self.PL = default_pl if planet_slots is None else int(planet_slots)
        if self.PL not in (nat.MAX_PLANETS, nat.MAX_PLANETS_WIDE):
            raise ValueError('planet_slots must be %d or %d' % (nat.MAX_PLANETS, nat.MAX_PLANETS_WIDE))
        if self.PL < default_pl:
            raise ValueError('config.max_planets=%d needs planet_slots=%d' % (int(config.max_planets), default_pl))
        self.config = config
        self.S = 1 if config.solo else 2
        self.D = 1 + 5 * self.S + 4
        self.n = int(n_games)
        self.n_tiles = -(-self.n // nat.TILE)
        self.n_pad = self.n_tiles * nat.TILE
        self.K = int(bullet_cap)
        self.precision = precision
        self.device = torch.device('cuda', torch.cuda.current_device() if device is None else int(device))
        self.rdtype = torch.float32 if precision == 32 else torch.float64
        self.np_rdtype = np.float32 if precision == 32 else np.float64
        self.seed, self.first_game = int(seed), int(first_game)
        dev, T, S, K = self.device, self.n_tiles, self.S, self.K
        self.ships = torch.zeros((T, S, 32, 4), dtype=self.rdtype, device=dev)
        self.ship_b = torch.zeros((T, S, 32), dtype=self.rdtype, device=dev)
        self.planets = torch.zeros((T, self.PL, 32, 4), dtype=self.rdtype, device=dev)
        # tile lists, two buffers (include/astro_b200.h): the current one is astro_bullet_buffer()
        self.bullets = torch.zeros((2, T, 32 * max(K, 1), 4), dtype=self.rdtype, device=dev)
        # every slot starts finished (empty); meta = nb | np<<10 | finished<<13 | tick<<14 (8 slots: np's bit 3 in bit 31)
        self.meta = torch.full((self.n_pad,), 1 << 13, dtype=torch.int32, device=dev)
        self.episode = torch.zeros((self.n_pad,), dtype=torch.int32, device=dev)
        self._reward = torch.zeros((self.n_pad, S), dtype=torch.float32, device=dev)
        self._done = torch.zeros((self.n_pad,), dtype=torch.uint8, device=dev)
        self._events = torch.zeros((self.n_pad,), dtype=torch.uint8, device=dev)
        self._actions = torch.zeros((self.n_pad, S), dtype=torch.uint8, device=dev)
        self._stats = torch.zeros((nat.N_STATS,), dtype=torch.int64, device=dev)
        self._pool = None
        self.tick_flags = 0      # extra ASTRO_TICK_* bits OR-ed into every tick (kernel A/B selection)

        L = nat.lib()
        cfg = nat.AstroConfig()
        for name, _ in nat.AstroConfig._fields_[:10]:
            setattr(cfg, name, float(getattr(config, name)))
        cfg.solo = int(bool(config.solo))
        cfg.planet_slots = self.PL
        handle = C.c_void_p()
        nat.check(L.astro_batch_create(C.byref(cfg), self.n_pad, self.K, precision, self.device.index, C.byref(handle)))
        self._h = handle
        bufs = nat.AstroBuffers(self.ships.data_ptr(), self.ship_b.data_ptr(), self.planets.data_ptr(),
                                self.bullets.data_ptr(), self.meta.data_ptr(), self.episode.data_ptr())
        nat.check(L.astro_batch_bind(self._h, C.byref(bufs)))
        self.schedule = None
        self.set_schedule_origin(0.0, 0.0)
        self.step_index = 0
        nat.check(L.astro_set_stream(self._h, self.seed, self.first_game, 0))

    def __del__(self):
        h = getattr(self, '_h', None)
        if h is not None and nat._lib is not None:
            nat._lib.astro_batch_destroy(h)
            self._h = None

    # ---- schedule / streams -------------------------------------------------------------------
    def set_schedule_origin(self, reload0, t0):
        """A game's tick counter 0 corresponds to (reload0, t0); see schedule.py."""
        if self.schedule is not None and self._origin == (reload0, t0):
            return
        self.schedule = Schedule(self.config, reload0, t0,
                                 max_ticks=nat.MAX_TICKS_WIDE if self.PL == nat.MAX_PLANETS_WIDE else nat.MAX_TICKS)
        self._origin = (reload0, t0)
        s = self.schedule
        nat.check(nat.lib().astro_set_schedule(self._h, s.fire_bits.ctypes.data_as(C.c_void_p), s.n_ticks, s.timeout_tick))

    def set_stream(self, seed=None, first_game=None, step=None):
        if seed is not None:
            self.seed = int(seed)
        if first_game is not None:
            self.first_game = int(first_game)
        if step is not None:
            self.step_index = int(step)
        nat.check(nat.lib().astro_set_stream(self._h, self.seed, self.first_game, self.step_index))

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    # ---- state in / out -------------------------------------------------------------------------
    def _split(self, index):
        index = np.asarray(index, dtype=np.int64)
        return index // nat.TILE, index % nat.TILE

    @property
    def bullet_buffer(self):
        """Which half of `self.bullets` holds the tile lists now (flips every tick)."""
        return int(nat.lib().astro_bullet_buffer(self._h))

    def _game_arrays(self, m, rows, episode=True):
        """Device tensors in the AstroGameArrays layout (float64, game-major) and the ctypes view of them."""
        torch = _torch()
        dev, f64, i32 = self.device, torch.float64, torch.int32
        t = dict(ships=torch.empty((m, self.S, 5), dtype=f64, device=dev),
                 planets=torch.empty((m, self.PL, 4), dtype=f64, device=dev),
                 bullets=torch.empty((m, max(rows, 1), 4), dtype=f64, device=dev),
                 n_planets=torch.empty((m,), dtype=i32, device=dev), n_bullets=torch.empty((m,), dtype=i32, device=dev),
                 tick=torch.empty((m,), dtype=i32, device=dev), finished=torch.empty((m,), dtype=torch.uint8, device=dev),
                 episode=torch.empty((m,), dtype=i32, device=dev) if episode else None)
        return t, self._arrays_struct(t, rows)

    @staticmethod
    def _arrays_struct(t, rows):
        ptr = lambda x: None if x is None else x.data_ptr()
        return nat.AstroGameArrays(ptr(t['ships']), ptr(t['planets']), ptr(t['bullets']), ptr(t['n_planets']), ptr(t['n_bullets']),
                                   ptr(t['tick']), ptr(t['finished']), ptr(t.get('episode')), int(rows), 0)

    def _index_tensor(self, index):
        torch = _torch()
        idx = np.asarray(index, dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= self.n_pad):
            raise IndexError('game index out of range 0..%d' % (self.n_pad - 1))
        return idx, torch.from_numpy(idx.astype(np.int32)).to(self.device)

    def set_arrays(self, ships, planets, n_planets, bullets=None, n_bullets=None, ticks=None, index=None,
                   episode=None, finished=None):
        """Load games from game-major host arrays: ships [m,S,5] (x,y,dx,dy,b), planets [m,PL,4],
        n_planets [m], bullets [m,<=K,4], n_bullets [m], ticks [m] (default 0) — ONE kernel
        (astro_import_games): the touched tiles' bullet lists are rebuilt on the device, every other
        game keeps its state."""
        torch = _torch()
        dev = self.device
        ships = np.ascontiguousarray(ships, dtype=np.float64)
        m = ships.shape[0]
        planets = np.ascontiguousarray(planets, dtype=np.float64)
        if planets.shape[1:] != (self.PL, 4):
            raise ValueError('planets must be [m, %d, 4] in a batch of %d planet slots' % (self.PL, self.PL))
        n_planets = np.asarray(n_planets, dtype=np.int64)
        n_bullets = np.zeros(m, dtype=np.int64) if n_bullets is None else np.asarray(n_bullets, dtype=np.int64)
        ticks = np.zeros(m, dtype=np.int64) if ticks is None else np.asarray(ticks, dtype=np.int64)
        if n_bullets.max(initial=0) > self.K:
            raise ValueError('a state holds more bullets than bullet_cap=%d' % self.K)
        if ticks.max(initial=0) > (nat.MAX_TICKS_WIDE if self.PL == nat.MAX_PLANETS_WIDE else nat.MAX_TICKS):
            raise ValueError('tick counter out of range')
        if m and not (np.abs(ships[:, :, 4]) <= nat.SINCOS_RANGE).all():
            raise ValueError('a bearing lies beyond the +-%d rad over which util.direction is reproduced' % nat.SINCOS_RANGE)
        rows = int(n_bullets.max(initial=0))
        bl = np.zeros((m, max(rows, 1), 4))
        if bullets is not None and rows:
            bl[:, :rows] = np.asarray(bullets, dtype=np.float64)[:, :rows]
        t = dict(ships=torch.from_numpy(ships).to(dev), planets=torch.from_numpy(planets).to(dev),
                 bullets=torch.from_numpy(bl).to(dev),
                 n_planets=torch.from_numpy(n_planets.astype(np.int32)).to(dev),
                 n_bullets=torch.from_numpy(n_bullets.astype(np.int32)).to(dev),
                 tick=torch.from_numpy(ticks.astype(np.int32)).to(dev),
                 finished=None if finished is None else torch.from_numpy(np.asarray(finished, dtype=np.uint8)).to(dev),
                 episode=None if episode is None else torch.from_numpy(np.asarray(episode, dtype=np.uint32).view(np.int32).copy()).to(dev))
        arrays = self._arrays_struct(t, rows)
        if index is None:
            idx_t = None
        else:
            idx, idx_t = self._index_tensor(index)
            if idx.size != m or np.unique(idx).size != m:
                raise ValueError('index must list %d distinct games' % m)
        nat.check(nat.lib().astro_import_games(self._h, None if idx_t is None else idx_t.data_ptr(), m, C.byref(arrays), self._stream()))
        _torch().cuda.current_stream(self.device).synchronize()   # the staging tensors die with this frame

    def set_states(self, states, index=None, ticks=None):
        """Load reference `State`s (core.py:15-18).  Without `ticks`, each state's (reload, t) must
        lie on this batch's schedule (true for anything produced by create + step)."""
        m, S, K = len(states), self.S, self.K
        ships = np.zeros((m, S, 5))
        planets = np.zeros((m, self.PL, 4))
        n_planets = np.zeros(m, dtype=np.int64)
        n_bullets = np.zeros(m, dtype=np.int64)
        kmax = max([np.shape(s.bullets.x)[0] for s in states] + [0])
        if kmax > K:
            raise ValueError('a state holds %d bullets, bullet_cap is %d' % (kmax, K))
        bullets = np.zeros((m, kmax, 4))
        tk = np.zeros(m, dtype=np.int64)
        for i, s in enumerate(states):
            if np.shape(s.ships.x)[0] != S:
                raise ValueError('cannot mix solo and duel games in one batch')
            ships[i, :, 0:2], ships[i, :, 2:4], ships[i, :, 4] = s.ships.x, s.ships.dx, s.ships.b
            p = np.shape(s.planets.x)[0]
            if not 1 <= p <= self.PL:
                raise ValueError('a state needs 1..%d planets (this batch has %d planet slots; at most %d with planet_slots=%d)'
                                 % (self.PL, self.PL, nat.MAX_PLANETS_WIDE, nat.MAX_PLANETS_WIDE))
            planets[i, :p, 0:2], planets[i, :p, 2:4] = s.planets.x, s.planets.dx
            n_planets[i] = p
            b = np.shape(s.bullets.x)[0]
            if b:
                bullets[i, :b, 0:2], bullets[i, :b, 2:4] = s.bullets.x, s.bullets.dx
            n_bullets[i] = b
            if ticks is None:
                k = self.schedule.tick_of(s.reload, s.t)
                if k is None:
                    raise ValueError('state %d: (reload=%r, t=%r) is not on the schedule of this batch; '
                                     'use set_schedule_origin() or pass ticks=' % (i, s.reload, s.t))
                tk[i] = k
        if ticks is not None:
            tk[:] = ticks
        self.set_arrays(ships, planets, n_planets, bullets, n_bullets, tk, index)

    def export_arrays(self, index=None, rows=None):
        """Games `index` (default: all) as game-major float64 DEVICE tensors, one kernel (astro_export_games)."""
        if index is None:
            m, idx_t = self.n, None
        else:
            idx, idx_t = self._index_tensor(index)
            m = idx.size
        rows = self.K if rows is None else int(rows)
        t, arrays = self._game_arrays(m, rows)
        nat.check(nat.lib().astro_export_games(self._h, None if idx_t is None else idx_t.data_ptr(), m, C.byref(arrays), self._stream()))
        if idx_t is not None:
            _torch().cuda.current_stream(self.device).synchronize()   # the index tensor dies with this frame
        return t

    def get_arrays(self, index=None):
        """Whole batch (or the listed games) as game-major float64 host arrays (the inverse of set_arrays)."""
        t = self.export_arrays(index)
        K = self.K
        return dict(ships=t['ships'].cpu().numpy(), planets=t['planets'].cpu().numpy(), bullets=t['bullets'].cpu().numpy()[:, :K],
                    n_bullets=t['n_bullets'].cpu().numpy(), n_planets=t['n_planets'].cpu().numpy(),
                    finished=t['finished'].cpu().numpy().astype(bool), tick=t['tick'].cpu().numpy().astype(np.int64),
                    episode=t['episode'].cpu().numpy().view(np.uint32).copy())

    def get_states(self, indices):
        """Reference `State`s (or None for finished games) of the listed games only — the read path of
        logs.GameRecorder and of the drop-in core.play."""
        a = self.get_arrays(np.asarray(indices, dtype=np.int64).reshape(-1))
        out = []
        for j in range(a['tick'].shape[0]):
            if a['finished'][j]:
                out.append(None)
                continue
            nb, npl, tick = int(a['n_bullets'][j]), int(a['n_planets'][j]), int(a['tick'][j])
            sh, pl, bl = a['ships'][j], a['planets'][j], a['bullets'][j]
            out.append(core.State(
                ships=core.Bodies(x=sh[:, 0:2].copy(), dx=sh[:, 2:4].copy(), b=sh[:, 4].copy()),
                planets=core.Bodies(x=pl[:npl, 0:2].copy(), dx=pl[:npl, 2:4].copy(), b=None),
                bullets=core.Bodies(x=bl[:nb, 0:2].copy(), dx=bl[:nb, 2:4].copy(), b=None),
                reload=float(self.schedule.reload[tick]), t=float(self.schedule.t[tick])))
        return out

    def to_state(self, i):
        """Game i as a reference `State` (float64 arrays), or None when the game has ended."""
        return self.get_states([int(i)])[0]

    # ---- reset pool ------------------------------------------------------------------------------
    def set_reset_pool(self, states):
        """Initial states (built by core.create) that finished games are re-created from."""
        torch = _torch()
        M, S = len(states), self.S
        ships = np.zeros((M, S, 5), dtype=self.np_rdtype)
        planets = np.zeros((M, self.PL, 4), dtype=self.np_rdtype)
        npl = np.zeros(M, dtype=np.int32)
        for i, s in enumerate(states):
            ships[i, :, 0:2], ships[i, :, 2:4], ships[i, :, 4] = s.ships.x, s.ships.dx, s.ships.b
            p = np.shape(s.planets.x)[0]
            planets[i, :p, 0:2], planets[i, :p, 2:4] = s.planets.x, s.planets.dx
            npl[i] = p
        self.set_reset_pool_arrays(ships, planets, npl)

    def set_reset_pool_arrays(self, ships, planets, n_planets):
        torch = _torch()
        dev = self.device
        if np.shape(planets)[1:] != (self.PL, 4):
            raise ValueError('reset pool planets must be [M, %d, 4] in a batch of %d planet slots' % (self.PL, self.PL))
        self._pool = (torch.from_numpy(np.ascontiguousarray(ships, dtype=self.np_rdtype)).to(dev),
                      torch.from_numpy(np.ascontiguousarray(planets, dtype=self.np_rdtype)).to(dev),
                      torch.from_numpy(np.ascontiguousarray(n_planets, dtype=np.int32)).to(dev))
        pool = nat.AstroResetPool(self._pool[0].data_ptr(), self._pool[1].data_ptr(), self._pool[2].data_ptr(),
                                  self._pool[0].shape[0], 0)
        nat.check(nat.lib().astro_set_reset_pool(self._h, C.byref(pool)))

    def create_on_device(self, seeds):
        """`core.create` (core.py:86-135) for every seed, on the device: returns cuda tensors
        (ships [m,S,5], planets [m,PL,4], n_planets int32 [m]) in the batch precision, bit-identical
        to core.create(config._replace(seed=s)) (rounded to float32 in the float32 build)."""
        torch = _torch()
        seeds = torch.as_tensor(np.asarray(seeds, dtype=np.uint32).astype(np.int64), dtype=torch.int64).to(torch.int32) \
            if not isinstance(seeds, torch.Tensor) else seeds
        seeds = seeds.to(device=self.device, dtype=torch.int32).contiguous()   # same 32 bits as uint32
        m = int(seeds.numel())
        ships = torch.empty((m, self.S, 5), dtype=self.rdtype, device=self.device)
        planets = torch.empty((m, self.PL, 4), dtype=self.rdtype, device=self.device)
        n_planets = torch.empty((m,), dtype=torch.int32, device=self.device)
        c = self.config
        cc = nat.AstroCreateConfig(float(c.inner_ship_position), float(c.outer_ship_position), float(c.planet_orbit),
                                   int(c.max_planets), 0)
        nat.check(nat.lib().astro_create_games(self._h, C.byref(cc), seeds.data_ptr(), m, ships.data_ptr(),
                                               planets.data_ptr(), n_planets.data_ptr(), self._stream()))
        return ships, planets, n_planets

    def set_reset_pool_on_device(self, size, skip=0):
        """Reset pool of `size` fresh games created ON THE DEVICE from the seeds of
        core.generate_configs(config) number skip .. skip+size-1 (same pool as pool.make_pool for
        skip=0).  Call again with a larger `skip` between rollouts for a pool that never repeats."""
        from . import rng
        ships, planets, n_planets = self.create_on_device(rng.config_seeds(self.config.seed, size, skip))
        self._pool = (ships, planets, n_planets)
        pool = nat.AstroResetPool(ships.data_ptr(), planets.data_ptr(), n_planets.data_ptr(), int(size), 0)
        nat.check(nat.lib().astro_set_reset_pool(self._h, C.byref(pool)))

    # ---- fresh games without a pool -----------------------------------------------------------------
    def enable_fresh_games(self, quota=48, skip=0):
        """Pool-free re-creation (astro_fresh_games_enable): every game that ends under auto_reset is re-created from the
        NEXT config of core.generate_configs(config) — core.create on the device, seeds from the library's host MT19937 —
        so no start state is ever re-used (core.py:77-135, rl.py:350,374).  `quota` pre-created games per 32-game tile
        between refills; `skip`: stream position to start from."""
        c = self.config
        cc = nat.AstroCreateConfig(float(c.inner_ship_position), float(c.outer_ship_position), float(c.planet_orbit),
                                   int(c.max_planets), 0)
        nat.check(nat.lib().astro_fresh_games_enable(self._h, C.byref(cc), int(c.seed) & 0xFFFFFFFF, int(skip), int(quota), self._stream()))
        self._fresh = True

    def fresh_positions(self):
        """(positions int64 [n], tile_used int64 [n_tiles], cursor): the generate_configs stream position of each game's
        current episode, the records each tile used since the last refill, the positions handed out so far."""
        torch = _torch()
        pos = torch.empty((self.n_pad,), dtype=torch.int32, device=self.device)
        used = torch.empty((self.n_tiles,), dtype=torch.int32, device=self.device)
        cur = C.c_int64(0)
        nat.check(nat.lib().astro_fresh_games_positions(self._h, pos.data_ptr(), used.data_ptr(), C.byref(cur), self._stream()))
        return (pos.cpu().numpy().view(np.uint32)[:self.n].astype(np.int64), used.cpu().numpy().view(np.uint32).astype(np.int64), int(cur.value))

    def reset_done(self):
        """Re-create every finished game from the pool (entry = pick(seed, game, current step))."""
        nat.check(nat.lib().astro_reset_done(self._h, self._stream()))
        if self.n != self.n_pad:
            self.meta[self.n:] = 1 << 13      # the padding slots of the last tile stay finished (empty)

    def reset_all(self):
        """(Re)start every game from the pool: game g starts as pool[pick(seed, g, key 0)] — or, in fresh-game mode, from
        the next n games of the generate_configs stream."""
        if getattr(self, '_fresh', False):
            nat.check(nat.lib().astro_fresh_games_reset_all(self._h, self._stream()))
            self.step_index = 0
            if self.n != self.n_pad:
                self.meta[self.n:] = 1 << 13
            return
        self.meta.fill_(1 << 13)
        self.episode.fill_(-1)
        self.set_stream(step=0)
        self.reset_done()

    # ---- the tick ---------------------------------------------------------------------------------
    def step(self, actions=None, auto_reset=False, stats=True, want_reward=True):
        """One `core.step` for every game.

        actions -- None (device counter stream, rng.actions), or uint8 cuda tensor / array
                   [n, S] of control codes 0..5.
        returns -- (reward f32 [n,S] or None, done u8 [n], events u8 [n]): views of buffers that
                   the next step overwrites.
        """
        torch = _torch()
        if actions is None:
            a_ptr = None
        else:
            if not isinstance(actions, torch.Tensor):
                actions = np.ascontiguousarray(actions)
                if actions.size and (actions.min() < 0 or actions.max() > 5):
                    raise ValueError('control codes must be 0..5 (core.py:220-227)')   # (device tensors: ASTRO_EV_BAD_CONTROL)
                actions = torch.from_numpy(actions.astype(np.uint8))
            actions = actions.to(device=self.device, dtype=torch.uint8).reshape(-1, self.S)
            if actions.shape[0] == self.n_pad and actions.is_contiguous():
                a_ptr = actions.data_ptr()
            else:
                if actions.shape[0] != self.n:
                    raise ValueError('actions must have shape [%d, %d]' % (self.n, self.S))
                self._actions[:self.n].copy_(actions)
                a_ptr = self._actions.data_ptr()
        flags = (nat.TICK_AUTO_RESET if auto_reset else 0) | (0 if stats else nat.TICK_NO_STATS) | self.tick_flags
        nat.check(nat.lib().astro_tick(self._h, a_ptr, self._reward.data_ptr() if want_reward else None,
                                       self._done.data_ptr(), self._events.data_ptr(), flags, self._stream()))
        self.step_index += 1
        n = self.n
        return (self._reward[:n] if want_reward else None), self._done[:n], self._events[:n]

    # ---- compact host traffic: one control byte per game, three event bit planes per tick ------------
    @staticmethod
    def pack_controls(actions):
        """[..., 2] control codes 0..5 -> [...] uint8, ship 0 in bits 0-2 and ship 1 in bits 3-5 (TICK_PACKED_CONTROLS)."""
        a = actions
        if hasattr(a, 'numpy') or hasattr(a, 'device'):
            return (a[..., 0] | (a[..., 1] << 3)).to(a.dtype)
        a = np.asarray(a)
        return (a[..., 0] | (a[..., 1] << 3)).astype(np.uint8)

    def planes_shape(self, n_ticks=None):
        """Shape of an int32 event-plane buffer (TICK_EVENT_PLANES): [3, n_tiles] per tick."""
        return (3, self.n_tiles) if n_ticks is None else (int(n_ticks), 3, self.n_tiles)

    def unpack_event_planes(self, planes):
        """int32 / uint32 [..., 3, n_tiles] bit planes (ended / ship 0 hit / ship 1 hit) -> uint8 events [..., n] with
        the ASTRO_EV_HIT0 / HIT1 / TIMEOUT bits of the byte-per-game form (host side, numpy)."""
        p = np.ascontiguousarray(planes.cpu().numpy() if hasattr(planes, 'cpu') else planes).view(np.uint32)
        bits = np.unpackbits(p.view(np.uint8).reshape(p.shape + (4,)), axis=-1, bitorder='little').reshape(p.shape[:-1] + (-1,))
        done, h0, h1 = bits[..., 0, :], bits[..., 1, :], bits[..., 2, :]
        ev = h0 | (h1 << 1) | ((done & (1 - (h0 | h1))) << 2)
        return ev[..., :self.n].astype(np.uint8)

    def _io_flags(self, auto_reset, stats, packed, planes):
        if packed and self.S != 2:
            raise ValueError('packed controls are for duel games')
        return ((nat.TICK_AUTO_RESET if auto_reset else 0) | (0 if stats else nat.TICK_NO_STATS) | self.tick_flags
                | (nat.TICK_PACKED_CONTROLS if packed else 0) | (nat.TICK_EVENT_PLANES if planes else 0))

    def step_many(self, n_ticks, actions=None, events=None, reward=None, done=None, auto_reset=False, stats=True,
                  packed=False, planes=False):
        """`n_ticks` consecutive `step()`s in as few launches as possible (astro_tick_many): the ticks of a tile run
        back to back inside a launch, state going from one tick to the next through L2.  For loops whose controls
        do not depend on the states inside the block (replays, random exploration, the counter stream).

        actions -- None (device counter stream) or uint8 cuda tensor [n_ticks, n_pad, S] ([n_ticks, n_pad] with packed=True)
        events / reward / done -- optional cuda tensors [n_ticks, n_pad] (uint8; int32 [n_ticks, 3, n_tiles] with planes=True)
                   / [n_ticks, n_pad, S] (float32) / [n_ticks, n_pad] (uint8) receiving every tick's outputs"""
        torch = _torch()
        T = int(n_ticks)

        def ptr(x, shape, dtype, name):
            if x is None:
                return None
            if tuple(x.shape) != shape or x.dtype != dtype or not x.is_contiguous() or x.device != self.device:
                raise ValueError('%s must be a contiguous %s cuda tensor %r' % (name, dtype, shape))
            return x.data_ptr()
        flags = self._io_flags(auto_reset, stats, packed, planes)
        a_shape = (T, self.n_pad) if packed else (T, self.n_pad, self.S)
        e_shape, e_dtype = ((T, 3, self.n_tiles), torch.int32) if planes else ((T, self.n_pad), torch.uint8)
        nat.check(nat.lib().astro_tick_many(
            self._h, ptr(actions, a_shape, torch.uint8, 'actions'),
            ptr(reward, (T, self.n_pad, self.S), torch.float32, 'reward'), ptr(done, (T, self.n_pad), torch.uint8, 'done'),
            ptr(events, e_shape, e_dtype, 'events'), T, flags, self._stream()))
        self.step_index += T

    def step_many_raw(self, actions_ptr, events_ptr, n_ticks, flags):
        """Bench path: a bare astro_tick_many with caller-held device pointers (or 0)."""
        nat.check(nat.lib().astro_tick_many(self._h, actions_ptr or None, None, None, events_ptr or None, int(n_ticks), flags,
                                            self._stream()))
        self.step_index += int(n_ticks)

    def step_raw(self, actions_ptr, flags):
        """Bench path: a bare astro_tick with a caller-held device pointer (or 0), events only."""
        nat.check(nat.lib().astro_tick(self._h, actions_ptr or None, None, None, self._events.data_ptr(), flags,
                                       self._stream()))
        self.step_index += 1

    def step_host(self, actions_host, events_host, reward_host=None, done_host=None, auto_reset=False, stats=True,
                  packed=False, planes=False):
        """End-to-end tick with HOST buffers (torch pinned tensors or numpy arrays): copies the
        actions in, ticks, copies events (and reward/done if given) out, synchronises.
        packed=True: actions_host is uint8 [n_pad] (pack_controls); planes=True: events_host is int32 [3, n_tiles]
        (unpack_event_planes) — 1.4 bytes per game and tick through host memory instead of 3."""
        def ptr(x):
            if x is None:
                return None
            return x.data_ptr() if hasattr(x, 'data_ptr') else x.ctypes.data
        flags = self._io_flags(auto_reset, stats, packed, planes)
        for x, nbytes in ((actions_host, self.n_pad * (1 if packed else self.S)), (events_host, self.n_tiles * 12 if planes else self.n_pad)):
            if x is not None and (x.numel() * x.element_size() if hasattr(x, 'numel') else x.nbytes) < nbytes:
                raise ValueError('host buffer too small: need %d bytes' % nbytes)
        nat.check(nat.lib().astro_tick_host(self._h, ptr(actions_host), ptr(reward_host), ptr(done_host),
                                            ptr(events_host), flags, self._stream()))
        self.step_index += 1

    def step_host_begin(self, actions_host, events_host, auto_reset=False, stats=True, packed=False, planes=False, stream=None):
        """step_host without the wait: enqueues copy in, tick, copy out on `stream` (a torch.cuda.Stream; default: the
        current one) and returns; step_host_end() blocks until the events are on the host.  For a closed loop over
        several batches on their own streams (see astro_tick_host_begin)."""
        def ptr(x):
            return x.data_ptr() if hasattr(x, 'data_ptr') else x.ctypes.data
        flags = self._io_flags(auto_reset, stats, packed, planes)
        st = self._stream() if stream is None else C.c_void_p(stream.cuda_stream)
        nat.check(nat.lib().astro_tick_host_begin(self._h, ptr(actions_host), ptr(events_host), flags, st))
        self.step_index += 1

    def step_host_end(self):
        nat.check(nat.lib().astro_tick_host_end(self._h))

    def rollout_host(self, actions_host, events_host, auto_reset=False, stats=True, packed=False, planes=False):
        """Pipelined end-to-end rollout with HOST buffers: actions_host uint8 [T, n_pad, S] ([T, n_pad] with
        packed=True), events_host uint8 [T, n_pad] (int32 [T, 3, n_tiles] with planes=True) — pinned torch tensors
        or numpy arrays.  Every tick's controls are copied in and its events copied out; copies of neighbouring
        ticks overlap the tick kernel."""
        def ptr(x):
            return x.data_ptr() if hasattr(x, 'data_ptr') else x.ctypes.data
        def nbytes(x):
            return x.numel() * x.element_size() if hasattr(x, 'numel') else x.nbytes
        T = int(actions_host.shape[0])
        need_a, need_e = T * self.n_pad * (1 if packed else self.S), T * (self.n_tiles * 12 if planes else self.n_pad)
        if nbytes(actions_host) != need_a or nbytes(events_host) < need_e:
            raise ValueError('need %d bytes of controls and %d bytes of events for %d ticks' % (need_a, need_e, T))
        flags = self._io_flags(auto_reset, stats, packed, planes)
        nat.check(nat.lib().astro_rollout_host(self._h, ptr(actions_host), ptr(events_host), T, flags, self._stream()))
        self.step_index += T

    # ---- observations ----------------------------------------------------------------------------
    def observe(self, n_rows=None, out=None, shared=False):
        """Feature batch float32, rows = planets, bullets, then -1 padding (rl.py:43-99).

        shared=False -- [n, S, n_rows, D]: obs[g, k] is game g seen by ship k (core.roll_ships).
        shared=True  -- [n, n_rows, D]: ship 0's view only; ship 1's view is the same block with
                        the ship column groups exchanged (see rl.ValueNetwork.forward_both)."""
        torch = _torch()
        if n_rows is None:
            n_rows = -(-(self.PL + self.K) // 4) * 4
        shape = (self.n_pad, n_rows, self.D) if shared else (self.n_pad, self.S, n_rows, self.D)
        if out is None:
            out = torch.empty(shape, dtype=torch.float32, device=self.device)
        elif tuple(out.shape) != shape or out.dtype != torch.float32 or not out.is_contiguous():
            raise ValueError('out must be a contiguous float32 tensor %r' % (shape,))
        fn = nat.lib().astro_observe_shared if shared else nat.lib().astro_observe
        nat.check(fn(self._h, out.data_ptr(), n_rows, self._stream()))
        return out[:self.n]

    # ---- scripted bots ----------------------------------------------------------------------------
    def script_controls(self, out=None, avoid_distance=0.1, avoid_threshold=0.45):
        """`script.ScriptBot` (script.py:13-91) for every ship of every game, each from its own
        perspective: uint8 cuda tensor [n, S] of control codes, ready to be passed to step()."""
        torch = _torch()
        if out is None:
            out = torch.empty((self.n_pad, self.S), dtype=torch.uint8, device=self.device)
        elif out.shape[0] != self.n_pad or out.dtype != torch.uint8 or not out.is_contiguous():
            raise ValueError('out must be a contiguous uint8 tensor [%d, %d]' % (self.n_pad, self.S))
        nat.check(nat.lib().astro_script_controls(self._h, float(avoid_distance), float(avoid_threshold), out.data_ptr(),
                                                  self._stream()))
        return out

    # ---- value network on the device --------------------------------------------------------------
    def set_policy(self, net):
        """Load a `rl.ValueNetwork` (or any module with the reference's layers f0, f[0..1], v[0..1],
        v0; rl.py:140-152) into the fused policy kernel."""
        parts = []
        for layer in (net.f0, net.f[0], net.f[1], net.v[0], net.v[1], net.v0):
            parts += [layer.weight.detach().float().cpu().numpy().ravel(), layer.bias.detach().float().cpu().numpy().ravel()]
        w = np.ascontiguousarray(np.concatenate(parts), dtype=np.float32)
        self.policy_nout = int(net.v0.weight.shape[0])
        nat.check(nat.lib().astro_policy_set_weights(self._h, w.ctypes.data_as(C.c_void_p), int(w.size), self.policy_nout))

    def value_forward(self, features, out=None):
        """`rl.ValueNetwork.forward` (rl.py:140-165) of the loaded network on a feature batch — float32 cuda
        [..., rows, D] as `observe()` / `get_features_batch` give it — in one tensor-core kernel (astro_value_forward);
        inference only.  Returns float32 [..., nout]."""
        torch = _torch()
        if not (features.is_cuda and features.dtype == torch.float32 and features.dim() >= 2):
            raise ValueError('value_forward needs a float32 cuda tensor [..., rows, D]')
        if features.shape[-1] != 1 + 5 * self.S + 4:
            raise ValueError('feature width %d does not match this batch (%d)' % (features.shape[-1], 1 + 5 * self.S + 4))
        x = features.contiguous()
        lead, rows = x.shape[:-2], int(x.shape[-2])
        n = 1
        for d in lead:
            n *= int(d)
        nout = self.policy_nout
        if out is None:
            out = torch.empty(tuple(lead) + (nout,), dtype=torch.float32, device=x.device)
        nat.check(nat.lib().astro_value_forward(self._h, x.data_ptr(), n, rows, out.data_ptr(), self._stream()))
        return out

    def policy_controls(self, out=None, q_out=None, ships=None):
        """Greedy controls argmax_a Q(s, a) of the loaded network for every ship of every game, each
        from its own perspective (rl.QBot, rl.py:168-200) — features and network fused in one
        kernel.  out: uint8 cuda [n_pad, S] (only the listed `ships` columns are written);
        q_out: optional float32 cuda [n_pad, S, nout] receiving the network outputs."""
        torch = _torch()
        if out is None:
            out = torch.full((self.n_pad, self.S), 2, dtype=torch.uint8, device=self.device)
        mask = sum(1 << int(k) for k in (range(self.S) if ships is None else ships))
        nat.check(nat.lib().astro_policy_controls(self._h, out.data_ptr(), None if q_out is None else q_out.data_ptr(),
                                                  mask, self._stream()))
        return out

    def explore_controls(self, actions, state=None, t_in=1.0, t_out=0.1, seed=0, ships=None):
        """`rl.EpsilonGreedy` (rl.py:10-30) laid over `actions` (uint8 cuda [n_pad, S], e.g. from policy_controls) the way
        `rl.QBotTrainer.__call__` does (rl.py:249-258): where a ship's random policy is active its control replaces the
        greedy one.  `state`: int32 cuda [n_pad, S] exploration state (created zeroed when None); returns it."""
        torch = _torch()
        if state is None:
            state = torch.zeros((self.n_pad, self.S), dtype=torch.int32, device=self.device)
        mask = sum(1 << int(k) for k in (range(self.S) if ships is None else ships))
        nat.check(nat.lib().astro_explore_controls(self._h, float(t_in), float(t_out), int(seed) & 0xFFFFFFFF, state.data_ptr(),
                                                   actions.data_ptr(), mask, self._stream()))
        return state

    def set_exploration(self, t_in=1.0, t_out=0.1, seed=0, state=None):
        """Parameters and state of the 'explore' bots of rollout_device (the greedy network with rl.EpsilonGreedy laid
        over it, rl.QBotTrainer's acting policy; the reference's t_in = 1.0, t_out = 0.1).  Returns the state tensor."""
        torch = _torch()
        if state is None:
            state = torch.zeros((self.n_pad, self.S), dtype=torch.int32, device=self.device)
        self._explore_state = state
        nat.check(nat.lib().astro_set_exploration(self._h, float(t_in), float(t_out), int(seed) & 0xFFFFFFFF, state.data_ptr()))
        return state

    # ---- whole game loops on the device -------------------------------------------------------------
    def rollout_device(self, n_ticks, bots=('stream', 'stream'), auto_reset=True, stats=True, avoid_distance=0.1,
                       avoid_threshold=0.45, record=None):
        """`n_ticks` of the play loop (core.play, core.py:377-410; rl.train's games, rl.py:350-374) for
        every game without the host between ticks.  bots: one of 'stream' (counter-stream random
        controls, both ships), 'script' (script.ScriptBot), 'policy' (greedy network loaded with
        set_policy), 'explore' (that network with rl.EpsilonGreedy laid over it: set_exploration), 'nothing'
        (script.NothingBot) per ship.  Outcomes accumulate in stats().
        record: a RecordRing (record_ring()) that receives every tick's controls, events and — if it holds them — the
        observations (astro_rollout_device_record); the results are the same as without it."""
        if isinstance(bots, str):
            bots = (bots,) * self.S
        modes = [nat.BOT_MODES[b] for b in bots] + [0]
        flags = (nat.TICK_AUTO_RESET if auto_reset else 0) | (0 if stats else nat.TICK_NO_STATS) | self.tick_flags
        n = int(n_ticks)
        if record is None:
            nat.check(nat.lib().astro_rollout_device(self._h, n, modes[0], modes[1], float(avoid_distance),
                                                     float(avoid_threshold), self._actions.data_ptr(), self._events.data_ptr(),
                                                     flags, self._stream()))
        else:
            if (record.n_pad, record.S) != (self.n_pad, self.S) or record.device != self.device:
                raise ValueError('the ring was made for another batch layout (record_ring of this batch)')
            nat.check(nat.lib().astro_rollout_device_record(self._h, n, modes[0], modes[1], float(avoid_distance),
                                                            float(avoid_threshold), self._actions.data_ptr(), C.byref(record._ring),
                                                            flags, self._stream()))
            record._recorded(self.step_index, n)
        self.step_index += n

    def record_ring(self, ticks, observations=True, n_rows=None):
        """A RecordRing of `ticks` rows for rollout_device(..., record=ring): per tick the controls, events and (observations=True)
        ship 0's observation of the state before the tick (n_rows as observe(); default the smallest multiple of 4 that holds
        the planet slots and bullet_cap).  A rollout_device call records at most ticks - 1 ticks."""
        return RecordRing(self, ticks, observations, n_rows)

    # ---- n-step replay ingestion ---------------------------------------------------------------------
    def nstep_experiences(self, events, carry=None, n_steps=100, discount=0.995):
        """`rl.QBotTrainer.reward` (rl.py:303-328) for every bot over the logged ticks `events` (uint8 cuda [T, n_pad]): which
        (state, action) pairs enter the replay buffer, with which discounted reward / discount / new state.  Returns
        (reward f32, discount f32, next i32) cuda tensors [n_steps + T, n_pad, S] (row n_steps + t = the pair of tick t; see
        astro_nstep_experiences) and the carry tensor int32 [n_pad, S] (pass it to the next window's call)."""
        torch = _torch()
        T = int(events.shape[0])
        if tuple(events.shape) != (T, self.n_pad) or events.dtype != torch.uint8 or not events.is_contiguous():
            raise ValueError('events must be a contiguous uint8 cuda tensor [T, %d]' % self.n_pad)
        if carry is None:
            carry = torch.zeros((self.n_pad, self.S), dtype=torch.int32, device=self.device)
        shape = (int(n_steps) + T, self.n_pad, self.S)
        rew = torch.zeros(shape, dtype=torch.float32, device=self.device)
        dis = torch.zeros(shape, dtype=torch.float32, device=self.device)
        nxt = torch.full(shape, -3, dtype=torch.int32, device=self.device)
        nat.check(nat.lib().astro_nstep_experiences(self._h, events.data_ptr(), T, int(n_steps), float(discount), carry.data_ptr(),
                                                    rew.data_ptr(), dis.data_ptr(), nxt.data_ptr(), self._stream()))
        return rew, dis, nxt, carry

    # ---- statistics ------------------------------------------------------------------------------
    def stats_tensor(self, clear=False):
        """Device int64 [12] counters (see _native.STAT_NAMES) — the input of the NCCL all-reduce."""
        nat.check(nat.lib().astro_stats(self._h, self._stats.data_ptr(), int(clear), self._stream()))
        return self._stats

    def stats_peer_init(self, dist):
        """Maps the exchange buffers of all ranks of `dist`'s default group (one node, one GPU per rank) for
        stats_allreduce: CUDA IPC handles travel through dist.all_gather.  Collective, and collective-safe: a rank
        whose create / open step fails still takes part in every exchange, and ALL ranks then return False (the
        caller keeps NCCL); True = every rank has mapped every buffer."""
        torch = _torch()
        rank, world = dist.get_rank(), dist.get_world_size()
        handle = (C.c_uint8 * 64)()
        err = None
        try:
            nat.check(nat.lib().astro_stats_peer_create(self._h, rank, world, handle))
        except nat.AstroError as exc:
            err = str(exc)
        mine = torch.tensor(list(handle) + [0 if err else 1], dtype=torch.uint8, device=self.device)
        everyone = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(everyone, mine)
        got = torch.stack(everyone).cpu().numpy()
        if err is None and got[:, 64].all():
            try:
                nat.check(nat.lib().astro_stats_peer_open(self._h, got[:, :64].tobytes()))
            except nat.AstroError as exc:
                err = str(exc)
        elif err is None:
            err = 'another rank could not create its exchange buffer'
        ok = torch.tensor([0.0 if err else 1.0], device=self.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)     # (also the barrier: nobody stores into a buffer that is not mapped and cleared)
        self.peer_error = err
        self._peer_ready = bool(float(ok) > 0)
        return self._peer_ready

    def stats_allreduce(self, clear=False):
        """The counters summed over all ranks, on the device (int64 [N_STATS]): ONE kernel per rank over peer memory
        (astro_stats_allreduce); collective, after stats_peer_init."""
        if not getattr(self, '_peer_ready', False):
            raise nat.AstroError('stats_allreduce: stats_peer_init has not succeeded on every rank')
        nat.check(nat.lib().astro_stats_allreduce(self._h, self._stats.data_ptr(), int(clear), self._stream()))
        return self._stats

    def stats(self, clear=False):
        v = self.stats_tensor(clear).cpu().numpy()
        return dict(zip(nat.STAT_NAMES, (int(x) for x in v)))

    @property
    def launches(self):
        return int(nat.lib().astro_launch_count(self._h))


class RecordRing:
    """The per-tick log of device rollouts (AstroRecordRing, astro_rollout_device_record) — what rl.QBotTrainer keeps per bot to
    build its Experiences (rl.py:212-228) — as cuda tensors, row = stream step % ticks:
      controls      uint8 [ticks, n_pad, S]                the control each ship flew on that tick
      events        uint8 [ticks, n_pad]                   that tick's ASTRO_EV_* byte (what step() returns as events)
      observations  float32 [ticks, n_pad, n_rows, D]      ship 0's observation (observe(shared=True)) of the state before the
                    or None                                tick; a rollout call also records the state after its last tick
    Rows of stream steps first .. end - 1 hold an unbroken history (a rollout that does not continue where the last one ended
    starts a new one)."""

    def __init__(self, games, ticks, observations=True, n_rows=None):
        torch = _torch()
        R = int(ticks)
        if R < 2:
            raise ValueError('a ring needs at least 2 rows')
        self.ticks, self.n_pad, self.S, self.D, self.device = R, games.n_pad, games.S, games.D, games.device
        self.n_rows = -(-(games.PL + games.K) // 4) * 4 if n_rows is None else int(n_rows)
        self.controls = torch.zeros((R, self.n_pad, self.S), dtype=torch.uint8, device=self.device)
        self.events = torch.zeros((R, self.n_pad), dtype=torch.uint8, device=self.device)
        self.observations = (torch.zeros((R, self.n_pad, self.n_rows, self.D), dtype=torch.float32, device=self.device)
                             if observations else None)
        self._ring = nat.AstroRecordRing(R, self.n_rows, self.controls.data_ptr(), self.events.data_ptr(),
                                         None if self.observations is None else self.observations.data_ptr())
        self.first = self.end = None

    def _recorded(self, s0, n):
        if self.end != s0:
            self.first = s0
        self.end = s0 + n
        # row end % R now holds the observation of step `end`: the controls / events of step end - R are gone with it
        self.first = max(self.first, self.end + 1 - self.ticks)

    def _rows(self, t0, n):
        """Ring rows of stream steps t0 .. t0 + n - 1 as an index tensor."""
        torch = _torch()
        return (torch.arange(t0, t0 + n, device=self.device) % self.ticks)

    def window_events(self, n_ticks):
        """The events of the last `n_ticks` recorded ticks, contiguous uint8 [n_ticks, n_pad]: the `events` input of
        BatchedGames.nstep_experiences (a view when the window does not wrap around the ring)."""
        T = int(n_ticks)
        if self.end is None or T > self.end - self.first:
            raise ValueError('the ring holds %d recorded ticks, not %d' % (0 if self.end is None else self.end - self.first, T))
        a = (self.end - T) % self.ticks
        if a + T <= self.ticks:
            return self.events[a:a + T]
        return self.events[self._rows(self.end - T, T)]

    def _view_of(self, rows, game, ship):
        """Observation rows [E, n_rows, D] of (ring row, game) seen by `ship`: ship 1 sees ship 0's block with the two ship column
        groups exchanged (core.roll_ships, core.py:306-327; equal to observe(shared=False)[:, 1])."""
        torch = _torch()
        x = self.observations[rows, game]
        if self.S == 2:
            swap = torch.tensor([0, 6, 7, 8, 9, 10, 1, 2, 3, 4, 5, 11, 12, 13, 14], device=self.device)
            x = torch.where((ship == 1)[:, None, None], x[..., swap], x)
        return x

    def experiences(self, reward, discount, nxt, n_steps):
        """The Experiences (rl.py:212-228) of one nstep_experiences call over the last window of this ring
        (nstep_experiences(ring.window_events(T), ...)): one entry per (state, action) pair it flushed, as cuda tensors
          features       float32 [E, n_rows, D]  the bot's own view of the pair's state (ship 1: column groups exchanged)
          action         uint8 [E]               the control it flew
          reward, discount float32 [E]           the n-step reward and discount
          next_features  float32 [E, n_rows, D]  the bot's view of the new state; all -1 (a finished game) when terminal
          terminal       bool [E]                the new state is None (the game ended)
          game, ship     int64 [E]
          tick           int64 [E]               the stream step of the pair's tick
        Pairs carried from earlier windows refer to their ticks, so the ring must hold n_steps ticks before the window as well
        as the window and the state after it: ticks >= n_steps + T + 1."""
        torch = _torch()
        if self.observations is None:
            raise ValueError('experiences need a ring that records observations')
        n_steps = int(n_steps)
        T = int(nxt.shape[0]) - n_steps
        if tuple(nxt.shape) != (n_steps + T, self.n_pad, self.S) or T < 0:
            raise ValueError('nxt must be [n_steps + T, %d, %d] as nstep_experiences returns it' % (self.n_pad, self.S))
        if self.ticks < n_steps + T + 1:
            raise ValueError('a ring of %d rows cannot hold the %d ticks before a window of %d ticks, the window and the state '
                             'after it: it needs ticks >= n_steps + T + 1 = %d' % (self.ticks, n_steps, T, n_steps + T + 1))
        if self.end is None or T > self.end - self.first:
            raise ValueError('the ring does not hold the last %d ticks' % T)
        s0 = self.end - T
        row, game, ship = (nxt >= -1).nonzero(as_tuple=True)
        tick = s0 + row - n_steps
        if tick.numel() and int(tick.min()) < self.first:
            raise ValueError('a carried pair refers to stream step %d, before the ring\'s history (from %d)' % (int(tick.min()), self.first))
        at = tick % self.ticks
        nx = nxt[row, game, ship]
        terminal = nx == -1
        next_features = self._view_of((s0 + nx.clamp(min=0)) % self.ticks, game, ship)
        next_features = torch.where(terminal[:, None, None], torch.full_like(next_features, -1.0), next_features)
        return dict(features=self._view_of(at, game, ship), action=self.controls[at, game, ship],
                    reward=reward[row, game, ship], discount=discount[row, game, ship], next_features=next_features,
                    terminal=terminal, game=game, ship=ship, tick=tick)
