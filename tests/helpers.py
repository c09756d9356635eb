"""Shared helpers of the parity tests: golden loaders, pools, oracle <-> BatchedGames glue."""
import itertools as it
import json
import os
import re
import shutil
import subprocess

import numpy as np

from astro_b200 import core, rng
from oracle import astro_oracle as ao

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool((bits(a) == bits(b)).all())


def config_from(d):
    return core.Config(**{k: d[k] for k in core.Config._fields})


def load_traj():
    z = np.load(os.path.join(G, 'traj.npz'))
    meta = json.load(open(os.path.join(G, 'traj.json')))
    return z, meta


def state_from_arrays(ships, planets, bullets, reload_, t):
    ships = np.asarray(ships, dtype=np.float64).reshape(-1, 5)
    planets = np.asarray(planets, dtype=np.float64).reshape(-1, 4)
    bullets = np.asarray(bullets, dtype=np.float64).reshape(-1, 4)
    return core.State(
        ships=core.Bodies(ships[:, 0:2].copy(), ships[:, 2:4].copy(), ships[:, 4].copy()),
        planets=core.Bodies(planets[:, 0:2].copy(), planets[:, 2:4].copy(), None),
        bullets=core.Bodies(bullets[:, 0:2].copy(), bullets[:, 2:4].copy(), None),
        reload=float(reload_), t=float(t))


from astro_b200.pool import make_pool  # noqa: E402,F401


def oracle_batch_from(arr, S, K):
    """get_arrays() dict -> oracle Batch (float64 image) + alive mask."""
    n = arr['ships'].shape[0]
    b = ao.Batch(n, S, K)
    b.ships[:] = arr['ships']
    b.planets[:] = arr['planets']
    b.np_[:] = arr['n_planets']
    b.bullets[:] = arr['bullets']
    b.nb[:] = arr['n_bullets']
    b.episode[:] = arr['episode']
    return b, (~arr['finished']).astype(np.uint8)


def start_from_pool(games, pool, seed, first_game):
    """Host twin of BatchedGames.reset_all(): game g <- pool[pick(seed, first_game+g, episode 0)]."""
    n = games.n
    pick = rng.pool_pick(seed, first_game + np.arange(n), np.zeros(n, dtype=np.uint32), pool['ships'].shape[0])
    return pick


def stress_fill(K, seed):
    """A start(games) that fills every game's bullet pool: random bullets (a share parked exactly at the arena bound),
    half the games at the cap K, every 8th game a full pool parked in a quiet corner (nothing despawns: overflow on
    fire ticks), tick counters spread over the first fire ticks."""
    def fill(games):
        r = np.random.RandomState(seed)
        n = games.n
        arr = games.get_arrays()
        bl = np.concatenate([r.uniform(-1.3, 1.3, (n, K, 2)), r.uniform(-2.0, 2.0, (n, K, 2))], axis=2)
        # a share of bullets parked exactly at / next to the arena bound and inside planets
        edge = r.rand(n, K) < 0.05
        bl[..., 0][edge] = np.where(r.rand(int(edge.sum())) < 0.5, 1.0, -1.0)
        nb = r.randint(0, K + 1, n)
        nb[r.rand(n) < 0.5] = K
        # every 8th game: a full pool parked in a quiet corner (nothing despawns) -> overflow on fire ticks
        quiet = np.arange(n) % 8 == 0
        q = int(quiet.sum())
        bl[quiet] = np.concatenate([0.95 + r.uniform(-0.01, 0.01, (q, K, 1)), r.uniform(-0.01, 0.01, (q, K, 1)),
                                    np.zeros((q, K, 2))], axis=2)
        nb[quiet] = K
        ticks = r.randint(0, 40, n)       # spread over fire ticks (14, 29)
        games.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], bl, nb, ticks)
    return fill


# ---- the production rollout's options: packed controls in, event planes out, auto-reset -------------------------

def tile_sums(nb):
    """Bullets per 32-game tile."""
    return np.bincount(np.arange(nb.shape[0]) // 32, weights=nb)


def run_launches(g, packed, launches, tile_totals=None, stats=True):
    """Ticks of `packed` (uint8 cuda [T, n_pad]) in astro_tick_many launches of the given lengths, with event planes
    and auto-reset; returns the event planes of every tick.  tile_totals: list receiving each tile's bullet count after
    every launch."""
    import torch
    T = packed.shape[0]
    assert sum(launches) == T
    planes = torch.zeros(g.planes_shape(T), dtype=torch.int32, device='cuda')
    k = 0
    for n in launches:
        g.step_many(n, packed[k:k + n], events=planes[k:k + n], auto_reset=True, stats=stats, packed=True, planes=True)
        k += n
        if tile_totals is not None:
            tile_totals.append(tile_sums(g.get_arrays()['n_bullets']))
    torch.cuda.synchronize()
    return planes.cpu().numpy()


def check_same(a_games, b_games, ev_a, ev_b):
    """Two batches hold the same state element for element (every bullet list in order), the same events and the same
    statistics."""
    a, b = a_games.get_arrays(), b_games.get_arrays()
    assert a.keys() == b.keys()
    for key in a:
        if key != 'bullets':
            assert np.array_equal(a[key], b[key]), key
    nb = b['n_bullets']
    live = np.arange(a['bullets'].shape[1])[None, :] < nb[:, None]
    assert np.array_equal(a['bullets'][live], b['bullets'][live])        # every list, item for item, in order
    assert np.array_equal(ev_a, ev_b)
    assert a_games.stats() == b_games.stats()


# ---- which kernels a library holds and which a call launches -------------------------------------------------------

def library_kernel_names():
    """The demangled names of every kernel of the built library (cuobjdump -symbols, then cu++filt: the spelling
    `tick_kernel<double, (int)1, (bool)0, (int)8>(...)`).  Skips the calling test when the tools are missing."""
    import pytest
    from astro_b200 import _native as nat
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    cufilt = shutil.which('cu++filt') or '/usr/local/cuda/bin/cu++filt'
    if not (os.path.exists(cuobjdump) and os.path.exists(cufilt)):
        pytest.skip('cuobjdump / cu++filt not available')
    syms = subprocess.run([cuobjdump, '-symbols', nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = re.findall(r'STO_ENTRY\s+(\S+)', syms)
    plain = subprocess.run([cufilt], input='\n'.join(names) + '\n', capture_output=True, text=True, check=True).stdout
    return [n for n in plain.split('\n') if n]


def launched(fn, form_of):
    """Runs fn() under torch.profiler with CUDA activity; returns its result and the set of form_of(name) over the kernels
    it launched (CUPTI's spelling: `tick_f32_kernel<2, true, false, false, true>(...)`), Nones left out."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = fn()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert names, 'the profiler returned no kernel records'
    return result, {f for f in map(form_of, names) if f is not None}
