"""The production rollout's fused tick (duel games, packed controls, event planes, auto-reset from the pool, several ticks
per launch) keeps each tile's bullets in shared memory between the ticks of a launch and writes the tile's list to HBM
only after the launch's last tick, or on a tick whose survivors and newborn overflow the staging buffer.  Every test runs
the same controls through launches of several ticks and through one launch per tick, and requires the same state
(bullet lists in order), event planes and episode statistics, element for element."""
import numpy as np
import pytest

from astro_b200 import core
from astro_b200.pool import make_pool
from astro_b200.schedule import Schedule
from tests import helpers as H

pytestmark = pytest.mark.gpu

CFG = core.DEFAULT_CONFIG
N = 2000            # not a multiple of 32: the last tile is padded
STAGE_ITEMS = 224   # bullets a tile's staging buffer holds (7 windows of 32)


def _batch(K, seed=0, warm=120, pool=None, fill=None):
    from astro_b200.batched import BatchedGames
    g = BatchedGames(CFG, N, bullet_cap=K, precision=32, seed=seed)
    pool = make_pool(CFG, 256) if pool is None else pool
    g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    g.reset_all()
    for _ in range(warm):
        g.step(None, auto_reset=True)
    if fill is not None:
        fill(g)
    g.stats(clear=True)
    return g


def _controls(g, T, seed):
    import torch
    gen = torch.Generator(device='cpu').manual_seed(seed)
    acts = torch.randint(0, 6, (T, g.n_pad, 2), dtype=torch.uint8, generator=gen)
    return g.pack_controls(acts).cuda()


_run, _check_same, _tile_sums = H.run_launches, H.check_same, H.tile_sums


def _compare(K, launches, seed=0, **kw):
    """Runs the ticks both ways; returns the tile totals before the first tick and after every tick of the one-launch-per-
    tick run, its event planes and its statistics."""
    T = sum(launches)
    fused, single = _batch(K, seed, **kw), _batch(K, seed, **kw)
    packed = _controls(fused, T, seed + 100)
    start = _tile_sums(single.get_arrays()['n_bullets'])
    totals = []
    ev_single = _run(single, packed, [1] * T, tile_totals=totals)
    ev_fused = _run(fused, packed, list(launches))
    _check_same(fused, single, ev_fused, ev_single)
    return start, np.array(totals), ev_single, single.stats()


@pytest.mark.parametrize('launches', [(2,), (7,), (20,), (64,), (256,), (20, 20), (64, 7)])
def test_fused_launches_equal_one_launch_per_tick(launches):
    _, totals, ev, _ = _compare(32, launches)
    assert totals.sum() > 0 and ev[:, 0].any()             # bullets in flight, games ending


def _parked(K, timeout_tick, T):
    """K - 1 bullets per game parked at rest in a corner (nothing culls them), every game one tick after a fire tick:
    every tile starts at 31 * (K - 1) <= 224 items (K = 8: 217), the next fire tick pushes it over the staging buffer
    (and over K, so some newborn overflow), and the odd games time out in the second half of the launch, which brings
    the tile back under."""
    def fill(g):
        r = np.random.RandomState(K)
        arr = g.get_arrays()
        n = arr['tick'].shape[0]
        bl = np.zeros((n, K - 1, 4))
        bl[..., 0] = 0.95 + r.uniform(-0.01, 0.01, (n, K - 1))
        bl[..., 1] = r.uniform(-0.01, 0.01, (n, K - 1))
        nb = np.full(n, K - 1)
        nb[np.arange(n) % 32 == 0] = 0
        fire = g.schedule.fire_ticks
        ticks = np.full(n, int(fire[0]) + 1)
        odd = np.arange(n) % 2 == 1
        ticks[odd] = timeout_tick - (T * 3) // 4
        g.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], bl, nb, ticks)
    return fill


@pytest.mark.parametrize('K', [4, 8])
def test_tiles_over_the_staging_buffer_and_back(K):
    T = 40
    start, totals, _, st = _compare(K, (T,), fill=_parked(K, Schedule(CFG).timeout_tick, T), warm=0)
    assert st['overflow'] > 0                                  # the m < K cap fired
    if K == 8:
        # tiles that started inside the staging buffer, went over it and came back inside the same launch
        assert (start <= STAGE_ITEMS).all()
        back = (totals > STAGE_ITEMS).any(axis=0) & (totals[-1] <= STAGE_ITEMS)
        assert back.any(), (start.max(), totals.max(axis=0))


def test_games_that_end_on_the_first_last_and_consecutive_ticks():
    """Half the reset pool holds games whose ships overlap: a game re-created from one ends on the next tick again, so
    its generation bit flips on consecutive ticks.  Other games time out on the first and on the last tick of the
    launch."""
    T = 20
    pool = make_pool(CFG, 256)
    pool['ships'][::2, 1, :2] = pool['ships'][::2, 0, :2]
    timeout_tick = Schedule(CFG).timeout_tick

    def fill(g):
        arr = g.get_arrays()
        n = arr['tick'].shape[0]
        ticks = arr['tick'].copy()
        ticks[np.arange(n) % 7 == 1] = timeout_tick
        ticks[np.arange(n) % 7 == 2] = timeout_tick - (T - 1)
        nb = arr['n_bullets']
        g.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], arr['bullets'][:, :max(1, nb.max())], nb, ticks)

    _, _, ev, _ = _compare(32, (T,), pool=pool, fill=fill, warm=60)
    done = ev[:, 0]                                           # [T, n_tiles] ended bits
    assert done[0].any() and done[T - 1].any()
    assert (done[1:] & done[:-1]).any()                       # some game ended on two consecutive ticks
