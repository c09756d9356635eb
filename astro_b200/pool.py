"""Reset pools: initial states built on the host by core.create (core.py:86-135) over the
re-seeded config stream core.generate_configs (core.py:77-83), as game-major arrays for
BatchedGames.set_reset_pool_arrays / astro_set_reset_pool."""
import itertools as it

import numpy as np

from . import core


def make_pool(config, size, planet_slots=None):
    """`size` initial states -> dict(ships [M,S,5] = x,y,dx,dy,b ; planets [M,PL,4] ; np [M]), PL = planet_slots
    (default: batched.planet_slots_for(config), 4 or 8)."""
    from .batched import planet_slots_for
    S = 1 if config.solo else 2
    PL = planet_slots_for(config) if planet_slots is None else int(planet_slots)
    ships = np.zeros((size, S, 5))
    planets = np.zeros((size, PL, 4))
    n_planets = np.zeros(size, dtype=np.int32)
    for i, c in enumerate(it.islice(core.generate_configs(config), size)):
        s = core.create(c)
        ships[i, :, 0:2], ships[i, :, 2:4], ships[i, :, 4] = s.ships.x, s.ships.dx, s.ships.b
        p = s.planets.x.shape[0]
        planets[i, :p, 0:2], planets[i, :p, 2:4] = s.planets.x, s.planets.dx
        n_planets[i] = p
    return dict(ships=ships, planets=planets, np=n_planets)
