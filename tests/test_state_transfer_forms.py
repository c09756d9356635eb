"""Every state-transfer and reset kernel instantiation, each checked against a host model of the tile layout.

astro_export_games / astro_import_games / astro_reset_done / astro_set_reset_pool (astro_b200.cu) choose
export_kernel<R, S, PL> (8 forms), import_kernel<R, S, PL> (8), import_map_kernel (1), reset_kernel<R, S, PL> (8) and
pack_pool_kernel<S, PL> (4) from the batch layout.  LEDGER lists all 29 and the tests that launch each one; a CPU test
holds it to the symbols of the built library, and every GPU test asserts, through torch.profiler, that it launched
exactly the state-transfer forms it is about.

The reference is pack() / unpack(): the layout of include/astro_b200.h and of the BatchedGames tensors (tiles of 32
games, the meta word in its 4- and 8-slot packings, each tile's bullet list in game order with finished games owning
no items) restated in plain numpy.  The tests write the raw tensors from the model and read them back through it, so
export and import are each compared with a reference rather than only with each other.

- export: every output bit against unpack(), over every planet count, stale dead planet slots, bullet counts 0 .. K
  (K = 1023 fills the whole nb field), finished games with stale counts in the middle of tiles, ticks at 0 and at the
  layout's maximum, episodes >= 2^31, a ragged last tile, lists in either bullet buffer, permuted and out-of-range
  indices, bullet_rows below, at and above K, and a null episode array.
- import: the raw tensors after astro_import_games against the model's import applied on the host: rebuilt lists of
  touched tiles, untouched tiles byte for byte, float32 rounding, the clamps of n_bullets / n_planets, null columns.
- reset_done: re-created games against the pool pick of the current stream step (game ids wrapping at 2^32), live
  games and every list untouched; observe() and the next tick against the oracle read none of the stale planet rows
  a re-created game keeps past its planet count.
- auto-reset: the packed pool records (NaN in their dead planet slots) against the pool they were packed from.
- core.step in every layout it picks (test_core_step_in_every_layout) launches export_kernel<double, S, PL> and
  import_kernel<double, S, PL> inside the CUDA graph of astro_step_single_host.  Those forms are listed under the export
  and import tests, so it adds none to the ledger; its profiler check names them all the same."""
import ctypes as C
import re

import numpy as np
import pytest

from astro_b200 import _native as nat
from astro_b200 import core, rng
from oracle import astro_oracle as ao
from tests import helpers as H

E_INVALID, E_STATE = -1, -3
TOL = 1e-5                        # the float32 tick's policy (test_tick_forms)
N = 173                           # 6 tiles, the last one ragged

# ------------------------------------------------------------------ kernel names and the ledger

_FORM = re.compile(r'\b(?:(import_map_kernel)\b(?!<)|(export_kernel|import_kernel|reset_kernel|pack_pool_kernel)<([^<>]*)>)')


def form_of(name):
    """A state-transfer kernel's name, as CUPTI writes it (`export_kernel<double, 2, 8>`) or as cu++filt does
    (`export_kernel<double, (int)2, (int)8>`), as a tuple: ('export_kernel', 'double', 2, 8); pack_pool_kernel<2, 4> ->
    ('pack_pool_kernel', 2, 4); import_map_kernel, not a template -> ('import_map_kernel',).  None for any other kernel."""
    m = _FORM.search(name)
    if m is None:
        return None
    if m.group(1):
        return (m.group(1),)
    out = [m.group(2)]
    for a in m.group(3).split(','):
        a = re.sub(r'^\(int\)', '', a.strip())
        out.append(int(a) if a.isdigit() else a)
    return tuple(out)


FORMS = [(r, S, PL) for r in ('float', 'double') for S in (1, 2) for PL in (4, 8)]
FORM_IDS = ['%s S=%d PL=%d' % f for f in FORMS]
POOL_FORMS = [(S, PL) for S in (1, 2) for PL in (4, 8)]
IMPORT_MAP = ('import_map_kernel',)


def export_form(r, S, PL):
    return ('export_kernel', r, S, PL)


def import_form(r, S, PL):
    return ('import_kernel', r, S, PL)


def reset_form(r, S, PL):
    return ('reset_kernel', r, S, PL)


def pack_form(S, PL):
    return ('pack_pool_kernel', S, PL)


def _ledger():
    led = {}

    def add(test, *forms):
        for f in forms:
            led.setdefault(f, []).append(test)
    for r, S, PL in FORMS:
        add('test_export_reads_the_tile_layout', export_form(r, S, PL))
        add('test_import_writes_the_tile_layout', import_form(r, S, PL))
        add('test_reset_done_recreates_finished_games_from_the_pool', reset_form(r, S, PL))
    add('test_import_writes_the_tile_layout', IMPORT_MAP)
    for S, PL in POOL_FORMS:
        add('test_auto_reset_reads_the_packed_pool', pack_form(S, PL))
        add('test_reset_done_recreates_finished_games_from_the_pool', pack_form(S, PL))    # (float32 batches pack their pool)
    add('test_export_and_import_refuse_bad_arguments', export_form('float', 2, 4), import_form('float', 2, 4), IMPORT_MAP)
    return {f: tuple(t) for f, t in led.items()}


LEDGER = _ledger()


def test_state_kernel_names_parse_in_both_spellings():
    assert form_of('void (anonymous namespace)::export_kernel<double, 2, 8>(const void *, int)') \
        == ('export_kernel', 'double', 2, 8)
    assert form_of('void <unnamed>::export_kernel<double, (int)2, (int)8>(const void *, int)') \
        == ('export_kernel', 'double', 2, 8)
    assert form_of('void <unnamed>::import_kernel<float, (int)1, (int)4>(void *, <unnamed>::GameArrays)') \
        == import_form('float', 1, 4)
    assert form_of('void (anonymous namespace)::reset_kernel<float, 2, 4>((anonymous namespace)::TickParams)') \
        == reset_form('float', 2, 4)
    assert form_of('void <unnamed>::pack_pool_kernel<(int)2, (int)8>(const float *, const float *, const int *, float *, int)') \
        == pack_form(2, 8)
    assert form_of('void (anonymous namespace)::pack_pool_kernel<1, 4>(float const*, float const*, int const*, float*, int)') \
        == pack_form(1, 4)
    assert form_of('<unnamed>::import_map_kernel(const int *, int, int, int *)') == IMPORT_MAP
    assert form_of('(anonymous namespace)::import_map_kernel(int const*, int, int, int*)') == IMPORT_MAP
    assert form_of('void <unnamed>::tick_kernel<double, (int)1, (bool)0, (int)8>(<unnamed>::TickParams)') is None
    assert form_of('void (anonymous namespace)::tick_f32_kernel<2, true, false, false, true>(TickParams)') is None
    assert form_of('void <unnamed>::observe_kernel<float, (int)2, (bool)1, (int)4>(const void *, int)') is None
    assert form_of('void <unnamed>::policy_mma_kernel<float, (int)2, (int)4>(const void *)') is None


def test_library_state_forms_equal_the_ledger():
    """The built library's export / import / import_map / reset / pack_pool instantiations are exactly the ledger's 29
    keys, and every test the ledger names exists here: a form added to the library without a test that launches it
    fails here, with no GPU."""
    forms = [f for f in map(form_of, H.library_kernel_names()) if f is not None]
    assert len(forms) == len(set(forms)) == 29
    assert set(forms) == set(LEDGER), (sorted(set(forms) - set(LEDGER)), sorted(set(LEDGER) - set(forms)))
    for form, tests in LEDGER.items():
        assert tests, form
        for t in tests:
            assert callable(globals().get(t)) and t.startswith('test_'), (form, t)


def _expect(forms, fn, listed=True):
    """fn() must launch exactly the state-transfer forms `forms`, each at least once; with `listed`, each must be in the
    ledger under the calling test."""
    import inspect
    test = next(f.function for f in inspect.stack(0) if f.function.startswith('test_'))
    for f in forms:
        assert not listed or test in LEDGER[f], (test, f)
    result, got = H.launched(fn, form_of)
    assert got == set(forms), (sorted(set(forms) - got), sorted(got - set(forms)))
    return result


# ------------------------------------------------------------------ the host model of the tile layout

def max_tick(PL):
    return nat.MAX_TICKS_WIDE if PL > nat.MAX_PLANETS else nat.MAX_TICKS


def meta_pack(nb, np_, fin, tick, PL):
    """The meta word(s): nb bits 0-9, np bits 10-12, finished bit 13, tick from bit 14; 8-slot batches keep np's bit 3 in
    bit 31 and the tick in bits 14-30."""
    nb, np_, fin, tick = (np.asarray(v).astype(np.uint64) for v in (nb, np_, fin, tick))
    w = nb | ((np_ & 7) << 10) | (fin << 13) | (tick << 14)
    if PL > nat.MAX_PLANETS:
        w |= (np_ & 8) << 28
    return (w & 0xFFFFFFFF).astype(np.uint32)


def meta_unpack(m, PL):
    """(nb field, np, finished, tick) of meta word(s)."""
    m = np.asarray(m, dtype=np.uint32).astype(np.int64)
    if PL > nat.MAX_PLANETS:
        return m & 1023, ((m >> 10) & 7) | ((m >> 28) & 8), ((m >> 13) & 1).astype(bool), (m >> 14) & 0x1FFFF
    return m & 1023, (m >> 10) & 7, ((m >> 13) & 1).astype(bool), m >> 14


def _live_nb(nb_field, finished):
    return np.where(finished, 0, nb_field)


def _list_starts(nb):
    """First list item of every game: the counts of the lower games of its tile (tile_list_offset)."""
    t = nb.reshape(-1, 32)
    return (np.cumsum(t, axis=1) - t).reshape(-1)


def pack(g, PL, K, dtype, cur, seed=0):
    """Raw tensors (numpy) of games-major state `g` (n = a multiple of 32): ships [T,S,32,4], ship_b [T,S,32],
    planets [T,PL,32,4] (every slot as given: stale values in dead slots stay), bullets [2,T,32K,4] with each tile's
    list in buffer `cur` (the rest of both buffers random junk), meta, episode (uint32 [n]) and cur.  g: ships [n,S,5],
    planets [n,PL,4], n_planets, n_bullets (the nb field, stale for finished games), finished, tick, episode, bullets
    [n,>=max nb,4]."""
    n, S = g['ships'].shape[:2]
    T = n // 32
    r = np.random.RandomState(seed)
    bullets = r.uniform(-9.0, 9.0, (2, T, 32 * max(K, 1), 4))
    nb = _live_nb(g['n_bullets'], g['finished'])
    first = _list_starts(nb)
    for i in range(n):
        bullets[cur, i // 32, first[i]:first[i] + nb[i]] = g['bullets'][i, :nb[i]]
    return dict(ships=g['ships'][..., :4].reshape(T, 32, S, 4).transpose(0, 2, 1, 3).astype(dtype),
                ship_b=g['ships'][..., 4].reshape(T, 32, S).transpose(0, 2, 1).astype(dtype),
                planets=g['planets'].reshape(T, 32, PL, 4).transpose(0, 2, 1, 3).astype(dtype),
                bullets=bullets.astype(dtype),
                meta=meta_pack(g['n_bullets'], g['n_planets'], g['finished'], g['tick'], PL),
                episode=np.asarray(g['episode']).astype(np.uint32), cur=int(cur))


def unpack(raw, rows=None):
    """Games-major float64 arrays of raw tensors, as astro_export_games documents them: dead planet slots and bullet rows
    past n_bullets zero, finished games n_bullets 0, `rows` bullet rows per game (default the cap; fewer cut the list
    off, n_bullets still counts it)."""
    T, S = raw['ships'].shape[:2]
    PL = raw['planets'].shape[1]
    K = raw['bullets'].shape[2] // 32
    rows = K if rows is None else rows
    n = T * 32
    nbf, npl, fin, tick = meta_unpack(raw['meta'], PL)
    nb = _live_nb(nbf, fin)
    ships = np.concatenate([raw['ships'].transpose(0, 2, 1, 3).reshape(n, S, 4),
                            raw['ship_b'].transpose(0, 2, 1).reshape(n, S, 1)], axis=2).astype(np.float64)
    planets = raw['planets'].transpose(0, 2, 1, 3).reshape(n, PL, 4).astype(np.float64)
    planets[np.arange(PL)[None, :] >= npl[:, None]] = 0.0
    first = _list_starts(nb)
    bullets = np.zeros((n, rows, 4))
    for i in range(n):
        k = min(int(nb[i]), rows)
        bullets[i, :k] = raw['bullets'][raw['cur'], i // 32, first[i]:first[i] + k]
    return dict(ships=ships, planets=planets, bullets=bullets, n_planets=npl, n_bullets=nb, tick=tick, finished=fin,
                episode=raw['episode'].copy())


def test_meta_model_matches_the_header_packing():
    """meta_pack / meta_unpack against hand-written words of include/astro_b200.h: 4 slots (np in bits 10-12, an 18-bit
    tick up to bit 31) and 8 slots (np = 8 as bit 31 with the low bits zero, a 17-bit tick in bits 14-30)."""
    cases = [
        # PL, nb, np, finished, tick, word
        (8, 1023, 8, 0, nat.MAX_TICKS_WIDE, 0xFFFFC3FF),
        (8, 1023, 8, 1, nat.MAX_TICKS_WIDE, 0xFFFFE3FF),
        (8, 0, 7, 0, 0, 0x00001C00),
        (8, 5, 8, 0, 1, 0x80004005),
        (8, 1, 4, 1, 2, 0x0000B001),
        (4, 1023, 4, 0, nat.MAX_TICKS, 0xFFFFD3FF),
        (4, 1023, 4, 1, nat.MAX_TICKS, 0xFFFFF3FF),
        (4, 0, 1, 1, 0, 0x00002400),
        (4, 33, 3, 0, 131072, 0x80000C21),
    ]
    for PL, nb, np_, fin, tick, word in cases:
        assert int(meta_pack(nb, np_, fin, tick, PL)) == word, (PL, nb, np_, fin, tick, hex(word))
        assert [int(v) for v in meta_unpack(word, PL)] == [nb, np_, fin, tick], (PL, hex(word))


def test_layout_model_round_trips():
    """unpack(pack(state)) is the state as export documents it, for both buffers and both slot counts: live lists in
    game order, finished games with no items, dead slots zero."""
    for PL in (4, 8):
        for cur in (0, 1):
            r = np.random.RandomState(PL + cur)
            g = random_games(64, 2, PL, 40, r)
            got = unpack(pack(g, PL, 40, np.float64, cur, seed=3))
            nb = _live_nb(g['n_bullets'], g['finished'])
            assert (got['n_bullets'] == nb).all() and (got['n_planets'] == g['n_planets']).all()
            assert (got['finished'] == g['finished']).all() and (got['tick'] == g['tick']).all()
            assert (got['episode'] == g['episode']).all() and H.same_bits(got['ships'], g['ships'])
            for i in range(64):
                assert (got['planets'][i, :g['n_planets'][i]] == g['planets'][i, :g['n_planets'][i]]).all()
                assert (got['planets'][i, g['n_planets'][i]:] == 0).all()
                assert (got['bullets'][i, :nb[i]] == g['bullets'][i, :nb[i]]).all() and (got['bullets'][i, nb[i]:] == 0).all()


def random_games(n, S, PL, K, r, fin=0.2, max_t=None, arena=False):
    """Games-major raw state of n games: every planet count 1..PL with random values in every slot (dead ones stale),
    bullet counts 0, 1, 31, 32, 33 and K at lanes 0-5 of every tile and random elsewhere, a share `fin` finished (lane
    13 always, lane 14 never) with stale nb fields up to 1023, ticks 0 (lane 7) and max_t (lane 8), episodes 2^31 (lane
    9) and 2^32 - 1 (lane 10).  arena=True: positions a tick may start from (ships inside the arena)."""
    max_t = max_tick(PL) if max_t is None else max_t
    lane, tile = np.arange(n) % 32, np.arange(n) // 32
    ships = np.concatenate([r.uniform(-0.9 if arena else -1.2, 0.9 if arena else 1.2, (n, S, 2)),
                            r.uniform(-0.3, 0.3, (n, S, 2)), r.uniform(-250, 250, (n, S, 1))], axis=2)
    planets = np.concatenate([r.uniform(-0.8, 0.8, (n, PL, 2)), r.uniform(-0.1, 0.1, (n, PL, 2))], axis=2)
    npl = 1 + r.permutation(np.arange(n) % PL)
    finished = r.rand(n) < fin
    finished[lane == 13] = True
    finished[(lane < 6) | (lane == 14)] = False
    nb = r.randint(0, K + 1, n)
    edge = np.array([0, 1, 31, 32, 33, K])
    nb[lane < 6] = np.minimum(edge[(lane + tile)[lane < 6] % 6], K)
    nb[finished] = r.randint(1, 1024, int(finished.sum()))
    tick = r.randint(0, max_t + 1, n)
    tick[lane == 7], tick[lane == 8] = 0, max_t
    episode = r.randint(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    episode[lane == 9], episode[lane == 10] = 1 << 31, 0xFFFFFFFF
    bullets = np.concatenate([r.uniform(-1.3, 1.3, (n, max(K, 1), 2)), r.uniform(-2, 2, (n, max(K, 1), 2))], axis=2)
    return dict(ships=ships, planets=planets, n_planets=npl, n_bullets=nb, finished=finished, tick=tick,
                episode=episode, bullets=bullets)


# ------------------------------------------------------------------ device glue: raw tensors, export, import

def _config(S, PL):
    cfg = core.SOLO_CONFIG if S == 1 else core.DEFAULT_CONFIG
    return cfg._replace(max_planets=PL)


def _batch(r, S, PL, n, K, seed=0, first_game=0):
    from astro_b200.batched import BatchedGames
    return BatchedGames(_config(S, PL), n, bullet_cap=K, precision=64 if r == 'double' else 32, seed=seed,
                        first_game=first_game)


def write_raw(games, raw):
    import torch
    for k in ('ships', 'ship_b', 'planets', 'bullets'):
        getattr(games, k).copy_(torch.from_numpy(np.ascontiguousarray(raw[k])))
    games.meta.copy_(torch.from_numpy(raw['meta'].view(np.int32)))
    games.episode.copy_(torch.from_numpy(raw['episode'].view(np.int32)))
    nat.check(nat.lib().astro_set_bullet_buffer(games._h, raw['cur']))
    torch.cuda.synchronize()


def read_raw(games):
    import torch
    torch.cuda.synchronize()
    out = {k: getattr(games, k).cpu().numpy() for k in ('ships', 'ship_b', 'planets', 'bullets')}
    out['meta'] = games.meta.cpu().numpy().view(np.uint32).copy()
    out['episode'] = games.episode.cpu().numpy().view(np.uint32).copy()
    out['cur'] = games.bullet_buffer
    return out


def _same(a, b):
    """Bit equality of two arrays of the same dtype and shape."""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    u = {1: np.uint8, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    return bool((a.view(u) == b.view(u)).all())


SENTINEL = dict(ships=-1.5e300, planets=-1.5e300, bullets=-1.5e300, n_planets=-123457, n_bullets=-123457, tick=-123457,
                finished=0xA5, episode=-0x5A5A5A5B)


def export(games, index, m, rows, episode=True):
    """astro_export_games through ctypes into outputs filled with SENTINEL first; returns numpy arrays (episode uint32,
    finished bool-free uint8) with bullets cut to `rows`."""
    import torch
    dev, f64, i32 = games.device, torch.float64, torch.int32
    t = dict(ships=torch.full((m, games.S, 5), SENTINEL['ships'], dtype=f64, device=dev),
             planets=torch.full((m, games.PL, 4), SENTINEL['planets'], dtype=f64, device=dev),
             bullets=torch.full((m, max(rows, 1), 4), SENTINEL['bullets'], dtype=f64, device=dev),
             n_planets=torch.full((m,), SENTINEL['n_planets'], dtype=i32, device=dev),
             n_bullets=torch.full((m,), SENTINEL['n_bullets'], dtype=i32, device=dev),
             tick=torch.full((m,), SENTINEL['tick'], dtype=i32, device=dev),
             finished=torch.full((m,), SENTINEL['finished'], dtype=torch.uint8, device=dev),
             episode=torch.full((m,), SENTINEL['episode'], dtype=i32, device=dev))
    idx = None if index is None else torch.from_numpy(np.asarray(index, dtype=np.int32)).to(dev)
    arrays = games._arrays_struct(dict(t, episode=t['episode'] if episode else None), rows)
    rc = nat.lib().astro_export_games(games._h, None if idx is None else idx.data_ptr(), m, C.byref(arrays), games._stream())
    assert rc == 0, nat.lib().astro_last_error()
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in t.items()}
    out['bullets'] = out['bullets'][:, :rows]
    out['episode'] = out['episode'].view(np.uint32)
    return out


def _expected_export(full, idx, rows):
    """Rows `idx` of unpack() output `full`, as the export's arrays (bullets cut to `rows`)."""
    return dict(ships=full['ships'][idx], planets=full['planets'][idx], bullets=full['bullets'][idx][:, :rows],
                n_planets=full['n_planets'][idx].astype(np.int32), n_bullets=full['n_bullets'][idx].astype(np.int32),
                tick=full['tick'][idx].astype(np.int32), finished=full['finished'][idx].astype(np.uint8),
                episode=full['episode'][idx])


def _check_export(got, want, what):
    for k, v in want.items():
        assert _same(got[k], v), (what, k, np.argwhere(got[k] != v)[:4])


def import_(games, index, m, arrays, rows):
    """astro_import_games through ctypes; arrays: numpy columns (a None column is passed as a null pointer)."""
    import torch
    dev = games.device
    dt = dict(ships=np.float64, planets=np.float64, bullets=np.float64, n_planets=np.int32, n_bullets=np.int32,
              tick=np.int32, finished=np.uint8, episode=np.uint32)
    t = {k: None if arrays.get(k) is None else
         torch.from_numpy(np.ascontiguousarray(arrays[k], dtype=dt[k]).view(np.int32 if k == 'episode' else dt[k])).to(dev)
         for k in dt}
    idx = None if index is None else torch.from_numpy(np.asarray(index, dtype=np.int32)).to(dev)
    struct = games._arrays_struct(t, rows)
    rc = nat.lib().astro_import_games(games._h, None if idx is None else idx.data_ptr(), m, C.byref(struct), games._stream())
    assert rc == 0, nat.lib().astro_last_error()
    torch.cuda.synchronize()


def import_model(raw, index, m, a, rows):
    """The raw tensors after astro_import_games(index, m, a, bullet_rows=rows), on the host: row i replaces game
    index[i] (rows 0..m-1 replace games 0..m-1 without an index; out-of-range entries replace nothing), n_bullets
    clamped to 0..min(K, rows) (0 when null or finished), n_planets to 0..PL, values rounded to the batch's type, dead
    planet slots zero, tick 0 when null, episode kept when null; every touched tile's list rebuilt in the current buffer
    in game order.  Returns (raw, {touched tile: list length})."""
    T, S = raw['ships'].shape[:2]
    PL = raw['planets'].shape[1]
    K = raw['bullets'].shape[2] // 32
    n = T * 32
    dtype = raw['ships'].dtype
    src = np.full(n, -1)
    if index is None:
        src[:m] = np.arange(m)
    else:
        for i, g in enumerate(index[:m]):
            if 0 <= g < n:
                src[g] = i
    old = unpack(raw)
    new = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in raw.items()}
    lists = [old['bullets'][g, :old['n_bullets'][g]].astype(dtype) for g in range(n)]
    for g in np.nonzero(src >= 0)[0]:
        i, t, l = src[g], g // 32, g % 32
        fin = bool(a['finished'][i]) if a.get('finished') is not None else False
        want = int(a['n_bullets'][i]) if a.get('n_bullets') is not None else 0
        nb = 0 if fin else min(max(want, 0), K, rows)
        npl = min(max(int(a['n_planets'][i]), 0), PL)
        new['ships'][t, :, l] = a['ships'][i, :, :4].astype(dtype)
        new['ship_b'][t, :, l] = a['ships'][i, :, 4].astype(dtype)
        new['planets'][t, :, l] = np.where(np.arange(PL)[:, None] < npl, a['planets'][i], 0.0).astype(dtype)
        tick = int(a['tick'][i]) if a.get('tick') is not None else 0
        new['meta'][g] = meta_pack(nb, npl, int(fin), tick, PL)
        if a.get('episode') is not None:
            new['episode'][g] = np.uint32(a['episode'][i])
        lists[g] = a['bullets'][i, :nb].astype(dtype) if nb else np.zeros((0, 4), dtype)
    totals = {}
    for t in sorted(set(np.nonzero(src >= 0)[0] // 32)):
        run = np.concatenate([lists[g] for g in range(32 * t, 32 * t + 32)]).reshape(-1, 4)
        new['bullets'][raw['cur'], t, :len(run)] = run
        totals[int(t)] = len(run)
    return new, totals


def _check_import(got, want, before, totals, what):
    for k in ('ships', 'ship_b', 'planets', 'meta', 'episode'):
        assert _same(got[k], want[k]), (what, k, np.argwhere(got[k] != want[k])[:4])
    assert got['cur'] == want['cur'], what
    c = want['cur']
    for t in range(got['ships'].shape[0]):
        if t in totals:
            assert _same(got['bullets'][c, t, :totals[t]], want['bullets'][c, t, :totals[t]]), (what, 'list of tile', t)
        else:
            assert _same(got['bullets'][c, t], before['bullets'][c, t]), (what, 'untouched tile', t)


# ------------------------------------------------------------------ export against the model, all 8 forms

@pytest.mark.gpu
@pytest.mark.parametrize('r,S,PL', FORMS, ids=FORM_IDS)
def test_export_reads_the_tile_layout(r, S, PL):
    """astro_export_games == unpack() bit for bit on raw tensors written from the model: every planet count, stale
    dead planet slots (exported as zeros), bullet counts 0, 1, 31, 32, 33 and K (K = 1023 in 8-slot batches: the whole
    nb field), finished games with stale nb in the middle of tiles (n_bullets 0, their neighbours' runs unshifted), ticks
    0 and the layout's maximum, episodes >= 2^31, 173 games (a ragged last tile), lists in bullet buffer 0 and 1.  Calls:
    no index; a permutation of every slot, padding included; bullet_rows 0, below, at and above K (rows past nb zero,
    a list longer than bullet_rows cut off with n_bullets still counting it); a null episode array; out-of-range index
    entries, whose rows keep the sentinel written before the call.  Export writes nothing into the batch."""
    K = 1023 if PL == 8 else 40
    rs = np.random.RandomState(FORMS.index((r, S, PL)))
    games = _batch(r, S, PL, N, K)
    n, n_pad = games.n, games.n_pad
    dtype = np.float32 if r == 'float' else np.float64

    def run():
        for cur in (0, 1):
            g = random_games(n_pad, S, PL, K, rs)
            raw = pack(g, PL, K, dtype, cur, seed=cur)
            write_raw(games, raw)
            full = unpack(raw, K + 9)
            live = ~full['finished']
            assert set(full['n_planets'][live]) == set(range(1, PL + 1))
            assert {0, 1, 31, 32, 33, K} <= set(full['n_bullets'][live])
            assert (np.nonzero(~live & (g['n_bullets'] > 0))[0] % 32 == 13).any()
            _check_export(export(games, None, n, K), _expected_export(full, np.arange(n), K), (cur, 'no index'))
            perm = rs.permutation(n_pad)
            _check_export(export(games, perm, n_pad, K), _expected_export(full, perm, K), (cur, 'permutation'))
            for rows in (0, 20, K + 9):
                got = export(games, None, n, rows)
                _check_export(got, _expected_export(full, np.arange(n), rows), (cur, 'rows', rows))
            assert (got['n_bullets'] > 20).any()                     # (rows 20: lists cut off, n_bullets still counts them)
            got = export(games, perm, n_pad, K, episode=False)
            want = _expected_export(full, perm, K)
            want['episode'] = np.full(n_pad, SENTINEL['episode'], dtype=np.int32).view(np.uint32)
            _check_export(got, want, (cur, 'null episode'))
            bad = perm.copy()
            at = np.array([0, 3, 40, 77, n_pad - 1])
            bad[at] = [-1, n_pad, n_pad + 5000, 2 ** 31 - 1, -2 ** 31]
            got = export(games, bad, n_pad, K)
            ok = np.ones(n_pad, dtype=bool)
            ok[at] = False
            want = _expected_export(full, perm, K)
            for k in want:
                want[k] = want[k].copy()
                want[k][~ok] = np.array(SENTINEL[k]).astype(want[k].dtype) if k != 'episode' else \
                    np.array(SENTINEL[k], dtype=np.int32).view(np.uint32)
            _check_export(got, want, (cur, 'out-of-range index'))
            after = read_raw(games)
            for k in ('ships', 'ship_b', 'planets', 'bullets', 'meta', 'episode'):
                assert _same(after[k], raw[k]), (cur, 'export wrote into', k)
    _expect([export_form(r, S, PL)], run)


# ------------------------------------------------------------------ import against the model, all 8 forms

def _import_rows(m, S, PL, K, rows, r):
    """Import columns for m rows: float64 values float32 cannot hold, every planet count (and 0 / PL + 3 / -2, which
    clamp), dead planet slots non-zero, bullet counts that grow, shrink or drop to 0, above rows and K (clamped), below 0,
    a share finished, ticks up to the layout's maximum, episodes >= 2^31.  Rows 0 and 1: np = PL at the largest tick
    (row 1 finished)."""
    a = random_games(m, S, PL, K, r, fin=0.15)
    a['bullets'] = np.concatenate([r.uniform(-1.3, 1.3, (m, max(rows, 1), 2)), r.uniform(-2, 2, (m, max(rows, 1), 2))], axis=2)
    a['n_bullets'] = r.randint(0, rows + 1, m)
    a['n_bullets'][np.arange(m) % 7 == 1] = 0
    extra = np.array([rows, rows + 2, K + 5, 5000, -3])
    a['n_bullets'][np.arange(m) % 7 == 2] = extra[np.arange(m)[np.arange(m) % 7 == 2] % 5]
    a['n_planets'][np.arange(m) % 11 == 4] = PL + 3
    a['n_planets'][np.arange(m) % 11 == 5] = 0
    a['n_planets'][np.arange(m) % 11 == 6] = -2
    a['n_planets'][:2], a['tick'][:2], a['finished'][:2] = PL, max_tick(PL), [False, True]
    return a


@pytest.mark.gpu
@pytest.mark.parametrize('r,S,PL', FORMS, ids=FORM_IDS)
def test_import_writes_the_tile_layout(r, S, PL):
    """astro_import_games (through ctypes, so the kernel's own clamps are reached) against import_model() on the raw
    tensors: a subset index touching three tiles partly (padding slots and out-of-range entries included) and leaving
    three alone; no index with m = 107 < n_games (the rest of tile 3 kept, its lists moved to their new places); null
    n_bullets / tick / finished / episode; counts that grow, shrink, drop to 0 or clamp at K and at bullet_rows;
    finished rows; np = PL at the largest tick.  Touched tiles' lists are rebuilt in game order, untouched tiles' current
    buffer is byte-identical, written games are rounded to the batch's type with dead planet slots zero, kept games and
    meta / episode words are exact."""
    K = 1023 if PL == 8 else 40
    rs = np.random.RandomState(50 + FORMS.index((r, S, PL)))
    games = _batch(r, S, PL, N, K)
    n_pad = games.n_pad
    dtype = np.float32 if r == 'float' else np.float64

    def step(raw, index, m, a, rows, what):
        want, totals = import_model(raw, index, m, a, rows)
        import_(games, index, m, a, rows)
        got = read_raw(games)
        _check_import(got, want, raw, totals, what)
        return got, totals

    def run():
        for cur in (1, 0):
            raw = pack(random_games(n_pad, S, PL, K, rs), PL, K, dtype, cur, seed=7 + cur)
            write_raw(games, raw)
            # 1. a subset index: tiles 0, 2 and 5 (padding slots 173.. included) partly, 1, 3 and 4 untouched
            lanes = {0: [0, 3, 4, 13, 17, 31], 2: [5, 6, 7, 8, 9, 20], 5: [0, 1, 12, 13, 14, 30]}
            index = np.array([32 * t + l for t, ls in lanes.items() for l in ls] + [-1, n_pad + 3])
            index = index[rs.permutation(index.size)]
            rows = K - 3
            a = _import_rows(index.size, S, PL, K, rows, rs)
            raw, totals = step(raw, index, index.size, a, rows, (cur, 'subset'))
            assert sorted(totals) == [0, 2, 5]
            # 2. no index, m = 107: tiles 0-2 and games 96..106 replaced, 107..127 kept behind them, tiles 4-5 untouched
            m = 107
            a = _import_rows(m, S, PL, K, K, rs)
            raw, totals = step(raw, None, m, a, K, (cur, 'first m'))
            assert sorted(totals) == [0, 1, 2, 3]
            # 3. null n_bullets / tick / finished / episode (and bullets): no bullets, tick 0, not finished, episode kept
            index = np.array([32 + 2, 32 + 3, 32 + 30, 128 + 0, 128 + 16])
            a = _import_rows(index.size, S, PL, K, 5, rs)
            for k in ('n_bullets', 'tick', 'finished', 'episode', 'bullets'):
                a[k] = None
            raw, totals = step(raw, index, index.size, a, 5, (cur, 'null columns'))
            assert sorted(totals) == [1, 4]
    _expect([import_form(r, S, PL), IMPORT_MAP], run)


# ------------------------------------------------------------------ reset_done against the model and the oracle

def _lib_pool(games, ships, planets, npl):
    """The pool as set_reset_pool_arrays stores it (rounded to the batch's type)."""
    games.set_reset_pool_arrays(ships, planets, npl)
    return [x.cpu().numpy() for x in games._pool]


def _rows_of(raw, k):
    """Games-major view of raw tensor k: ships [n,S,4], ship_b [n,S], planets [n,PL,4]."""
    a = raw[k].swapaxes(1, 2)
    return a.reshape((a.shape[0] * 32,) + a.shape[2:])


def _check_recreated(got, before, pool, picks, dead, what):
    """Re-created games (dead) hold pool[picks] in their live slots, meta (nb 0, np, live, tick 0), episode + 1 (mod 2^32);
    every other game and the whole current bullet buffer are as in `before`."""
    ps, pp, pn = pool
    PL = got['planets'].shape[1]
    live = ~dead
    for k in ('ships', 'ship_b', 'planets'):
        assert _same(_rows_of(got, k)[live], _rows_of(before, k)[live]), (what, 'live game changed', k)
    assert _same(got['meta'][live], before['meta'][live]) and _same(got['episode'][live], before['episode'][live]), what
    c = got['cur']
    assert c == before['cur'] and _same(got['bullets'][c], before['bullets'][c]), (what, 'bullet lists changed')
    g = np.nonzero(dead)[0]
    k = picks[g]
    assert _same(_rows_of(got, 'ships')[g], ps[k][..., :4]), (what, 'ships')
    assert _same(_rows_of(got, 'ship_b')[g], ps[k][..., 4]), (what, 'bearings')
    planets = _rows_of(got, 'planets')[g]
    for j in range(PL):
        sel = j < pn[k]
        assert _same(planets[sel, j], pp[k][sel, j]), (what, 'planet', j)
    assert _same(got['meta'][g], meta_pack(0, pn[k], 0, 0, PL)), (what, 'meta')
    assert _same(got['episode'][g], (before['episode'][g].astype(np.uint64) + 1).astype(np.uint32)), (what, 'episode')


def _oracle_tick(cfg, games, state, acts, K):
    """ao.step_one for every game of unpack() output `state` (reload / t from the batch's schedule)."""
    out = []
    for i in range(state['ships'].shape[0]):
        if state['finished'][i]:
            out.append(None)
            continue
        P, B, tk = int(state['n_planets'][i]), int(state['n_bullets'][i]), int(state['tick'][i])
        out.append(ao.step_one(cfg, state['ships'][i], state['planets'][i, :P], state['bullets'][i, :B],
                               games.schedule.reload[tk], games.schedule.t[tk], acts[i], bullet_cap=K))
    return out


def _check_tick(games, state, after, outs, events, exact, what):
    """The state after one tick (unpack of the raw tensors) against the oracle's: events and done of the first n games,
    bullet counts exactly, every value bit for bit (exact) or within TOL relative."""
    worst = 0.0
    n = games.n
    for i, o in enumerate(outs):
        if o is None:
            assert after['finished'][i], (what, i)
            continue
        if i < n:
            assert events[i] == o['events'], (what, i, events[i], o['events'])
        assert bool(after['finished'][i]) == o['done'], (what, i)
        if o['done']:
            continue
        P, B = int(state['n_planets'][i]), len(o['bullets'])
        assert after['n_bullets'][i] == B and after['n_planets'][i] == P and after['tick'][i] == state['tick'][i] + 1, (what, i)
        for got, ref in ((after['ships'][i], o['ships']), (after['planets'][i, :P], o['planets']),
                         (after['bullets'][i, :B], o['bullets'])):
            if exact:
                assert H.same_bits(got, ref), (what, i)
            elif ref.size:
                err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
                worst = max(worst, float(err.max()))
                assert (err <= TOL).all(), (what, i, float(err.max()))
    return worst


def _check_observe(games, state, what):
    obs = games.observe().cpu().numpy()
    S, n_rows = games.S, obs.shape[2]
    for i in range(games.n):
        for me in range(S):
            if state['finished'][i]:
                assert (obs[i, me] == -1).all(), (what, i)
                continue
            P, B = int(state['n_planets'][i]), int(state['n_bullets'][i])
            want = ao.features(S, state['ships'][i], state['planets'][i, :P], state['bullets'][i, :B], me, n_rows)
            assert H.same_bits(obs[i, me], want), (what, i, me)


@pytest.mark.gpu
@pytest.mark.parametrize('r,S,PL', FORMS, ids=FORM_IDS)
def test_reset_done_recreates_finished_games_from_the_pool(r, S, PL):
    """astro_reset_done refuses to run without a pool (ASTRO_E_STATE).  With one: every finished game — scattered
    through tiles whose live games hold bullets, padding slots included — equals pool[pool_pick(seed, first_game + g,
    step, M)] bit for bit in its live slots, with meta (nb 0, np, live, tick 0) and its episode + 1 (2^32 - 1 wraps to
    0); live games and every bullet list are untouched.  first_game = 2^32 - 70 (game ids wrap inside the batch), stream
    step 777, a pool of 37 entries and then a pool of 1, pool entries with fewer planets than the games they replace.
    Then observe() equals ao.features bit for bit and one tick equals the oracle (bit for bit in float64, within 1e-5 in
    float32) from the model's state: the stale planet rows a re-created game keeps past its planet count are never read."""
    K = 40
    rs = np.random.RandomState(100 + FORMS.index((r, S, PL)))
    seed, first = 5, (1 << 32) - 70
    games = _batch(r, S, PL, N, K, seed=seed, first_game=first)
    games.set_stream(step=777)
    n_pad = games.n_pad
    cfg = games.config
    dtype = np.float32 if r == 'float' else np.float64
    ids = (first + np.arange(n_pad)) % (1 << 32)

    def run():
        before = games.launches
        assert nat.lib().astro_reset_done(games._h, games._stream()) == E_STATE
        assert games.launches == before
        g = random_games(n_pad, S, PL, K, rs, fin=0.3, max_t=games.schedule.timeout_tick - 2, arena=True)
        g['n_planets'][g['finished']] = PL                       # finished games hold PL planets, pool entries fewer
        g['episode'][g['finished'] & (np.arange(n_pad) % 32 == 13)] = 0xFFFFFFFF
        raw = pack(g, PL, K, dtype, 1, seed=4)
        write_raw(games, raw)
        for M, step_what in ((37, 'pool of 37'), (1, 'pool of 1')):
            pool = H.make_pool(cfg, M, PL)
            assert M == 1 or pool['np'].min() < PL
            lp = _lib_pool(games, pool['ships'], pool['planets'], pool['np'])
            dead = meta_unpack(raw['meta'], PL)[2]
            assert dead[:games.n].any() and (~dead).any()
            nat.check(nat.lib().astro_reset_done(games._h, games._stream()))
            got = read_raw(games)
            picks = rng.pool_pick(seed, ids, np.full(n_pad, 777, dtype=np.uint32), M)
            _check_recreated(got, raw, lp, picks, dead, step_what)
            raw = got
            if M == 37:                                          # finish another set of games (stale nb, np kept) for the next pool
                again = (rs.rand(n_pad) < 0.25) & (np.arange(n_pad) % 32 != 14)
                nbf, npl, _, tk = meta_unpack(raw['meta'], PL)
                raw['meta'] = np.where(again, meta_pack(rs.randint(1, 1024, n_pad), npl, 1, tk, PL), raw['meta']).astype(np.uint32)
                write_raw(games, raw)
        state = unpack(raw)
        assert not state['finished'].any()
        _check_observe(games, state, 'observe after the reset')
        acts = rs.randint(0, 6, (n_pad, S)).astype(np.uint8)
        import torch
        _, _, ev = games.step(torch.from_numpy(acts).cuda())
        outs = _oracle_tick(cfg, games, state, acts, K)
        return _check_tick(games, state, unpack(read_raw(games)), outs, ev.cpu().numpy(), r == 'double', 'tick after the reset')
    forms = [reset_form(r, S, PL)] + ([pack_form(S, PL)] if r == 'float' else [])
    worst = _expect(forms, run)
    print('worst relative error of the tick after the reset %s: %.3g' % ((r, S, PL), worst))


# ------------------------------------------------------------------ auto-reset from the packed pool records

@pytest.mark.gpu
@pytest.mark.parametrize('S,PL', POOL_FORMS, ids=['S=%d PL=%d' % f for f in POOL_FORMS])
def test_auto_reset_reads_the_packed_pool(S, PL):
    """pack_pool_kernel<S, PL>'s records, read by the float32 one-tick kernel on auto-reset: a pool of 53 entries with
    planet counts 1..PL, NaN in every dead planet slot and a non-zero bearing on every ship; every live game one tick
    before the timeout (so every one of them ends and is re-created), game ids wrapping at 2^32.  Each re-created game
    equals pool[pick(seed, first_game + g, step + 1)] as float32 bits in its live slots, with meta (nb 0, np, live,
    tick 0) and its episode + 1; finished games are skipped untouched.  One more tick equals the oracle within 1e-5: no
    tick reads a dead slot of a record."""
    import torch
    K, M = 32, 53
    rs = np.random.RandomState(200 + POOL_FORMS.index((S, PL)))
    seed, first = 9, (1 << 32) - 50
    games = _batch('float', S, PL, N, K, seed=seed, first_game=first)
    n_pad = games.n_pad
    cfg = games.config
    ids = (first + np.arange(n_pad)) % (1 << 32)
    ships = np.concatenate([rs.uniform(-0.9, 0.9, (M, S, 2)), rs.uniform(-0.2, 0.2, (M, S, 2)),
                            rs.uniform(0.5, 6.0, (M, S, 1)) * rs.choice([-1, 1], (M, S, 1))], axis=2)
    npl = 1 + np.arange(M) % PL
    planets = np.concatenate([rs.uniform(-0.8, 0.8, (M, PL, 2)), rs.uniform(-0.1, 0.1, (M, PL, 2))], axis=2)
    planets[np.arange(PL)[None, :] >= npl[:, None]] = np.nan

    def run():
        lp = _lib_pool(games, ships, planets, npl)
        g = random_games(n_pad, S, PL, K, rs, fin=0.1, arena=True)
        g['tick'][:] = games.schedule.timeout_tick
        raw = pack(g, PL, K, np.float32, 0, seed=6)
        write_raw(games, raw)
        games.set_stream(step=41)
        games.step_many(1, None, auto_reset=True)
        got = read_raw(games)
        dead = ~meta_unpack(raw['meta'], PL)[2]                  # every live game ends on this tick and is re-created
        assert dead.sum() > n_pad // 2 and (~dead).any()
        picks = rng.pool_pick(seed, ids, np.full(n_pad, 42, dtype=np.uint32), M)
        # (the tick wrote the new lists, all empty, into the other buffer: compare the games, not the buffers)
        _check_recreated(got, dict(raw, bullets=got['bullets'], cur=got['cur']), lp, picks, dead, 'auto-reset')
        state = unpack(got)
        assert (state['n_bullets'] == 0).all()
        acts = rs.randint(0, 6, (n_pad, S)).astype(np.uint8)
        _, _, ev = games.step(torch.from_numpy(acts).cuda())
        outs = _oracle_tick(cfg, games, state, acts, K)
        return _check_tick(games, state, unpack(read_raw(games)), outs, ev.cpu().numpy(), False, 'tick after the auto-reset')
    worst = _expect([pack_form(S, PL)], run)
    print('worst relative error of the tick after the auto-reset %s: %.3g' % ((S, PL), worst))


# ------------------------------------------------------------------ core.step in every layout it picks

def _single_state(S, npl, nb, r, reload_, t):
    """A float64 State: ships in two corners, npl planets on a ring of radius 0.5, nb bullets in the middle, none of which
    reach a ship in one tick."""
    ships = np.zeros((S, 5))
    ships[:, 0:2] = np.array([[0.9, 0.85], [-0.88, -0.9]])[:S] + r.uniform(-0.02, 0.02, (S, 2))
    ships[:, 2:4], ships[:, 4] = r.uniform(-0.05, 0.05, (S, 2)), r.uniform(-3, 3, S)
    phase = r.uniform(0, 2 * np.pi) + 2 * np.pi * np.arange(npl) / npl
    planets = np.stack([0.5 * np.sin(phase), 0.5 * np.cos(phase), 0.1 * np.cos(phase), -0.1 * np.sin(phase)], axis=1)
    bullets = np.concatenate([r.uniform(-0.55, 0.55, (nb, 2)), r.uniform(-1.5, 1.5, (nb, 2))], axis=1)
    body = lambda a, b: core.Bodies(x=a[:, 0:2].copy(), dx=a[:, 2:4].copy(), b=b)
    return core.State(ships=body(ships, ships[:, 4].copy()), planets=body(planets, None), bullets=body(bullets, None),
                      reload=reload_, t=t), (ships, planets, bullets)


@pytest.mark.gpu
def test_core_step_in_every_layout():
    """core.step (astro_step_single_host: import -> tick -> export of one float64 game under a CUDA graph) equals
    ao.step_one bit for bit for solo and duel games in 4- and 8-slot handles: bullet counts with nb + S = 32 and 33 (either
    side of the handle's cap rounding), one handle stepping 7 then 5 planets (8 slots) or 4 then 2 (4 slots), so that
    its pinned record holds stale planet rows; the fire, plain and timeout codes, the last returning None."""
    r = np.random.RandomState(12)

    def run():
        n_none = 0
        for S in (1, 2):
            cfg = core.SOLO_CONFIG if S == 1 else core.DEFAULT_CONFIG
            fire, plain, timeout = (cfg.reload_time - 0.01, 1.0), (0.0, 1.0), (0.0, cfg.max_time - 0.01)
            for hi, lo in ((7, 5), (4, 2)):
                for total in (32, 33):
                    for npl, (reload_, t) in ((hi, fire), (lo, plain), (lo, fire), (hi, timeout)):
                        state, (sh, pl, bl) = _single_state(S, npl, total - S, r, reload_, t)
                        control = r.randint(0, 6, S)
                        got, reward = core.step(state, control, cfg)
                        want = ao.step_one(cfg, sh, pl, bl, reload_, t, control)
                        what = (S, npl, total, reload_, t)
                        assert (got is None) == want['done'], what
                        assert (np.asarray(reward, dtype=np.float64) == want['reward']).all(), what
                        if got is None:
                            n_none += 1
                            continue
                        assert H.same_bits(np.concatenate([got.ships.x, got.ships.dx, got.ships.b[:, None]], 1), want['ships']), what
                        assert H.same_bits(np.concatenate([got.planets.x, got.planets.dx], 1), want['planets']), what
                        assert H.same_bits(np.concatenate([got.bullets.x, got.bullets.dx], 1).reshape(-1, 4), want['bullets']), what
                        assert got.reload == want['reload'] and got.t == want['t'], what
                        if reload_ == fire[0]:
                            assert len(want['bullets']) > 0 and got.bullets.x.shape[0] <= total, what
        return n_none
    # the graph launches forms that the export and import tests list: no ledger entry of its own
    forms = [f('double', S, PL) for f in (export_form, import_form) for S in (1, 2) for PL in (4, 8)]
    assert _expect(forms, run, listed=False) >= 8


# ------------------------------------------------------------------ ABI errors of export / import

@pytest.mark.gpu
def test_export_and_import_refuse_bad_arguments():
    """astro_export_games / astro_import_games return ASTRO_E_INVALID, launching nothing, for a null arrays struct, a null
    required column (export: every column but episode; import: ships, planets, n_planets; bullets when rows are wanted),
    m > n_games without an index, m < 0 and bullet_rows < 0; m = 0 returns ASTRO_OK and launches nothing.  A valid
    export, and the import of what it returned (through an index), still work after them."""
    games = _batch('float', 2, 4, 64, 8)
    pool = H.make_pool(games.config, 16)
    games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
    games.reset_all()
    L, h, st = nat.lib(), games._h, games._stream()

    def run():
        t, good = games._game_arrays(8, 8)
        before = games.launches
        for fn, required in ((L.astro_export_games, ('ships', 'planets', 'n_planets', 'n_bullets', 'tick', 'finished', 'bullets')),
                             (L.astro_import_games, ('ships', 'planets', 'n_planets', 'bullets'))):
            assert fn(h, None, 8, None, st) == E_INVALID
            for k in required:
                bad = games._arrays_struct(dict(t, **{k: None}), 8)
                assert fn(h, None, 8, C.byref(bad), st) == E_INVALID, (fn, k)
            assert fn(h, None, games.n_pad + 1, C.byref(good), st) == E_INVALID
            assert fn(h, None, -1, C.byref(good), st) == E_INVALID
            assert fn(h, None, 8, C.byref(games._arrays_struct(t, -1)), st) == E_INVALID
            assert fn(h, None, 0, C.byref(good), st) == 0
        assert games.launches == before
        arr = games.get_arrays()
        games.set_arrays(arr['ships'], arr['planets'], arr['n_planets'], arr['bullets'], arr['n_bullets'], arr['tick'],
                         index=np.arange(games.n)[::-1], episode=arr['episode'])
        return arr
    arr = _expect([export_form('float', 2, 4), import_form('float', 2, 4), IMPORT_MAP], run)
    again = games.get_arrays()
    for k in arr:
        assert np.array_equal(again[k], arr[k][::-1]), k
