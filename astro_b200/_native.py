"""ctypes binding of include/astro_b200.h.  There is no CPU fallback: if the CUDA library is
missing this module raises, and every compute entry point needs a CUDA device."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('ASTRO_B200_LIB') or os.path.join(HERE, 'libastro_b200.so')   # env: A/B builds

ABI_VERSION = 5
TILE = 32
MAX_PLANETS = 4
MAX_PLANETS_WIDE = 8     # AstroConfig.planet_slots = 8: games of up to eight planets
MAX_BULLET_CAP = 1023
MAX_TICKS = 262143
MAX_TICKS_WIDE = 131071   # 17-bit tick counter of 8-slot batches
SINCOS_RANGE = 71476       # |bearing| over which util.direction (numpy float32 sin/cos) is reproduced bit for bit
N_STATS = 14
STAT_NAMES = ('episodes', 'wins0', 'wins1', 'both_lost', 'timeouts', 'env_steps', 'bullets_spawned',
              'overflow', 'planets_live', 'bullets_in', 'bullets_out', 'skipped', 'bad_controls', 'awaiting')

EV_HIT0, EV_HIT1, EV_TIMEOUT, EV_FIRED, EV_OVERFLOW, EV_SKIPPED, EV_BAD_CONTROL, EV_AWAIT = 1, 2, 4, 8, 16, 32, 64, 128
EV_DONE_MASK = 7
TICK_AUTO_RESET, TICK_NO_STATS, TICK_GENERIC_KERNEL, TICK_CREATE_DTYPES, TICK_ALL_CREATE_DTYPES = 1, 2, 4, 8, 16
TICK_PACKED_CONTROLS, TICK_EVENT_PLANES = 32, 64

EXPORTS = ('astro_abi_version', 'astro_last_error', 'astro_batch_create', 'astro_batch_destroy',
           'astro_batch_bind', 'astro_set_schedule', 'astro_set_stream', 'astro_set_reset_pool',
           'astro_tick', 'astro_tick_host', 'astro_rollout_host', 'astro_reset_done', 'astro_observe', 'astro_stats',
           'astro_launch_count', 'astro_script_controls', 'astro_create_games', 'astro_observe_shared', 'astro_policy_set_weights',
           'astro_policy_controls', 'astro_rollout_device', 'astro_bullet_buffer', 'astro_set_bullet_buffer', 'astro_tick_many', 'astro_explore_controls', 'astro_set_exploration',
           'astro_tick_host_begin', 'astro_tick_host_end', 'astro_fresh_games_enable', 'astro_fresh_games_reset_all',
           'astro_fresh_games_refill', 'astro_fresh_games_positions', 'astro_config_seeds', 'astro_nstep_experiences', 'astro_export_games', 'astro_import_games', 'astro_single_game_bytes', 'astro_step_single_host',
           'astro_stats_peer_create', 'astro_stats_peer_open', 'astro_stats_allreduce', 'astro_value_forward', 'astro_value_forward_views',
           'astro_rollout_device_record', 'astro_rollout_device_follow')


class AstroConfig(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        'gravity', 'dt', 'max_time', 'reload_time', 'bullet_speed', 'ship_thrust', 'ship_rspeed',
        'ship_radius', 'planet_mass', 'planet_radius')] + [('solo', C.c_int32), ('planet_slots', C.c_int32)]


class AstroBuffers(C.Structure):
    _fields_ = [('ships', C.c_void_p), ('ship_b', C.c_void_p), ('planets', C.c_void_p),
                ('bullets', C.c_void_p), ('meta', C.c_void_p), ('episode', C.c_void_p)]


class AstroResetPool(C.Structure):
    _fields_ = [('ships', C.c_void_p), ('planets', C.c_void_p), ('np', C.c_void_p),
                ('size', C.c_int32), ('reserved', C.c_int32)]


class AstroCreateConfig(C.Structure):
    _fields_ = [('inner_ship_position', C.c_double), ('outer_ship_position', C.c_double), ('planet_orbit', C.c_double),
                ('max_planets', C.c_int32), ('reserved', C.c_int32)]


class AstroGameArrays(C.Structure):
    _fields_ = [('ships', C.c_void_p), ('planets', C.c_void_p), ('bullets', C.c_void_p), ('n_planets', C.c_void_p),
                ('n_bullets', C.c_void_p), ('tick', C.c_void_p), ('finished', C.c_void_p), ('episode', C.c_void_p),
                ('bullet_rows', C.c_int32), ('reserved', C.c_int32)]


class AstroRecordRing(C.Structure):
    _fields_ = [('ticks', C.c_int32), ('n_rows', C.c_int32), ('controls', C.c_void_p), ('events', C.c_void_p),
                ('observations', C.c_void_p)]


class AstroFollowRing(C.Structure):
    _fields_ = [('m', C.c_int32), ('reserved', C.c_int32), ('index', C.c_void_p), ('ships', C.c_void_p), ('planets', C.c_void_p),
                ('bullets', C.c_void_p), ('info', C.c_void_p)]


class AstroSingleGame(C.Structure):
    _fields_ = [('ships', C.c_double * 5 * 2), ('planets', C.c_double * 4 * MAX_PLANETS_WIDE),
                ('n_planets', C.c_int32), ('n_bullets', C.c_int32), ('tick', C.c_int32), ('reserved', C.c_int32),
                ('episode', C.c_uint32), ('finished', C.c_uint8 * 4), ('control', C.c_uint8 * (TILE * 2)),
                ('events', C.c_uint8 * TILE)]


BOT_STREAM, BOT_SCRIPT, BOT_POLICY, BOT_NOTHING, BOT_EXPLORE = 0, 1, 2, 3, 4
BOT_MODES = {'stream': BOT_STREAM, 'random': BOT_STREAM, 'script': BOT_SCRIPT, 'policy': BOT_POLICY, 'nothing': BOT_NOTHING, 'explore': BOT_EXPLORE}


class AstroError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded CUDA library.  Raises if it has not been built — there is no other path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'astro_b200: %s is missing. Build it with `python -m astro_b200.build` '
            '(nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
    L.astro_abi_version.restype = C.c_int
    L.astro_last_error.restype = C.c_char_p
    L.astro_batch_create.argtypes = [C.POINTER(AstroConfig), i32, i32, i32, i32, C.POINTER(vp)]
    L.astro_batch_destroy.argtypes = [vp]
    L.astro_batch_bind.argtypes = [vp, C.POINTER(AstroBuffers)]
    L.astro_set_schedule.argtypes = [vp, vp, i32, i32]
    L.astro_set_stream.argtypes = [vp, u32, i64, u32]
    L.astro_set_reset_pool.argtypes = [vp, C.POINTER(AstroResetPool)]
    L.astro_tick.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    L.astro_tick_host.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    L.astro_tick_many.argtypes = [vp, vp, vp, vp, vp, i32, i32, vp]
    L.astro_tick_host_begin.argtypes = [vp, vp, vp, i32, vp]
    L.astro_tick_host_end.argtypes = [vp]
    L.astro_fresh_games_enable.argtypes = [vp, C.POINTER(AstroCreateConfig), u32, i64, i32, vp]
    L.astro_fresh_games_reset_all.argtypes = [vp, vp]
    L.astro_fresh_games_refill.argtypes = [vp, vp]
    L.astro_fresh_games_positions.argtypes = [vp, vp, vp, C.POINTER(i64), vp]
    L.astro_config_seeds.argtypes = [u32, i64, i64, vp]
    L.astro_nstep_experiences.argtypes = [vp, vp, i32, i32, C.c_double, vp, vp, vp, vp, vp]
    L.astro_explore_controls.argtypes = [vp, C.c_double, C.c_double, u32, vp, vp, i32, vp]
    L.astro_set_exploration.argtypes = [vp, C.c_double, C.c_double, u32, vp]
    L.astro_rollout_host.argtypes = [vp, vp, vp, i32, i32, vp]
    L.astro_reset_done.argtypes = [vp, vp]
    L.astro_observe.argtypes = [vp, vp, i32, vp]
    L.astro_stats.argtypes = [vp, vp, i32, vp]
    L.astro_value_forward.argtypes = [vp, vp, i32, i32, vp, vp]
    L.astro_value_forward_views.argtypes = [vp, vp, i32, i32, vp, vp, i32, vp, vp]
    L.astro_stats_peer_create.argtypes = [vp, i32, i32, vp]
    L.astro_stats_peer_open.argtypes = [vp, vp]
    L.astro_stats_allreduce.argtypes = [vp, vp, i32, vp]
    L.astro_observe_shared.argtypes = [vp, vp, i32, vp]
    L.astro_policy_set_weights.argtypes = [vp, vp, i32, i32]
    L.astro_policy_controls.argtypes = [vp, vp, vp, i32, vp]
    L.astro_rollout_device.argtypes = [vp, i32, i32, i32, C.c_double, C.c_double, vp, vp, i32, vp]
    L.astro_rollout_device_record.argtypes = [vp, i32, i32, i32, C.c_double, C.c_double, vp, C.POINTER(AstroRecordRing), i32, vp]
    L.astro_rollout_device_follow.argtypes = [vp, i32, i32, i32, C.c_double, C.c_double, vp, C.POINTER(AstroRecordRing),
                                              C.POINTER(AstroFollowRing), i32, vp]
    L.astro_create_games.argtypes = [vp, C.POINTER(AstroCreateConfig), vp, i32, vp, vp, vp, vp]
    L.astro_script_controls.argtypes = [vp, C.c_double, C.c_double, vp, vp]
    L.astro_export_games.argtypes = [vp, vp, i32, C.POINTER(AstroGameArrays), vp]
    L.astro_import_games.argtypes = [vp, vp, i32, C.POINTER(AstroGameArrays), vp]
    L.astro_single_game_bytes.argtypes = [i32]
    L.astro_single_game_bytes.restype = i64
    L.astro_step_single_host.argtypes = [vp, vp, vp, i32, vp]
    L.astro_bullet_buffer.argtypes = [vp]
    L.astro_set_bullet_buffer.argtypes = [vp, i32]
    L.astro_launch_count.argtypes = [vp]
    L.astro_launch_count.restype = i64
    if L.astro_abi_version() != ABI_VERSION:
        raise ImportError('astro_b200: %s has ABI %d, expected %d — rebuild it'
                          % (LIB_PATH, L.astro_abi_version(), ABI_VERSION))
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise AstroError('astro_b200 error %d: %s' % (rc, lib().astro_last_error().decode()))
