#!/usr/bin/env python
"""bench.py — env-steps/s of the batched Astro tick on N B200s, as a fraction of the HBM roofline,
next to the CPU step loop timed on the same box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one game tick (astro.core.step) of every game of the batch.  Workload (BASELINE.json
configs[3] shape, weak scaling): 1,048,576 duel games PER GPU, default planets (max_planets=4),
uniform random controls, bullet pool K=32, finished games re-created from a 4,096-state pool built
by core.create; the population is pre-rolled to its stationary bullet count before timing.  The
state (0.67 GB per GPU) and the controls exceed the 126 MB L2, so no flush is needed between steps.

Numbers on the JSON line:
  value     whole-job env-steps/s, controls already resident in HBM (a ring of pre-generated arrays, one control byte
            per game, a different array every tick), every tick's events written to HBM (three bit planes); CUDA events,
            max over ranks (`per_rank_ms` lists every rank).  The ticks go through astro_tick_many, --fuse ticks per
            launch: games do not interact, so the kernel runs the ticks of a tile back to back and the state travels
            from one tick to the next through L2.  The timed region ends with the episode statistics and their NCCL
            all-reduce (`collective_us` = that part alone).
  per_tick_launch  the same loop as one launch per tick (what a policy in the loop needs) with ITS roofline: this is the
            HBM-bound form (DRAM traffic ~ algorithmic bytes).
  roofline  the dominant kernel of the timed region: algorithmic bytes per launch (device counters) / average launch
            duration against MEASURED_PEAKS.json hbm_gbs; `traffic` = DRAM bytes of an ncu capture of the SAME launch
            shape (or null); `secondary` = the issue-slot numbers of that capture (the fused form is issue-bound).
  e2e       through BatchedGames.rollout_host(): pinned HOST controls in (1 B/game), event planes out (12 B / 32 games),
            copies inside the timed region, pipelined; `closed_loop_value` = step_host: copy in, tick, copy out,
            synchronise on every tick; `byte_form_value` = the round-1 forms (2 + 1 B/game).
  strong    BASELINE configs[3] as stated: 1,048,576 games in TOTAL over the N GPUs (the headline weak-scales).
  fresh_games  the headline loop with pool-free re-creation (every ended game gets the next generate_configs seed).
  rollout   BASELINE configs[4]: 16,384 games x 1,000 ticks, observation -> astro.rl network -> step (rank 0).
  drop_in   astro_b200.core.step on one game, microseconds per call (BASELINE configs[0] shape).
  cpu_baseline  the oracle port of the reference loop on all host cores (rank 0, every N).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'env-steps/sec'
UNIT = 'env-steps/s'
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


# --------------------------------------------------------------------------- multi-rank helpers
def shard_plan(world, rank, games_per_gpu):
    """Env-parallel sharding: rank r owns the contiguous global games [r*n, (r+1)*n)."""
    return dict(first_game=rank * games_per_gpu, n_games=games_per_gpu, total=world * games_per_gpu)


def reduce_stats(stats, dist=None):
    """Sum the int64 counter vector over ranks (the only collective of the path)."""
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def reduce_max(value, device, dist=None):
    import torch
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def algorithmic_bytes(st, S, packed=False, planes=False, events=True, with_reward=False):
    """Bytes the tick must move per the layout in include/astro_b200.h: every live byte of state
    read once and written once, controls read (S bytes per game, 1 when packed), events written (1 byte per game,
    12 per 32 games as bit planes).  st = device counters."""
    per_step = (2 * (4 + 16 * S + 4 * S) + (1 if packed else S) + ((12.0 / 32 if planes else 1) if events else 0)
                + ((4 * S + 1) if with_reward else 0))
    return (st['env_steps'] * per_step + 32 * st['planets_live'] + 16 * (st['bullets_in'] + st['bullets_out']))


# --------------------------------------------------------------------------- BASELINE config #5 and the drop-in
def config5_rollout(args, local, pool):
    """BASELINE configs[4]: self-play rollout, 16,384 games x 1,000 ticks, observation extraction feeding the astro.rl
    policy batch every tick, both ships driven by the network (greedy), auto-reset.  Three forms of the same loop:
    observe() -> PyTorch ValueNetwork -> argmax -> step; observe(shared) -> forward_both; observe() -> the same forward as ONE
    tensor-core kernel (ValueNetwork.forward under no_grad = astro_value_forward); the fused policy kernel
    inside astro_rollout_device (no observation tensor, no host between ticks)."""
    import torch
    from astro_b200 import core, rl
    from astro_b200.batched import BatchedGames
    N, T = args.rollout_games, args.rollout_ticks
    torch.manual_seed(7)
    net = rl.ValueNetwork(solo=False, nout=6).cuda(local)
    with torch.no_grad():
        for prm in net.parameters():
            prm.mul_(3.0)
    out = dict(config='BASELINE configs[4]: %d games x %d ticks, observe -> astro.rl ValueNetwork (both ships) -> step, auto-reset' % (N, T),
               games=N, ticks=T, unit=UNIT)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for form in ('observe+torch', 'observe_shared+forward_both', 'observe -> ValueNetwork.forward (astro_value_forward kernel)',
                 'fused policy kernel (rollout_device)'):
        g = BatchedGames(core.DEFAULT_CONFIG, N, bullet_cap=args.bullet_cap, precision=32, device=local, seed=3)
        g.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        g.reset_all()
        g.set_policy(net)
        buf = {}

        def observe(shared):
            if 'o' not in buf:
                buf['o'] = g.observe(shared=shared)          # (N is a multiple of 32: the view is the whole buffer)
            else:
                g.observe(shared=shared, out=buf['o'])
            return buf['o']

        def loop(ticks):
            with torch.no_grad():
                if form.startswith('fused'):
                    g.rollout_device(ticks, bots=('policy', 'policy'), auto_reset=True)
                    return
                for _ in range(ticks):
                    if form.startswith('observe+'):
                        a = net.forward_torch(observe(False)).argmax(-1).to(torch.uint8)
                    elif form.startswith('observe ->'):
                        a = net(observe(False)).argmax(-1).to(torch.uint8)     # (no_grad, cuda float32: the fused inference kernel)
                    else:
                        a = net.forward_both(observe(True)).argmax(-1).to(torch.uint8)
                    g.step(a, auto_reset=True, want_reward=False)
        loop(3)
        g.stats(clear=True)
        torch.cuda.synchronize()
        e0.record()
        loop(T)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        st = g.stats()
        out[form] = dict(value=st['env_steps'] / (ms * 1e-3), ms_per_tick=ms / T, episodes=st['episodes'])
        del g
    return out


def drop_in_step(args):
    """The drop-in astro_b200.core.step on ONE game (BASELINE configs[0] shape: the reference's own CPU-runnable case):
    microseconds per call of the lean single-game path, beside the oracle port on one host core."""
    from astro_b200 import core, rng
    from oracle import astro_oracle as ao
    cfg = core.DEFAULT_CONFIG
    controls = [rng.actions(5, [0], k, 2)[0] for k in range(400)]
    t_gpu = 0.0
    for warm in (True, False):
        state = core.create(cfg)
        t0 = time.perf_counter()
        for k in range(400):
            nxt, _ = core.step(state, controls[k], cfg)
            state = core.create(cfg) if nxt is None else nxt
        t_gpu = time.perf_counter() - t0
    sh = np.zeros((2, 5)); pl = np.zeros((1, 4)); sh[:, 0] = (-0.5, 0.5); pl[0, 1] = 0.9
    t0 = time.perf_counter()
    for k in range(2000):
        ao.step_one(cfg, sh, pl, np.zeros((0, 4)), 0.0, 0.0, np.array([2, 2]))
    t_cpu = time.perf_counter() - t0
    return dict(api='astro_b200.core.step (one game: pinned record in, import -> tick -> export, record out)',
                us_per_step=1e6 * t_gpu / 400, steps_per_s=400 / t_gpu,
                oracle_port_us_per_step=1e6 * t_cpu / 2000,
                reference_python_us_per_step=202.0,
                reference_note='astro.core.step measured in the build container (SURVEY section 6: 202 us/tick, 1 core); the Python '
                               'reference cannot travel to the GPU box')


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the GPU is under load."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {}
        for n in dir(nv):
            if n.startswith('nvmlClocksThrottleReason') or n.startswith('nvmlClocksEventReason'):
                v = getattr(nv, n)
                if isinstance(v, int) and v:
                    names[v] = n.replace('nvmlClocksThrottleReason', '').replace('nvmlClocksEventReason', '')
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit and bit & (bit - 1) == 0:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join()
        idle = {'GpuIdle', 'None', 'ApplicationsClocksSetting'}
        return dict(sm_mhz=(float(np.median(self.samples)) if self.samples else None), sm_max_mhz=self.max_mhz,
                    reasons=sorted(r for r in self.reasons if r not in idle), samples=len(self.samples))


# --------------------------------------------------------------------------- CPU baseline (oracle)
CPU_GAMES = 65536      # the bounded CPU sample: the same workload on 65,536 games (both the cpu_baseline leg and --impl reference)


class CpuLoop:
    """The oracle port of the reference step loop on all host cores (same workload: duel, default planets,
    counter-stream random controls, auto-reset from a create() pool), warmed up once and timed in segments."""

    def __init__(self, n_games, threads, seed=0, pool_size=1024, warm_ticks=100):
        from astro_b200 import core, rng
        from oracle import astro_oracle as ao
        from astro_b200.pool import make_pool
        self.ao, self.cfg, self.seed, self.threads, self.n = ao, core.DEFAULT_CONFIG, seed, threads, n_games
        self.pool = make_pool(self.cfg, pool_size)
        b = self.b = ao.Batch(n_games, 2, 32)
        pick = rng.pool_pick(seed, np.arange(n_games), np.zeros(n_games, dtype=np.uint32), pool_size)
        b.ships[:], b.planets[:], b.np_[:] = self.pool['ships'][pick], self.pool['planets'][pick], self.pool['np'][pick]
        self.step = 0
        self.run(warm_ticks)

    def run(self, ticks):
        """-> (env-steps done, seconds)"""
        t0 = time.perf_counter()
        st = self.ao.rollout(self.cfg, self.b, self.pool, self.seed, 0, self.step, ticks, threads=self.threads)
        dt = time.perf_counter() - t0
        self.step += ticks
        return int(st[5]), dt


def cpu_baseline(seconds, threads=None):
    threads = threads or os.cpu_count() or 1
    loop = CpuLoop(CPU_GAMES, threads)
    steps, dt = loop.run(40)                                      # calibrate
    ticks = int(max(100, min(200000, seconds * (steps / dt) / CPU_GAMES)))
    steps, dt = loop.run(ticks)
    return dict(value=steps / dt, unit=UNIT, cores=threads, kind='port',
                sample='%d games x %d ticks of the same workload (%.1f s), oracle C port of astro/core.py step with auto-reset, '
                       'one thread per host core' % (CPU_GAMES, ticks, dt))


def run_reference(args):
    """--impl reference: the reference's CPU step loop (oracle port; the Python reference cannot travel to the GPU box) on
    all host cores, same metric / config as our arm.  One "step" = a bounded sample of the workload: `ticks_per_step`
    ticks of CPU_GAMES games, sized after a short calibration so that the timed region lasts >= 2.5 s whatever --steps is
    (a 25 ms region measured thread start-up, not the loop)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    loop = CpuLoop(CPU_GAMES, threads)
    steps, dt = loop.run(40)
    rate0 = steps / dt
    per_step = int(max(1, np.ceil(args.ref_seconds * rate0 / (CPU_GAMES * args.steps))))
    for _ in range(args.warmup):
        loop.run(per_step)
    total, t0 = 0, time.perf_counter()
    for _ in range(args.steps):
        total += loop.run(per_step)[0]
    dt = time.perf_counter() - t0
    rate = total / dt
    sample = ('each step = %d ticks of %d games of the %d-games-per-GPU workload (%.1f s timed), oracle C port of astro/core.py step '
              'with auto-reset, one thread per host core' % (per_step, CPU_GAMES, args.games_per_gpu, dt))
    line = dict(metric=METRIC, value=rate, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f64', data='synthetic', impl='reference', config=workload_config(args),
                cpu_baseline=dict(value=rate, unit=UNIT, cores=threads, kind='port', sample=sample),
                e2e=dict(value=rate, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), flush=True)


def workload_config(args):
    return dict(workload='BASELINE configs[3] shape, weak-scaled: %d duel games per GPU, default planets '
                         '(max_planets=4), uniform random controls, auto-reset from a %d-state create() pool'
                         % (args.games_per_gpu, args.pool),
                games_per_gpu=args.games_per_gpu, bullet_cap=args.bullet_cap, reset_pool=args.pool,
                preroll_ticks=args.preroll, state_precision='fp32 state, fp64-exact predicates',
                ticks_per_launch=args.fuse,
                io_form='one control byte per game (both ships), three event bit planes per tick',
                l2_policy='state (0.67 GB/GPU) and controls exceed the 126 MB L2; no flush between steps; inside a launch the '
                          'ticks of a tile run back to back, so a tile\'s state deliberately stays in L2 from one tick to the next',
                parallelism='env-parallel shards, one process per GPU, NCCL only for the stats reduce')


def bind_to_gpu_numa_node(index):
    """Pins this rank to the CPUs NVML lists as local to its GPU, BEFORE the pinned host buffers are allocated
    (first touch puts them on that NUMA node): the end-to-end leg moves 1.4 MB per tick and GPU through host memory,
    and with several ranks per box a buffer on the far socket costs every copy a trip over the socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and 64 * w + b < n_cpu}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return sorted(cpus)
    except Exception:
        pass
    return None


def profile_entry(ticks_per_launch):
    """ncu summary of the tick kernel captured at this launch shape (profiles/tick_kernel_ncu_summary.json, keyed by
    ticks per launch), or None: DRAM traffic is only printed beside a launch of the shape it was measured on."""
    try:
        prof = json.load(open(os.path.join(ROOT, 'profiles', 'tick_kernel_ncu_summary.json')))
        return prof.get(str(int(round(ticks_per_launch))))
    except Exception:
        return None


DUMP_GAMES = 16384          # --dump-outputs: games in the fixed sample whose state is written
DUMP_BYTES = 60 << 20       # ... and the most the sample may take (a large --bullet-cap shrinks it)


def dump_outputs(out_dir, games, planes, stats):
    """--dump-outputs: what the timed loop hands its caller after its last tick, as float64 DIR/<name>.npy, for comparing
    two builds output for output.  A fixed sample of games (seeded, sorted; every game when there are fewer than
    DUMP_GAMES): their state as get_arrays() returns it (bullet and planet rows past a game's counts zeroed) and their bits
    of that tick's three event planes (ended, ship 0 hit, ship 1 hit); and the 14 episode counters (nat.STAT_NAMES order)."""
    from astro_b200 import _native as nat
    per_game = 8 * (games.S * 5 + nat.MAX_PLANETS * 4 + games.K * 4 + 5 + 3 + 1)    # state, 5 counters, 3 event bits, index
    m = min(games.n, DUMP_GAMES, DUMP_BYTES // per_game)
    idx = np.sort(np.random.default_rng(0).choice(games.n, size=m, replace=False))
    out = games.get_arrays(idx)
    out['bullets'][np.arange(out['bullets'].shape[1])[None, :] >= out['n_bullets'][:, None]] = 0.0
    out['planets'][np.arange(out['planets'].shape[1])[None, :] >= out['n_planets'][:, None]] = 0.0
    words = planes.cpu().numpy().view(np.uint32)                      # [3, n_tiles]: bit g % 32 of word g // 32 is game g
    out['events'] = ((words[:, idx // 32] >> (idx % 32).astype(np.uint32)) & 1).T
    out['game_index'] = idx
    out['episode_stats'] = np.asarray(stats)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a, dtype=np.float64))


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from astro_b200 import core
    from astro_b200 import _native as nat
    from astro_b200.batched import BatchedGames
    from astro_b200.pool import make_pool

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        raise SystemExit('--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run for N>1)' % (args.gpus, world))
    torch.cuda.set_device(local)
    bind_to_gpu_numa_node(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    cfg = core.DEFAULT_CONFIG
    S, K = 2, args.bullet_cap
    pool = make_pool(cfg, args.pool)     # host: core.create over generate_configs (seed 42)
    io_flags = nat.TICK_PACKED_CONTROLS | nat.TICK_EVENT_PLANES
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', FALLBACK_HBM_GBS))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def gather_ms(my_ms):
        """every rank's time, as a list (rank order)"""
        if world == 1:
            return [my_ms]
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = my_ms
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t.cpu()]

    def timed_rollout(n_games, first_game, steps, warmup, fuse, collective=True):
        """The timed region of the headline: `steps` ticks of n_games games on this rank, `fuse` ticks per launch, controls
        resident in HBM (a different array every tick), every tick's events written, then the episode statistics and their
        NCCL all-reduce.  -> dict(ms per rank, counters, launches, games)"""
        games = BatchedGames(cfg, n_games, bullet_cap=K, precision=32, device=local, seed=args.seed, first_game=first_game)
        games.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        games.reset_all()
        flags = nat.TICK_AUTO_RESET | args.tick_flags
        for _ in range(args.preroll):        # reach the stationary population (device counter-stream controls)
            games.step_raw(0, flags)
        torch.cuda.synchronize()
        flags |= args.timed_flags | io_flags
        R = max(8, fuse)
        gen = torch.Generator(device='cpu').manual_seed(1234 + rank)
        host_ring = BatchedGames.pack_controls(torch.randint(0, 6, (R, games.n_pad, S), dtype=torch.uint8, generator=gen)).contiguous().pin_memory()
        dev_ring = host_ring.to(dev)
        events_dev = torch.empty(games.planes_shape(R), dtype=torch.int32, device=dev)

        # (device addresses worked out once: indexing a tensor costs the host microseconds that the timed region of a single
        # launch would count while the GPU idles)
        ring_ptr, ring_stride = dev_ring.data_ptr(), dev_ring[0].numel() * dev_ring.element_size()
        ev_ptr, ev_stride = events_dev.data_ptr(), events_dev[0].numel() * events_dev.element_size()

        def run_steps(k_steps):
            done, n_launch = 0, 0
            while done < k_steps:
                r0 = done % R
                t = min(fuse, k_steps - done, R - r0)
                games.step_many_raw(ring_ptr + r0 * ring_stride, ev_ptr + r0 * ev_stride, t, flags)
                done += t
                n_launch += 1
            return n_launch
        run_steps(warmup)
        games.stats_tensor(clear=True)
        align = torch.zeros(1, device=dev)
        peer = None
        if world > 1:
            dist.all_reduce(align)       # (NCCL warm-up for this size)
            if collective and args.stats_reduce == 'peer':
                # the statistics reduction over peer memory (astro_stats_allreduce: one kernel per rank, P2P stores through
                # NVSwitch); every rank must have mapped the others' buffers, else all of them use NCCL
                if games.stats_peer_init(dist):
                    games.stats_allreduce(clear=True)        # (first touch of the peer mappings)
                    peer = 'peer'
                else:
                    peer = 'nccl (peer exchange unavailable: %s)' % str(games.peer_error or 'on another rank')[:120]
        launches0 = games.launches
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            # the ranks leave the host barrier tens of microseconds apart; a tiny all-reduce in front of the first event
            # lines the STREAMS up, so that the timed region of every rank starts at the same moment on the devices
            dist.all_reduce(align)
        torch.cuda.synchronize() if world == 1 else None
        e0.record()
        n_launches = run_steps(steps)
        if peer == 'peer':
            st_t = games.stats_allreduce(clear=True)     # the episode-statistics reduction, once per rollout: peer memory ...
        else:
            st_t = games.stats_tensor(clear=True)
            if collective:
                reduce_stats(st_t, dist)                 # ... or NCCL
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return dict(games=games, ms=gather_ms(e0.elapsed_time(e1)), stats=dict(zip(nat.STAT_NAMES, (int(x) for x in st_t.cpu().numpy()))),
                    launches=games.launches - launches0, n_launches=n_launches, run_steps=run_steps, flags=flags, stats_reduce=peer or ('nccl' if world > 1 else 'none'),
                    host_ring=host_ring, dev_ring=dev_ring, R=R, last_events=events_dev[(steps - 1) % R])

    plan = shard_plan(world, rank, args.games_per_gpu)
    n = plan['n_games']
    sampler = ClockSampler(local)
    sampler.start()
    main = timed_rollout(n, plan['first_game'], args.steps, args.warmup, args.fuse)
    games, flags, R, run_steps = main['games'], main['flags'], main['R'], main['run_steps']
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, games, main['last_events'], [main['stats'][k] for k in nat.STAT_NAMES])
    ms = max(main['ms'])
    per_rank_ms, timed_launches = [round(x, 4) for x in main['ms']], main['launches']
    total = main['stats']
    value = total['env_steps'] / (ms * 1e-3)

    # the collective alone: episode counters -> device vector -> NCCL all-reduce (what the timed region ends with)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    reps = 20
    t0 = time.perf_counter()
    for _ in range(reps):
        reduce_stats(games.stats_tensor(clear=False), dist)
    torch.cuda.synchronize()
    collective_us = max(gather_ms(1e6 * (time.perf_counter() - t0) / reps))
    collective = dict(used=main['stats_reduce'], nccl_us=collective_us)
    if main['stats_reduce'] == 'peer':
        # the same through astro_stats_allreduce, checked against NCCL on the way
        want = games.stats_tensor(clear=False).clone()
        reduce_stats(want, dist)
        got = games.stats_allreduce(clear=False).clone()
        assert bool((want == got).all()), 'astro_stats_allreduce disagrees with the NCCL all-reduce'
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            games.stats_allreduce(clear=False)
        torch.cuda.synchronize()
        collective['peer_us'] = max(gather_ms(1e6 * (time.perf_counter() - t0) / reps))
        collective_us = collective['peer_us']

    # kernel-only window on this rank (no collective inside): the roofline numbers
    games.stats_tensor(clear=True)
    torch.cuda.synchronize()
    e0.record()
    k_launches = run_steps(args.steps)
    e1.record()
    torch.cuda.synchronize()
    kern_ms = e0.elapsed_time(e1)
    local_stats = games.stats(clear=True)
    alg = algorithmic_bytes(local_stats, S, packed=True, planes=True)
    achieved = alg / (kern_ms * 1e-3) / 1e9
    tpl = args.steps / k_launches
    prof = profile_entry(tpl)
    roofline = dict(bound='hbm', achieved=achieved, peak=peak, unit='GB/s', frac=achieved / peak,
                    traffic=(prof or {}).get('dram_bytes_per_launch'),
                    kernel='tick_f32_kernel<2,true,%s>' % ('true' if args.fuse > 1 else 'false'),
                    peak_source='MEASURED_PEAKS.json hbm_gbs' if peaks else 'fallback',
                    ticks_per_launch=tpl, algorithmic_bytes_per_launch=alg / k_launches,
                    bytes_per_env_step=alg / max(1, local_stats['env_steps']),
                    mean_planets=local_stats['planets_live'] / max(1, local_stats['env_steps']),
                    mean_bullets=local_stats['bullets_in'] / max(1, local_stats['env_steps']),
                    avg_launch_us=1e3 * kern_ms / k_launches,
                    traffic_source=('ncu --set full on a launch of %d ticks (profiles/tick_kernel_ncu_summary.json)' % round(tpl)) if prof else
                                   'no ncu capture at this launch shape: not printed',
                    kind='ALGORITHMIC bytes (every live byte of state read and written once PER TICK) / time. With several ticks of a tile '
                         'per launch most of them never leave L2 (compare traffic): frac says how fast the ticks go relative to a tick-by-tick '
                         'HBM roofline, not how busy DRAM is; the HBM-bound form is per_tick_launch.roofline',
                    secondary=dict(bound='issue', issue_active_pct=(prof or {}).get('issue_active_pct'),
                                   warp_instr_per_tile_tick=((prof or {}).get('warp_instructions') or 0) / (n / 32 * max(1, round(tpl))) if prof else None,
                                   l2_hit_pct=(prof or {}).get('l2_hit_pct'), source='same ncu capture'))

    # the same loop as one launch per tick (a policy between the ticks needs this form): the HBM-bound kernel
    pt_steps = max(R, min(args.steps, 400))
    games.stats_tensor(clear=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for k in range(pt_steps):
        games.step_many_raw(main['dev_ring'][k % R].data_ptr(), 0, 1, flags)
    e1.record()
    torch.cuda.synchronize()
    pt_local = e0.elapsed_time(e1)
    pt_ms = max(gather_ms(pt_local))
    pt_stats = games.stats(clear=True)
    pt_alg = algorithmic_bytes(pt_stats, S, packed=True, planes=False, events=False)
    prof1 = profile_entry(1)
    per_tick = dict(value=world * n * pt_steps / (pt_ms * 1e-3), unit=UNIT, ms_per_step=pt_ms / pt_steps, steps=pt_steps,
                    kernel='tick_f32_kernel<2,true,false>',
                    roofline=dict(bound='hbm', achieved=pt_alg / (pt_local * 1e-3) / 1e9, peak=peak, unit='GB/s',
                                  frac=pt_alg / (pt_local * 1e-3) / 1e9 / peak, traffic=(prof1 or {}).get('dram_bytes_per_launch'),
                                  algorithmic_bytes_per_launch=pt_alg / pt_steps, avg_launch_us=1e3 * pt_local / pt_steps,
                                  issue_active_pct=(prof1 or {}).get('issue_active_pct')))
    per_tick['frac_of_hbm_peak'] = per_tick['roofline']['frac']

    # e2e: the public API with HOST buffers; every tick's controls are copied in from pinned host memory and its events
    # copied out, all inside the timed region (copies of neighbouring ticks overlap the kernel:
    # BatchedGames.rollout_host -> astro_rollout_host).  One control byte per game in, three bit planes per tick out.
    host_ring = main['host_ring']
    E = max(R, (args.e2e_call // R) * R) if args.e2e_steps >= args.e2e_call else R
    e2e_steps = max(E, (max(3, min(max(args.steps, 256), args.e2e_steps)) // E) * E)
    e2e_ring = host_ring if E == R else host_ring.repeat(E // R, 1).pin_memory()
    planes_ring = torch.empty(games.planes_shape(E), dtype=torch.int32).pin_memory()
    games.rollout_host(e2e_ring, planes_ring, auto_reset=True, packed=True, planes=True)      # warm-up: E ticks
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for k in range(e2e_steps // E):
        games.rollout_host(e2e_ring, planes_ring, auto_reset=True, packed=True, planes=True)
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = max(gather_ms(e0.elapsed_time(e1)))
    e2e_value = world * n * e2e_steps / (e2e_ms * 1e-3)
    # closed loop: copy in, tick, copy out, synchronise, EVERY tick (a host policy that needs tick k's events before it
    # gives tick k + 1's controls); the tick is cut into slices of tiles so that copies overlap kernels within the tick
    planes_one = torch.empty(games.planes_shape(), dtype=torch.int32).pin_memory()
    closed_steps = 2 * R
    for k in range(4):
        games.step_host(host_ring[k % R], planes_one, auto_reset=True, packed=True, planes=True)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(closed_steps):
        games.step_host(host_ring[k % R], planes_one, auto_reset=True, packed=True, planes=True)
    closed_ms = max(gather_ms(1e3 * (time.perf_counter() - t0)))
    closed_value = world * n * closed_steps / (closed_ms * 1e-3)
    # closed loop over TWO half-batches on their own streams (astro_tick_host_begin / _end): while one half's tick runs, the
    # other half's events travel back and its next controls travel in; each half still gets its tick k events before it
    # gives its tick k + 1 controls
    halves = []
    for h in range(2):
        gh = BatchedGames(cfg, n // 2, bullet_cap=K, precision=32, device=local, seed=args.seed, first_game=plan['first_game'] + h * (n // 2))
        gh.set_reset_pool_arrays(pool['ships'], pool['planets'], pool['np'])
        gh.reset_all()
        for _ in range(min(args.preroll, 300)):
            gh.step_raw(0, nat.TICK_AUTO_RESET)
        halves.append((gh, torch.cuda.Stream(device=dev), host_ring[:, h * (n // 2):(h + 1) * (n // 2)].contiguous().pin_memory(),
                       torch.empty(gh.planes_shape(), dtype=torch.int32).pin_memory()))
    torch.cuda.synchronize()

    def pingpong(steps):
        for gh, st, ring, pl in halves:
            gh.step_host_begin(ring[0], pl, auto_reset=True, packed=True, planes=True, stream=st)
        for k in range(1, steps):
            for gh, st, ring, pl in halves:
                gh.step_host_end()              # tick k - 1's events of this half are on the host ...
                gh.step_host_begin(ring[k % R], pl, auto_reset=True, packed=True, planes=True, stream=st)   # ... before its tick k controls go in
        for gh, st, ring, pl in halves:
            gh.step_host_end()
    pingpong(8)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    pingpong(closed_steps)
    pp_ms = max(gather_ms(1e3 * (time.perf_counter() - t0)))
    pingpong_value = world * 2 * (n // 2) * closed_steps / (pp_ms * 1e-3)
    del halves
    # ... and the round-1 byte forms (2 control bytes + 1 event byte per game) through the same calls, for comparison
    gen = torch.Generator(device='cpu').manual_seed(99 + rank)
    byte_ring = torch.randint(0, 6, (R, games.n_pad, S), dtype=torch.uint8, generator=gen).pin_memory()
    byte_events = torch.empty((R, games.n_pad), dtype=torch.uint8).pin_memory()
    games.rollout_host(byte_ring, byte_events, auto_reset=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for k in range(max(1, 128 // R)):
        games.rollout_host(byte_ring, byte_events, auto_reset=True)
    e1.record()
    torch.cuda.synchronize()
    byte_value = world * n * R * max(1, 128 // R) / (max(gather_ms(e0.elapsed_time(e1))) * 1e-3)
    clocks = sampler.stop()
    # the fused form's own roofline: instruction issue.  Warp-instructions per tile and tick of the ncu capture of this launch shape x
    # the tiles and ticks of the timed launch / its live duration, against one instruction per scheduler (4 per SM) and clock
    sec = roofline.get('secondary') or {}
    if sec.get('warp_instr_per_tile_tick') and clocks and clocks.get('sm_mhz'):
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        peak_issue = 4.0 * sms * float(clocks['sm_mhz']) * 1e6
        got = sec['warp_instr_per_tile_tick'] * (n / 32) * tpl / (roofline['avg_launch_us'] * 1e-6)
        sec.update(achieved_warp_instr_per_s=got, peak_warp_instr_per_s=peak_issue, frac=got / peak_issue,
                   peak_source='4 schedulers x %d SMs x the SM clock sampled under load (clocks.sm_mhz)' % sms)
    e2e = dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=games.n_pad, d2h_bytes_per_step=games.n_tiles * 12, steps=e2e_steps,
               api='BatchedGames.rollout_host(packed=True, planes=True) -> astro_rollout_host (copies overlap the kernel)',
               ticks_per_call=E, loop='open: the controls of a call\'s %d ticks are known up front' % E,
               closed_loop_value=pingpong_value,
               closed_loop_api='two half-batches alternating through BatchedGames.step_host_begin / step_host_end (astro_tick_host_begin / '
                               '_end) on their own streams: every half gets its tick k events on the host before its tick k + 1 controls go in',
               closed_loop_single_batch_value=closed_value,
               closed_loop_single_batch_api='BatchedGames.step_host(packed=True, planes=True) -> astro_tick_host: copy in, tick, copy out, '
                                            'synchronise, every tick, one batch (two slices of tiles on internal streams)',
               unpipelined_value=closed_value,
               byte_form_value=byte_value, byte_form_bytes_per_step=[games.n_pad * S, games.n_pad])
    del games, main
    torch.cuda.empty_cache()

    # BASELINE config #4 as stated: 1,048,576 games in total, sharded across the GPUs (strong scaling)
    strong = None
    if args.strong_total > 0 and args.strong_total % (32 * world) == 0:
        per = args.strong_total // world
        sr = timed_rollout(per, rank * per, args.steps, args.warmup, args.fuse)
        s_ms = max(sr['ms'])
        strong = dict(config='BASELINE configs[3] as stated: %d games in total, %d per GPU' % (args.strong_total, per),
                      games_total=args.strong_total, games_per_gpu=per, n_gpus=world, value=sr['stats']['env_steps'] / (s_ms * 1e-3),
                      unit=UNIT, ms_per_step=s_ms / args.steps, ticks_per_launch=args.fuse, scaling='strong')
        del sr
        torch.cuda.empty_cache()

    # fresh-game mode (no reset pool: every re-creation takes the next config of the generate_configs stream), same loop
    fresh = None
    if not args.no_fresh:
        gf = BatchedGames(cfg, n, bullet_cap=K, precision=32, device=local, seed=args.seed, first_game=plan['first_game'])
        gf.enable_fresh_games(quota=48, skip=rank * (1 << 26))
        gf.reset_all()
        f_flags = nat.TICK_AUTO_RESET | args.tick_flags
        for _ in range(min(args.preroll, 300) // 20):
            gf.step_many_raw(0, 0, 20, f_flags)
        gf.stats_tensor(clear=True)
        f_steps = max(args.fuse, (min(max(args.steps, 200), 640) // args.fuse) * args.fuse)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(f_steps // args.fuse):
            gf.step_many_raw(0, 0, args.fuse, f_flags)
        e1.record()
        torch.cuda.synchronize()
        f_ms = max(gather_ms(e0.elapsed_time(e1)))
        f_st = gf.stats(clear=True)
        fresh = dict(value=world * f_st['env_steps'] / (f_ms * 1e-3) if world == 1 else world * n * f_steps / (f_ms * 1e-3), unit=UNIT,
                     ms_per_step=f_ms / f_steps, steps=f_steps, ticks_per_launch=args.fuse, quota=48, awaiting=f_st['awaiting'],
                     episodes_rank0=f_st['episodes'],
                     note='astro_fresh_games_enable: every game that ends is re-created by core.create from the NEXT seed of '
                          'core.generate_configs (host MT19937 = numpy RandomState); controls from the device counter stream')
        del gf
        torch.cuda.empty_cache()

    # the other ranks are done: they leave before rank 0 times the CPU legs (a rank waiting in a barrier spins on a core)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        rollout = None if args.no_rollout else config5_rollout(args, local, pool)
        drop_in = None if args.no_rollout else drop_in_step(args)
        cpu = None if args.no_cpu_baseline else cpu_baseline(args.cpu_seconds)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling='weak', vs_baseline=None,
                    dtype='f32', data='synthetic', config=workload_config(args), roofline=roofline,
                    cpu_baseline=cpu, clocks=clocks, e2e=e2e, gpu_launches=timed_launches,
                    per_tick_launch=per_tick, per_rank_ms=per_rank_ms, collective_us=collective_us, collective=collective, strong=strong, fresh_games=fresh, rollout=rollout, drop_in=drop_in,
                    episode_stats={k: total[k] for k in ('episodes', 'wins0', 'wins1', 'both_lost', 'timeouts', 'overflow', 'bad_controls')})
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=100)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--games-per-gpu', type=int, default=1 << 20)
    ap.add_argument('--bullet-cap', type=int, default=32)
    ap.add_argument('--pool', type=int, default=4096)
    ap.add_argument('--preroll', type=int, default=600)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--e2e-steps', type=int, default=256)
    ap.add_argument('--e2e-call', type=int, default=128, help='ticks per rollout_host call of the e2e leg')
    ap.add_argument('--cpu-seconds', type=float, default=10.0)
    ap.add_argument('--ref-seconds', type=float, default=4.0, help='--impl reference: length of the timed region')
    ap.add_argument('--strong-total', type=int, default=1 << 20, help='BASELINE configs[3] as stated: games in total over all GPUs (0 = skip)')
    ap.add_argument('--rollout-games', type=int, default=16384)
    ap.add_argument('--rollout-ticks', type=int, default=1000)
    ap.add_argument('--no-rollout', action='store_true', help='skip the config #5 / drop-in legs')
    ap.add_argument('--no-fresh', action='store_true', help='skip the fresh-game-mode leg')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--stats-reduce', default='peer', choices=['peer', 'nccl'], help='N > 1: the episode-statistics reduction through astro_stats_allreduce (peer memory) or NCCL')
    ap.add_argument('--fuse', type=int, default=64, help='ticks per launch of the timed loop (astro_tick_many); 1 = one launch per tick')
    ap.add_argument('--tick-flags', type=int, default=0, help='extra ASTRO_TICK_* bits (kernel A/B)')
    ap.add_argument('--timed-flags', type=int, default=0, help='extra tick bits after the pre-roll (experiment builds)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what their last tick handed back (rank 0: a fixed sample of game states '
                         'and their events, and the episode counters) as float64 DIR/<name>.npy')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
