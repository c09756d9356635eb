"""What 8 planet slots cost: the float32 tick at 1,048,576 duel games, random controls (the counter stream), auto-reset
from a reset pool created on the device, in four setups —

    max_planets = 4 in a 4-slot batch (today's layout)    max_planets = 4 in an 8-slot batch
    max_planets = 6 (8 slots)                             max_planets = 8 (8 slots)

each timed at one launch per tick and at 20 and 64 ticks per launch (astro_tick_many).  Per run: env-steps/s, us per
tick, the mean live planets P and bullets B per env-step from the device counters, and the algorithmic HBM traffic of
DESIGN.md section 5 — 91 + 32 P + 16 (B_in + B_out) bytes per env-step — over the time, against the HBM peak of the
card's data sheet (7.7 TB/s for a B200).  The card's name and power limit are read in the same run.

    python tools/bench_planets.py [--games 1048576] [--ticks 640] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12   # bytes/s, B200 data sheet (one GPU)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = 'unknown'
    return name, out


def run(setup, n_games, ticks, per_launch, pool_size, warmup):
    import torch
    from astro_b200 import core
    from astro_b200.batched import BatchedGames
    cfg = core.DEFAULT_CONFIG._replace(max_planets=setup['max_planets'])
    g = BatchedGames(cfg, n_games, bullet_cap=32, precision=32, seed=1, planet_slots=setup['slots'])
    g.set_reset_pool_on_device(pool_size)
    g.reset_all()
    for _ in range(0, warmup, per_launch):        # steady state: bullets in the air, games of every age
        g.step_many(per_launch, None, auto_reset=True)
    torch.cuda.synchronize()
    g.stats(clear=True)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(ticks // per_launch):
        g.step_many(per_launch, None, auto_reset=True)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    st = g.stats()
    steps = st['env_steps']
    P, b_in, b_out = st['planets_live'] / steps, st['bullets_in'] / steps, st['bullets_out'] / steps
    bytes_step = 91 + 32 * P + 16 * (b_in + b_out)
    rate = steps / (ms * 1e-3)
    return dict(setup=setup['name'], slots=g.PL, ticks_per_launch=per_launch, env_steps=steps,
                env_steps_per_s=rate, us_per_tick=ms * 1e3 / (steps / n_games), P=P, B_in=b_in, B_out=b_out,
                bytes_per_step=bytes_step, hbm_GBps=bytes_step * rate / 1e9, hbm_share=bytes_step * rate / HBM_PEAK)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--games', type=int, default=1 << 20)
    ap.add_argument('--ticks', type=int, default=640)
    ap.add_argument('--warmup', type=int, default=128)
    ap.add_argument('--pool', type=int, default=16384)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    setups = [dict(name='max_planets=4, 4 slots', max_planets=4, slots=4),
              dict(name='max_planets=4, 8 slots', max_planets=4, slots=8),
              dict(name='max_planets=6', max_planets=6, slots=8),
              dict(name='max_planets=8', max_planets=8, slots=8)]
    name, power = card()
    print('card: %s | power.limit, clocks.max.sm: %s | %d games, %d timed ticks per run' % (name, power, a.games, a.ticks))
    print('%-24s %6s %10s %12s %10s %6s %6s %6s %8s %9s %7s' % ('setup', 'slots', 'ticks/lnch', 'env-steps/s', 'us/tick',
                                                             'P', 'B_in', 'B_out', 'B/step', 'GB/s', 'of HBM'))
    rows = []
    for s in setups:
        for per_launch in (1, 20, 64):
            ticks = max(per_launch, a.ticks // per_launch * per_launch)
            r = run(s, a.games, ticks, per_launch, a.pool, a.warmup)
            rows.append(r)
            print('%-24s %6d %10d %12.4g %10.1f %6.3f %6.2f %6.2f %8.1f %9.1f %6.1f%%' % (
                r['setup'], r['slots'], per_launch, r['env_steps_per_s'], r['us_per_tick'], r['P'], r['B_in'], r['B_out'],
                r['bytes_per_step'], r['hbm_GBps'], 100 * r['hbm_share']), flush=True)
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(dict(card=name, power_limit_max_sm_clock=power, games=a.games, rows=rows), f, indent=1)


if __name__ == '__main__':
    main()
