"""What following games for their logs costs (record_ring(..., follow=games), astro_rollout_device_follow): us per tick of
rollout_device at 16,384 duel games for ScriptBot against ScriptBot, policy against ScriptBot, explore against explore and
counter-stream controls, each without a ring, with a ring of controls and events, and with that ring following 1, 64 and
1,024 games (spread over the batch).  Following gives up the many-tick launches of the scripted and counter-stream rollouts:
every tick becomes follow -> bots -> tick.  Only the device rollout is timed, not the host's conversion of the rows into
core.Games (GameRecorder.rollout).  Calls of --call ticks into a ring of --call + 1 rows, timed with CUDA events after
--warmup calls.  The card's name and power limit are read in the same run.

    python tools/bench_follow.py [--call 100] [--calls 5] [--json out.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_planets import card  # noqa: E402

N_GAMES = 16384
RECORDS = ('none', 'ring', 'follow 1', 'follow 64', 'follow 1024')


def run(bots, record, call, calls, warmup):
    import numpy as np
    import torch
    from astro_b200 import core, rl
    from astro_b200.batched import BatchedGames
    g = BatchedGames(core.DEFAULT_CONFIG, N_GAMES, bullet_cap=32, precision=32, seed=1)
    g.set_reset_pool_on_device(16384)
    g.reset_all()
    torch.manual_seed(0)
    g.set_policy(rl.ValueNetwork(solo=False, nout=6).cuda())
    g.set_exploration(1.0, 0.1, seed=0)
    ring = None
    if record != 'none':
        m = int(record.split()[1]) if record.startswith('follow') else 0
        follow = [int(i) for i in np.linspace(0, N_GAMES - 1, m).astype(int)] if m else None
        ring = g.record_ring(call + 1, observations=False, follow=follow)
    for _ in range(warmup):
        g.rollout_device(call, bots=bots, record=ring)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(calls):
        g.rollout_device(call, bots=bots, record=ring)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1)
    return dict(games=N_GAMES, bots='-'.join(bots), record=record, ticks=call * calls, us_per_tick=ms * 1e3 / (call * calls))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=100, help='ticks per rollout_device call (the ring has one row more)')
    ap.add_argument('--calls', type=int, default=5, help='timed calls per setup')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    name, power = card()
    print('card: %s | power.limit, clocks.max.sm: %s | %d games, %d ticks per call, %d timed calls'
          % (name, power, N_GAMES, a.call, a.calls))
    print('%-16s %-12s %10s %10s' % ('bots', 'record', 'us/tick', 'vs none'))
    rows, base = [], {}
    for bots in (('script', 'script'), ('policy', 'script'), ('explore', 'explore'), ('stream', 'stream')):
        for rec in RECORDS:
            r = run(bots, rec, a.call, a.calls, a.warmup)
            base.setdefault(r['bots'], r['us_per_tick'])
            r['vs_none'] = r['us_per_tick'] / base[r['bots']]
            rows.append(r)
            print('%-16s %-12s %10.2f %9.3fx' % (r['bots'], rec, r['us_per_tick'], r['vs_none']), flush=True)
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(dict(card=name, power=power, rows=rows), f, indent=1)


if __name__ == '__main__':
    main()
