"""What the per-tick recording ring costs (BatchedGames.rollout_device(..., record=ring), astro_rollout_device_record): us per
tick of rollout_device at 16,384 duel games for ScriptBot against ScriptBot (the bots inside the tick), policy against policy,
explore against explore (rl.QBotTrainer's acting policy) and counter-stream controls, each without a ring, with a ring of
controls and events, and with a ring that also holds every tick's observation; then the counter stream at 1,048,576 games
without and with a ring of controls and events (a ring of observations would take 2.2 GB per row there).  Calls of --call
ticks into a ring of --call + 1 rows, the n-step window of rl.QBotTrainer; timed with CUDA events after --warmup calls.  The
card's name and power limit are read in the same run.

    python tools/bench_record.py [--call 100] [--calls 5] [--json out.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_planets import card  # noqa: E402


def run(n_games, bots, record, call, calls, warmup):
    import torch
    from astro_b200 import core, rl
    from astro_b200.batched import BatchedGames
    g = BatchedGames(core.DEFAULT_CONFIG, n_games, bullet_cap=32, precision=32, seed=1)
    g.set_reset_pool_on_device(16384)
    g.reset_all()
    torch.manual_seed(0)
    g.set_policy(rl.ValueNetwork(solo=False, nout=6).cuda())
    g.set_exploration(1.0, 0.1, seed=0)
    ring = None if record == 'none' else g.record_ring(call + 1, observations=record == 'observations')
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
    return dict(games=n_games, bots='-'.join(bots), record=record, ticks=call * calls, us_per_tick=ms * 1e3 / (call * calls))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--call', type=int, default=100, help='ticks per rollout_device call (the ring has one row more)')
    ap.add_argument('--calls', type=int, default=5, help='timed calls per setup')
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--json', default=None)
    a = ap.parse_args()
    name, power = card()
    print('card: %s | power.limit, clocks.max.sm: %s | %d ticks per call, %d timed calls' % (name, power, a.call, a.calls))
    setups = [(16384, bots, rec) for bots in (('script', 'script'), ('policy', 'policy'), ('explore', 'explore'), ('stream', 'stream'))
              for rec in ('none', 'controls+events', 'observations')]
    setups += [(1 << 20, ('stream', 'stream'), rec) for rec in ('none', 'controls+events')]
    print('%9s %-16s %-16s %10s %10s' % ('games', 'bots', 'record', 'us/tick', 'vs none'))
    rows, base = [], {}
    for n, bots, rec in setups:
        r = run(n, bots, rec, a.call, a.calls, a.warmup)
        key = (n, r['bots'])
        base.setdefault(key, r['us_per_tick'])
        r['vs_none'] = r['us_per_tick'] / base[key]
        rows.append(r)
        print('%9d %-16s %-16s %10.2f %9.3fx' % (n, r['bots'], rec, r['us_per_tick'], r['vs_none']), flush=True)
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(dict(card=name, power=power, rows=rows), f, indent=1)


if __name__ == '__main__':
    main()
