"""Runs in a process of its own (tests/test_rollout_logs.py): one short followed rollout_device call of a batch of the given
layout under torch.profiler, printing the kernel names it launched as JSON.

A profiling session of its own process keeps CUPTI out of the test process, whose later launch counts (the exact counts
of test_recording_fast_paths_keep_their_launches) must not depend on which tests profiled before them.

    python tests/follow_worker.py SOLO MAX_PLANETS BOT
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def main():
    import torch
    from torch.profiler import ProfilerActivity, profile
    from astro_b200 import core
    from tests.test_rollout_record import _batch, _net
    solo, max_planets, bot = bool(int(sys.argv[1])), int(sys.argv[2]), sys.argv[3]
    cfg = core.DEFAULT_CONFIG._replace(solo=solo, max_planets=max_planets)
    g = _batch(cfg, 256, _net(solo))
    ring = g.record_ring(8, observations=False, follow=[0, 5, 40])
    bots = (bot,) * g.S
    g.rollout_device(3, bots=bots, record=ring)          # (module loading and first launches outside the window)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.rollout_device(3, bots=bots, record=ring)        # 3 ticks: no graph chunk
        torch.cuda.synchronize()
    print(json.dumps(sorted({e.key for e in prof.key_averages()})))


if __name__ == '__main__':
    main()
