"""The value network on the observations of 16,384 games in the stationary population, forms timed in one process,
alternating (median and range over rounds of 20 calls each):
  astro_value_forward on observe()                       net(obs)                 value_forward_kernel, two views in memory
  forward_both on observe(shared=True), kernel           net.forward_both(shared) the same kernel reading ship 1's columns
  forward_both on observe(shared=True), PyTorch          net.forward_both_torch(shared)
and, for one 100-tick window of an explore rollout of those games (n_steps 100, carried pairs included), the values of
every replay pair: RecordRing.experience_values against experiences() + net() on its two feature tensors — time and peak
allocated memory.  Prints the GPU's name and power limit beside the numbers."""
import os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from astro_b200 import core, rl
from astro_b200.batched import BatchedGames


def power_limit():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                              capture_output=True, text=True, timeout=30).stdout.strip() or 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def timed(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / calls      # us per call


def summary(ts):
    ts = sorted(ts)
    return '%.2f us (median of %d rounds, range %.2f .. %.2f)' % (ts[len(ts) // 2], len(ts), ts[0], ts[-1])


print('GPU: %s, power limit %s' % (torch.cuda.get_device_name(0), power_limit()))
N, T, n_steps = 16384, 100, 100
g = BatchedGames(core.DEFAULT_CONFIG, N, bullet_cap=32, precision=32, device=0)
g.set_reset_pool_on_device(4096)
g.reset_all()
g.step_many(300, None, auto_reset=True)
torch.manual_seed(0)
net = rl.ValueNetwork(solo=False, nout=6).cuda()
obs, shared = g.observe(), g.observe(shared=True)
forms = (('astro_value_forward on observe()', lambda: net(obs)),
         ('forward_both on observe(shared=True), kernel', lambda: net.forward_both(shared)),
         ('forward_both on observe(shared=True), PyTorch', lambda: net.forward_both_torch(shared)))
with torch.no_grad():
    for _, f in forms:
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    times = {name: [] for name, _ in forms}
    for _ in range(15):
        for name, f in forms:
            times[name].append(timed(f, 20))
    for name, _ in forms:
        print('%-48s %s per call (16,384 games x 2 views x 36 rows)' % (name, summary(times[name])))
    want = net(obs)
    print('forward_both kernel == astro_value_forward on both views, bit for bit: %s; max |kernel - PyTorch| = %.3g'
          % (torch.equal(net.forward_both(shared), want), float((net.forward_both_torch(shared) - want).abs().max())))

    # one 100-tick window of replay pairs: a second window, so that the first one's pending pairs are carried into it
    g.set_policy(net)
    g.set_exploration(1.0, 0.1, seed=5)
    ring = g.record_ring(n_steps + T + 1)
    carry = None
    for _ in range(2):
        g.rollout_device(T, bots='explore', record=ring)
        rew, dis, nxt, carry = g.nstep_experiences(ring.window_events(T), carry, n_steps=n_steps, discount=0.995)

    def values():
        return ring.experience_values(net, rew, dis, nxt, n_steps)

    def materialised():
        exp = ring.experiences(rew, dis, nxt, n_steps)
        return net(exp['features']), net(exp['next_features'])

    E = int((nxt >= -1).sum())
    for name, f in (('experience_values', values), ('experiences + 2 x net()', materialised)):
        f()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ms = sorted(timed(f, 3) / 1e3 for _ in range(3))
        peak = torch.cuda.max_memory_allocated() - base
        print('%-26s %.2f ms per window (median of 3 x 3 calls, range %.2f .. %.2f), peak allocated %.3f GB '
              '(E = %d pairs, one E x 36 x 15 float32 tensor = %.2f GB)' % (name, ms[1], ms[0], ms[2], peak / 1e9, E,
                                                                           E * ring.n_rows * 15 * 4 / 1e9))
    v, (q, nq) = values(), materialised()
    print('experience_values == net(experiences()), bit for bit: %s' % (torch.equal(v['q'], q) and torch.equal(v['next_q'], nq)))
