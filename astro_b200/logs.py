"""Game logs of batched rollouts in the reference's JSONL format.

The reference records a game as `Game(config, winner, ticks)` with one `Tick(state, control,
reward, bot_data)` per step, `state` being the PRE-step state (core.play, core.py:377-410), and
writes it with `save_log` (core.py:413-427; util.to_jsonable, util.py:13-30): a header line
{config, winner}, then one Tick per line, arrays as {_values, _shape}, namedtuples tagged
`_type: astro.core:<Name>` — the format `static/astro.js:82-112` replays.

`GameRecorder` follows a handful of game slots of a `BatchedGames` rollout: before every tick it
gathers their states from HBM (a few hundred bytes per followed game, nothing else leaves the
GPU), after the tick their rewards; a followed game that ends becomes a `core.Game` (and, with a
folder given, a .jsonl file), and with auto-reset the slot's next episode starts a new one.

`GameRecorder.rollout` logs the same games through `BatchedGames.rollout_device` instead: a RecordRing
that follows them (record_ring(..., follow=indices)) receives their states from a small kernel before
every tick (astro_rollout_device_follow), next to every tick's controls and event byte; the rewards
are rebuilt from the event bytes (event_rewards).  The logs are the ones a step() loop would write.
"""
import os

import numpy as np

from . import _native as nat
from . import core


def event_rewards(events, S, solo):
    """The per-ship rewards step() returns for ticks with these ASTRO_EV_* bytes (float32 [..., S]), as the tick kernel
    fills its reward array (core.py:253-260): when a ship is hit, -1 for each ship hit and +1 for the other; on a timeout
    the config's timeout reward (1 for solo games, 0 for duels); 0 otherwise."""
    ev = np.asarray(events).astype(np.int64)[..., None]
    hit = (ev >> np.arange(S)) & 1
    timeout = np.float32(1.0 if solo else 0.0)
    r = np.where((ev & (nat.EV_HIT0 | nat.EV_HIT1)) != 0, 1 - 2 * hit,
                 np.where((ev & nat.EV_TIMEOUT) != 0, timeout, 0.0))
    return r.astype(np.float32)


class GameRecorder:
    def __init__(self, games, indices, folder=None, prefix='game', bot_data=None):
        self.games = games
        self.indices = [int(i) for i in indices]
        self.folder = folder
        self.prefix = prefix
        self.bot_data = bot_data if bot_data is not None else [None] * games.S
        self.finished = []          # completed core.Game objects, in completion order
        self.paths = []             # files written (when folder is given)
        self._ticks = {i: [] for i in self.indices}
        self._pending = None
        self._episode = {i: 0 for i in self.indices}

    def before_step(self, actions=None):
        """Call right before games.step(actions): records the pre-step state and the controls.
        actions -- what step() receives: [n, S] array / cuda tensor of control codes, or None for
        the device counter stream (the controls are then regenerated on the host, rng.actions)."""
        g = self.games
        states = g.get_states(self.indices)
        if actions is None:
            from . import rng
            ctl = rng.actions(g.seed, g.first_game + np.asarray(self.indices), g.step_index, g.S)
        else:
            a = actions[self.indices] if isinstance(actions, np.ndarray) else actions[self.indices].cpu().numpy()
            ctl = np.asarray(a, dtype=np.int64).reshape(len(self.indices), g.S)
        self._pending = (states, ctl)

    def after_step(self, reward, done):
        """Call right after games.step(...) with its (reward, done) results."""
        states, ctl = self._pending
        self._pending = None
        r = reward[self.indices].cpu().numpy() if hasattr(reward, 'cpu') else np.asarray(reward)[self.indices]
        d = done[self.indices].cpu().numpy() if hasattr(done, 'cpu') else np.asarray(done)[self.indices]
        self._append(states, ctl, r, d)

    def _append(self, states, ctl, r, d):
        """One tick of the followed games: pre-step states, controls [m, S], rewards [m, S], done flags [m]."""
        for j, i in enumerate(self.indices):
            if states[j] is None:       # the slot held a finished game: nothing happened
                continue
            rew = np.asarray(r[j], dtype=np.float32)
            self._ticks[i].append(core.Tick(state=states[j], control=ctl[j].copy(), reward=rew, bot_data=list(self.bot_data)))
            if d[j]:
                winner = None if np.max(rew) < 1 else int(np.argmax(rew))   # core.py:409
                game = core.Game(config=self.games.config, winner=winner, ticks=self._ticks[i])
                self.finished.append(game)
                if self.folder is not None:
                    path = os.path.join(self.folder, '%s_%d_%d.jsonl' % (self.prefix, i, self._episode[i]))
                    core.save_log(path, game)
                    self.paths.append(path)
                self._ticks[i] = []
                self._episode[i] += 1

    def step(self, actions=None, **kw):
        """before_step + games.step + after_step in one call; returns what games.step returns."""
        self.before_step(actions)
        out = self.games.step(actions, **kw)
        self.after_step(out[0], out[1])
        return out

    def rollout(self, n_ticks, ring, **rollout_kwargs):
        """games.rollout_device(n_ticks, record=ring, **rollout_kwargs), logged tick by tick as a loop of step() calls
        through before_step / after_step would have logged it.  `ring` is a RecordRing that follows exactly this recorder's
        games, in the same order (games.record_ring(ticks, follow=recorder.indices)); a call logs at most ring.ticks - 1
        ticks.  Following games costs the many-tick launches of scripted and counter-stream rollouts (astro_rollout_device_follow)."""
        if ring.follow != self.indices:
            raise ValueError('the ring follows games %r, this recorder %r' % (ring.follow, self.indices))
        g = self.games
        s0, n = g.step_index, int(n_ticks)
        g.rollout_device(n, record=ring, **rollout_kwargs)
        rows = ring._rows(s0, n)
        idx = ring._follow_index.long()
        ctl = ring.controls[rows][:, idx].cpu().numpy().astype(np.int64)        # [n, m, S]
        ev = ring.events[rows][:, idx].cpu().numpy()                            # [n, m]
        rew = event_rewards(ev, g.S, g.config.solo)
        done = ev & nat.EV_DONE_MASK
        for k in range(n):
            self._append(ring.follow_states(s0 + k), ctl[k], rew[k], done[k])
