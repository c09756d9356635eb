"""Observation extraction of `astro.rl.ValueNetwork` (reference: astro/rl.py:36-112) over the
CUDA observe kernel.

    ValueNetwork.get_features(state)         -> float32 [P+B, 1+5S+4]
    ValueNetwork.to_batch(list of features)  -> float32 [n, max rows, D], -1 padded
    ValueNetwork.get_features_batch(states)  -> the two combined

Rows are planets then bullets (array order); column 0 is the type flag (0 planet / 1 bullet,
-1 padding: consumers mask on `features[..., 0] < 0`, rl.py:126-128); columns 1..5S hold every
ship's (x, y, dx, dy, norm_angle(b)/pi), ship 0 first; the last 4 the object's (x, y, dx, dy).
For rollouts use `BatchedGames.observe()` directly: it writes the padded batch for every game
and both perspectives in one launch and never leaves the GPU.
"""

import numpy as np
import torch

from . import core
from .batched import BatchedGames

_CACHE = {}
_BOTH = {}
_SWAP = [0, 6, 7, 8, 9, 10, 1, 2, 3, 4, 5, 11, 12, 13, 14]     # ship 1's feature columns in ship 0's view (core.roll_ships)

def _games(solo, n, cap, device=None):
    n_pad = max(32, -(-n // 32) * 32)
    key = (bool(solo), n_pad, cap, device)
    g = _CACHE.get(key)
    if g is None:
        cfg = core.SOLO_CONFIG if solo else core.DEFAULT_CONFIG
        g = _CACHE[key] = BatchedGames(cfg, n_pad, bullet_cap=cap, precision=64, **({} if device is None else dict(device=device)))
    return g

def _both_views(n, device):
    """forward_views' (index, view) of forward_both on n items: every item as ship 0, then as ship 1.  One pair per device,
    for the largest n asked so far; smaller n take its first 2n entries."""
    iv = _BOTH.get(device)
    if iv is None or iv[0].shape[0] < 2 * n:
        iv = _BOTH[device] = (torch.arange(n, device=device).repeat_interleave(2),
                              torch.arange(2 * n, device=device).remainder(2).to(torch.uint8))
    return iv[0][:2 * n], iv[1][:2 * n]

class ValueNetwork(torch.nn.Module):
    """The reference's Q-network (rl.py:32-165) with the feature extraction on the GPU.

    Same constructor, layer names (`f0`, `f`, `v`, `v0` — state dicts interchange), feature
    methods and `evaluate*` entry points.  The network body is the consumer of the observation
    batches, plain PyTorch as in the reference: 15 (10 solo) -> 32, two softsign/linear blocks per
    object, max-pool over the objects whose type flag is >= 0, two linear/softsign blocks,
    linear -> tanh.  `forward` takes [..., N, D] feature batches on any device — for rollouts feed
    it `BatchedGames.observe()` directly.
    """

    def __init__(self, solo, nout):
        super().__init__()
        width, depth = 32, 2
        self.activation = torch.nn.functional.softsign
        self.f0 = torch.nn.Linear(10 if solo else 15, width)
        self.f = torch.nn.ModuleList([torch.nn.Linear(width, width) for _ in range(depth)])
        self.pool = self.masked_max
        self.v = torch.nn.ModuleList([torch.nn.Linear(width, width) for _ in range(depth)])
        self.v0 = torch.nn.Linear(width, nout)

    @staticmethod
    def masked_max(x, features):
        """Max over the object axis (-2), padding rows (type flag < 0) excluded (rl.py:115-128)."""
        pad = (features[..., 0] < 0).unsqueeze(-1).to(x.dtype)
        return torch.max(x - 1e9 * pad, dim=-2)[0]

    @staticmethod
    def masked_sum(x, features):
        live = (features[..., 0] >= 0).unsqueeze(-1).to(x.dtype)
        return torch.sum(x * live, dim=-2)

    def _fused(self, x):
        """The batch that holds this module's weights for the fused inference kernel (astro_value_forward), re-uploaded
        whenever a parameter has changed (tensor version counters); None when the call must go through autograd or
        the tensor is not a float32 cuda feature batch of this network's width."""
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() >= 2 and x.shape[-2] >= 1 and x.numel() > 0):
            return None
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return None
        if self.pool != self.masked_max or self.activation is not torch.nn.functional.softsign or x.shape[-1] != self.f0.in_features:
            return None
        params = list(self.parameters())
        if any(p.device != x.device for p in params) or self.f0.in_features not in (10, 15) or self.v0.out_features > 8:
            return None
        g = _games(self.f0.in_features == 10, 32, 32, x.device.index)
        stamp = (id(self), tuple(p._version for p in params), tuple(p.data_ptr() for p in params))
        if getattr(g, '_net_stamp', None) != stamp:
            g.set_policy(self)
            g._net_stamp = stamp
        return g

    def forward(self, x):
        g = self._fused(x)
        if g is not None:
            return g.value_forward(x)
        return self.forward_torch(x)

    def forward_torch(self, x):
        """The reference's forward, layer by layer in PyTorch (training, CPU tensors, float64 features)."""
        h = self.f0(x)
        for layer in self.f:
            h = layer(self.activation(h))
        h = self.pool(h, features=x)
        for layer in self.v:
            h = self.activation(layer(h))
        return torch.tanh(self.v0(h))

    def forward_both(self, x):
        """Both ships' values from ONE perspective-0 feature batch x [..., N, 15] -> [..., 2, nout].

        Ship 1's features are ship 0's with the ship column groups exchanged (core.roll_ships,
        core.py:306-327 + rl.py:62-70); exchanging the matching COLUMNS of the first layer's weight
        gives the same pre-activations without a second observation tensor
        (`BatchedGames.observe(shared=True)`).  Under the conditions of `forward`'s kernel this is
        forward_views of every item as ship 0 and as ship 1 (value_forward_kernel reads ship 1's
        columns in place): bit for bit forward() of the two-view tensor observe() gives."""
        if x.shape[-1] != 15:
            raise ValueError('forward_both needs duel features [..., N, 15]')
        g = self._fused(x)
        if g is not None:
            flat = x.reshape(-1, x.shape[-2], 15)
            index, view = _both_views(flat.shape[0], x.device)
            return g.value_forward_views(flat, index, view).view(tuple(x.shape[:-2]) + (2, -1))
        return self.forward_both_torch(x)

    def forward_both_torch(self, x):
        """forward_both layer by layer in PyTorch (training, CPU tensors, float64 features)."""
        swap = torch.tensor(_SWAP, device=x.device)
        w = torch.cat((self.f0.weight, self.f0.weight[:, swap]), dim=0)           # [64, 15]
        b = torch.cat((self.f0.bias, self.f0.bias), dim=0)
        h = torch.nn.functional.linear(x, w, b)                                    # [..., N, 64]
        h = h.unflatten(-1, (2, -1)).movedim(-2, -3)                               # [..., 2, N, 32]
        for layer in self.f:
            h = layer(self.activation(h))
        h = self.pool(h, features=x.unsqueeze(-3))
        for layer in self.v:
            h = self.activation(layer(h))
        return torch.tanh(self.v0(h))

    def forward_views(self, x, index, view=None):
        """The network on gathered views of ONE perspective-0 feature batch x [M, N, D] -> [E, nout]: output e is forward()
        of item index[e] as ship view[e] sees it (ship 1: the ship column groups exchanged, as forward_both), index -1 an
        item whose every entry is -1 (a finished game: the new state of a terminal pair).  index: int64 [E] on x's device;
        view: uint8 [E] (0 = ship 0, otherwise ship 1) or None (ship 0; solo features, D = 10, take none).

        Under the conditions of `forward`'s kernel (cuda float32, no autograd) this is one value_forward_kernel launch that
        reads each row where the view has it, so no [E, N, D] tensor is made; otherwise the gather, the column exchange and
        forward_torch in PyTorch, with the same values.  Raises ValueError before any launch on a dtype or shape that does
        not fit, or an index outside -1 .. M - 1 (one reduction over index)."""
        D = self.f0.in_features
        if not (x.dim() == 3 and x.shape[-1] == D and x.shape[-2] >= 1 and x.is_floating_point()):
            raise ValueError('forward_views needs a feature batch [M, N, %d] (N >= 1)' % D)
        if not (isinstance(index, torch.Tensor) and index.dtype == torch.int64 and index.dim() == 1 and index.device == x.device):
            raise ValueError('index must be an int64 tensor [E] on the features\' device')
        if view is not None and not (D == 15 and isinstance(view, torch.Tensor) and view.dtype == torch.uint8
                                     and view.shape == index.shape and view.device == x.device):
            raise ValueError('view must be a uint8 tensor shaped like index on the features\' device (duel features only)')
        if index.numel():
            lo, hi = (int(v) for v in torch.aminmax(index))
            if lo < -1 or hi >= x.shape[0]:
                raise ValueError('index values %d .. %d outside -1 .. %d' % (lo, hi, x.shape[0] - 1))
        g = self._fused(x)
        if g is not None:
            return g.value_forward_views(x, index, view)
        return self.forward_torch(self._gather_views(x, index, view))

    @staticmethod
    def _gather_views(x, index, view):
        """The [E, N, D] tensor forward_views evaluates: x[index], all -1 where index is -1, the ship column groups
        exchanged where view is set."""
        items = x[index.clamp(min=0)] if x.shape[0] else x.new_full((index.shape[0],) + tuple(x.shape[1:]), -1.0)
        items = torch.where((index < 0)[:, None, None], torch.full_like(items, -1.0), items)
        if view is not None:
            items = torch.where((view != 0)[:, None, None], items[..., torch.tensor(_SWAP, device=x.device)], items)
        return items

    def evaluate(self, state):
        dev = next(self.parameters()).device
        return self(torch.from_numpy(self.get_features(state)).to(dev))

    def evaluate_batch(self, states):
        dev = next(self.parameters()).device
        return self(torch.from_numpy(self.get_features_batch(states)).to(dev))

    @staticmethod
    def get_features_shape(state):
        return (state.planets.x.shape[0] + state.bullets.x.shape[0], 1 + 4 + 5 * state.ships.x.shape[0])

    @classmethod
    def get_features_batch(cls, states, perspective=0):
        if not states:
            raise ValueError('no states')
        nships = {np.shape(s.ships.x)[0] for s in states}
        if len(nships) != 1:
            raise ValueError('Feature dimensions do not match - cannot mix solo & nonsolo games in a single batch')
        solo = nships.pop() == 1
        kmax = max(np.shape(s.bullets.x)[0] for s in states)
        cap = max(32, -(-kmax // 32) * 32)
        g = _games(solo, len(states), cap)
        g.meta.fill_(1 << 13)
        g.set_states(list(states), ticks=np.zeros(len(states), dtype=np.int64))
        rows = max(np.shape(s.planets.x)[0] + np.shape(s.bullets.x)[0] for s in states)
        obs = g.observe()[:len(states), perspective, :rows]
        return obs.cpu().numpy()

    @classmethod
    def get_features(cls, state):
        n_rows, _ = cls.get_features_shape(state)
        return cls.get_features_batch([state])[0, :n_rows]

    @staticmethod
    def to_batch(features):
        """Pad a list of [N_i, D] feature arrays to [n, max N_i, D] with -1 (rl.py:75-99)."""
        if any(f.shape[1] != features[0].shape[1] for f in features):
            raise ValueError('Feature dimensions do not match - cannot mix solo & nonsolo games in a single batch')
        out = np.full((len(features), max(f.shape[0] for f in features), features[0].shape[1]), -1, dtype=np.float32)
        for i, f in enumerate(features):
            out[i, :f.shape[0]] = f
        return out
