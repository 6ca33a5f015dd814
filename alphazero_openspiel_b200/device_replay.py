"""The replay buffer on the device (SURVEY 8(f) ranks 1 and 3): positions as canonical bitboards, policy / value targets and a
64-bit hash of the reference's info-state key as device tensors; `Trainer.remove_duplicates` (train.py:156-201) as a
sort + segment mean, and the minibatch of `Trainer.net_step` (train.py:106-112) built on the device by a gather kernel
(az_observations: bitboards -> state_to_board planes) instead of `np.array([python list of numpy boards])` + host-to-device
copies every optimisation step.

Semantics are those of replay.ExampleBatch (whose arrays it uploads once per generation): examples with the same key are
merged into the FIRST occurrence, groups keep first-occurrence order (the reference's dict order, so the same
`np.random.randint` sample ids pick the same examples as the list path), targets are float64 means.  The sums are device
reductions, so they can differ from the sequential host sums in the last bit (tests bound it at 1e-12); everything the
network sees is fp32, as in the reference (`.float()`, train.py:112-120).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from .engine import parse_game_name, reflect_actions


def key_hash(batch):
    """64-bit hash of every example's de-duplication key (action history incl. its length, plus the start position of a
    random-start game): a polynomial hash over the key columns, wrap-around uint64 arithmetic, vectorised over examples."""
    n = len(batch)
    h = np.full(n, 0x9E3779B97F4A7C15, dtype=np.uint64)
    mul = np.uint64(0x100000001B3)
    cols = [batch.hist_len.astype(np.int64)] + [batch.hist[:, j].astype(np.int64) for j in range(batch.hist.shape[1])]
    with np.errstate(over="ignore"):
        for c in cols:
            h = (h ^ (c + 2).astype(np.uint64)) * mul
            h ^= h >> np.uint64(29)
        for j in range(3):
            h = (h ^ batch.start[:, j]) * mul
            h ^= h >> np.uint64(32)
    return h.view(np.int64)


class DeviceReplay:
    def __init__(self, game_name, device):
        self.game_name = game_name
        self.game_id, self.rows, self.cols = parse_game_name(game_name)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.EngineUnavailable("DeviceReplay needs a CUDA device; there is no CPU fallback")
        self.lib = L.load()
        self.game_ptr = np.zeros(1, np.int64)        # host: examples of game g are rows game_ptr[g] : game_ptr[g+1]
        self.bb = self.ply = self.key = self.policy = self.value = None
        self._reflect_perm = None

    def __len__(self):
        return 0 if self.bb is None else int(self.bb.shape[0])

    @property
    def n_games(self):
        return len(self.game_ptr) - 1

    def append(self, batch):
        """Upload the examples of a replay.ExampleBatch (one generation) behind the ones already held."""
        if len(batch) == 0:
            return
        dev = self.device
        new = {
            "bb": torch.from_numpy(np.ascontiguousarray(batch.bb).view(np.int64)).to(dev),
            "ply": torch.from_numpy(np.ascontiguousarray(batch.ply.astype(np.int32))).to(dev),
            "key": torch.from_numpy(key_hash(batch)).to(dev),
            "policy": torch.from_numpy(np.ascontiguousarray(batch.policy)).to(dev),
            "value": torch.from_numpy(np.ascontiguousarray(batch.value)).to(dev),
        }
        if self.bb is None:
            self.bb, self.ply, self.key, self.policy, self.value = (new[k] for k in ("bb", "ply", "key", "policy", "value"))
        else:
            self.bb = torch.cat([self.bb, new["bb"]])
            self.ply = torch.cat([self.ply, new["ply"]])
            self.key = torch.cat([self.key, new["key"]])
            self.policy = torch.cat([self.policy, new["policy"]])
            self.value = torch.cat([self.value, new["value"]])
        self.game_ptr = np.concatenate([self.game_ptr, batch.game_ptr[1:] + self.game_ptr[-1]])

    def keep_last_games(self, n_games):
        """The reference trims its buffer list from the front (train.py:232-234)."""
        if n_games >= self.n_games:
            return
        g0 = self.n_games - n_games
        lo = int(self.game_ptr[g0])
        self.game_ptr = self.game_ptr[g0:] - lo
        self.bb, self.ply, self.key = self.bb[lo:].contiguous(), self.ply[lo:].contiguous(), self.key[lo:].contiguous()
        self.policy, self.value = self.policy[lo:].contiguous(), self.value[lo:].contiguous()

    @torch.no_grad()
    def remove_duplicates(self):
        """train.py:156-201 on the device: -> (first, policy, value): index of the first example of every key in
        first-occurrence order and that key's averaged targets (float64); the averages are also written back into rows
        `first`, like the reference's in-place accumulator."""
        n = len(self)
        if n == 0:
            z = torch.zeros(0, dtype=torch.int64, device=self.device)
            return z, torch.zeros((0, 0), dtype=torch.float64, device=self.device), torch.zeros(0, dtype=torch.float64,
                                                                                                 device=self.device)
        uniq, inverse = torch.unique(self.key, return_inverse=True)             # sort by key
        g = uniq.numel()
        pos = torch.arange(n, device=self.device)
        first = torch.full((g,), n, dtype=torch.int64, device=self.device).scatter_reduce_(0, inverse, pos, reduce="amin")
        order = torch.argsort(first)                                           # groups in first-occurrence order
        rank = torch.empty(g, dtype=torch.int64, device=self.device)
        rank[order] = torch.arange(g, device=self.device)
        grp = rank[inverse]
        first = first[order]
        count = torch.bincount(grp, minlength=g).to(torch.float64)
        pol = torch.zeros((g, self.policy.shape[1]), dtype=torch.float64, device=self.device).index_add_(0, grp, self.policy)
        val = torch.zeros(g, dtype=torch.float64, device=self.device).index_add_(0, grp, self.value)
        pol /= count[:, None]
        val /= count
        self.policy[first] = pol
        self.value[first] = val
        return first, pol, val

    @property
    def reflect_perm(self):
        """The action reflection (engine.reflect_actions) as a device index tensor: a reflected policy row is p[:, perm]."""
        if self._reflect_perm is None:
            self._reflect_perm = torch.from_numpy(reflect_actions(self.game_name)).to(self.device)
        return self._reflect_perm

    @torch.no_grad()
    def boards(self, ids, reflect=None):
        """state_to_board planes (network.py:9-18) of examples `ids` (int64 device tensor): float32 [n, 4, rows, cols],
        gathered and encoded by the az_observations kernel.  reflect (uint8 / bool device tensor [n], optional): rows where
        it is set hold the planes of the left-right reflected position (columns flipped)."""
        ids = ids.to(self.device, torch.int64).contiguous()
        n = int(ids.numel())
        if reflect is not None:
            reflect = reflect.to(self.device, torch.uint8).contiguous()
            assert reflect.numel() == n
        out = torch.empty((n, 4, self.rows, self.cols), dtype=torch.float32, device=self.device)
        st = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        L.check(self.lib.az_observations_reflected(self.game_id, self.rows, self.cols, n, C.c_void_p(self.bb.data_ptr()),
                                                   C.c_void_p(self.ply.data_ptr()), C.c_void_p(ids.data_ptr()),
                                                   None if reflect is None else C.c_void_p(reflect.data_ptr()),
                                                   C.c_void_p(out.data_ptr()), L.OBS_F32_NCHW, st))
        return out
