"""Thin Python handle over the C-ABI engine (include/az_b200.h).  torch is used for device buffers and streams only."""
import ctypes as C
import re

import numpy as np
import torch

from . import _lib as L


def parse_game_name(name):
    """pyspiel.load_game names used by the reference (train.py:24): -> (game_id, rows, cols)."""
    name = name.strip()
    if name in ("connect_four", "connect_four()"):
        return L.GAME_CONNECT_FOUR, 6, 7
    m = re.fullmatch(r"breakthrough(?:\((.*)\))?", name)
    if not m:
        raise ValueError("unsupported game for the B200 engine: %r" % (name,))
    rows = cols = 8
    if m.group(1) and m.group(1).strip():
        for kv in m.group(1).split(","):
            k, v = [t.strip() for t in kv.split("=")]
            if k == "rows":
                rows = int(v)
            elif k == "columns":
                cols = int(v)
            else:
                raise ValueError("unsupported breakthrough parameter %r" % k)
    return L.GAME_BREAKTHROUGH, rows, cols


def game_shape(name):
    """(state_shape [3,H,W], num_distinct_actions) -- game.information_state_normalized_vector_shape()."""
    gid, rows, cols = parse_game_name(name)
    return [3, rows, cols], (7 if gid == L.GAME_CONNECT_FOUR else rows * cols * 12)


def record_dtype(max_children, stride):
    return np.dtype({
        "names": ["tree", "game_seq", "ply", "action", "n_legal", "kind", "root_n", "end", "bb", "root_q", "v_a0c",
                  "v_offpolicy", "counts", "actions"],
        "formats": ["<i4", "<i4", "<i4", "<i4", "<i4", "<i4", "<i4", "<i4", ("<u8", (2,)), "<f8", "<f8", "<f8",
                    ("<i4", (max_children,)), ("<i2", (max_children,))],
        "offsets": [0, 4, 8, 12, 16, 20, 24, 28, 32, 48, 56, 64, 72, 72 + 4 * max_children],
        "itemsize": stride,
    })


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class Engine:
    """n_trees independent search trees on one GPU.  See include/az_b200.h for the model."""

    def __init__(self, game_name, n_trees, n_playouts=100, c_puct=2.5, dirichlet_ratio=0.25, temperature=1.0,
                 num_probabilistic_actions=1000, noise_mode=L.NOISE_DIRICHLET, eval_mode=L.EVAL_EXTERNAL,
                 eval_shift=None, flags=L.F_KEEP_TREE, seed=0, device=0, node_capacity=0, max_sims_per_step=0,
                 start_plies_mod=0, record_capacity=0, max_games=0, leaves_per_tree=1, step_cycle_budget=0,
                 eval_cache_log2=0):
        self.lib = L.load()
        if not torch.cuda.is_available():
            raise L.EngineUnavailable("the B200 engine needs a CUDA device; there is no CPU fallback")
        gid, rows, cols = parse_game_name(game_name)
        self.game_name = game_name
        self.game_id, self.rows, self.cols = gid, rows, cols
        self.device = torch.device("cuda", device)
        cfg = L.AzConfig()
        cfg.game_id, cfg.rows, cfg.cols = gid, rows, cols
        cfg.n_trees, cfg.node_capacity, cfg.n_playouts = n_trees, node_capacity, n_playouts
        cfg.c_puct, cfg.dirichlet_ratio = c_puct, dirichlet_ratio
        cfg.dirichlet_alpha, cfg.noise_weight, cfg.temperature = 0.3, 0.25, temperature
        cfg.num_probabilistic_actions = num_probabilistic_actions
        cfg.noise_mode, cfg.eval_mode = noise_mode, eval_mode
        cfg.eval_shift = (2 if gid == L.GAME_CONNECT_FOUR else 4) if eval_shift is None else eval_shift
        cfg.max_sims_per_step, cfg.start_plies_mod = max_sims_per_step, start_plies_mod
        if flags & L.F_EVAL_CACHE:   # table size: 2^eval_cache_log2 entries, 0 = the engine's default
            flags |= int(eval_cache_log2) << L.EVAL_CACHE_LOG2_SHIFT
        cfg.record_capacity, cfg.device, cfg.flags, cfg.seed = record_capacity, device, flags, seed
        cfg.max_games = max_games
        cfg.leaves_per_tree = leaves_per_tree if (flags & L.F_VIRTUAL_LOSS) else 1
        cfg.step_cycle_budget = step_cycle_budget
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            L.check(self.lib.az_create(C.byref(cfg), C.byref(h)))
        self.h = h
        eff = L.AzConfig()
        L.check(self.lib.az_config_get(self.h, C.byref(eff)))
        self.cfg = eff
        self.eval_cache_log2 = (eff.flags >> L.EVAL_CACHE_LOG2_SHIFT) & 31   # F_EVAL_CACHE table in use (0 = off)
        self.n_trees = n_trees
        self.flags = flags
        self.rows_per_tree = int(eff.leaves_per_tree)        # evaluator rows per tree (1 unless AZ_F_VIRTUAL_LOSS)
        self.n_rows = n_trees * self.rows_per_tree
        self.max_children = self.lib.az_max_children(self.h)
        self.num_actions = self.lib.az_num_actions(self.h)
        self.record_stride = self.lib.az_record_stride(self.h)
        self.rec_dtype = record_dtype(self.max_children, self.record_stride)
        self.device_bytes = self.lib.az_device_bytes(self.h)
        self._rec_host = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.az_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def new_obs(self, obs_format):
        if obs_format == L.OBS_BF16_NHWC:
            return torch.zeros((self.n_rows, self.rows, self.cols, 4), dtype=torch.bfloat16, device=self.device)
        return torch.zeros((self.n_rows, 4, self.rows, self.cols), dtype=torch.float32, device=self.device)

    # ---- C-ABI calls
    def reset(self):
        L.check(self.lib.az_reset(self.h, self._stream()))

    def step(self, priors=None, values=None, noise=None, obs=None, obs_format=None):
        if obs is None:
            obs_format = L.OBS_NONE
        elif obs_format is None:
            obs_format = L.OBS_BF16_NHWC if obs.dtype == torch.bfloat16 else L.OBS_F32_NCHW
        if priors is not None:
            want = torch.float64 if (self.flags & L.F_PRIORS_F64) else torch.float32
            assert priors.dtype == want and values.dtype == want, "priors/values dtype must be %s" % want
            assert priors.is_contiguous() and values.is_contiguous()
            assert priors.numel() == self.n_rows * self.num_actions and values.numel() == self.n_rows
        if noise is not None:
            assert noise.dtype == torch.float64 and noise.numel() == self.n_trees * self.max_children
        L.check(self.lib.az_step(self.h, _ptr(priors), _ptr(values), _ptr(noise), _ptr(obs), obs_format,
                                 self._stream()))

    def compact(self, stream=None):
        """Re-root compaction of the trees that just moved (only needed with F_ASYNC_COMPACT)."""
        st = self._stream() if stream is None else C.c_void_p(stream.cuda_stream)
        L.check(self.lib.az_compact(self.h, st))

    def invalidate_eval_cache(self):
        """F_EVAL_CACHE: the evaluator's weights change after the rows already computed (az_eval_cache_invalidate)."""
        L.check(self.lib.az_eval_cache_invalidate(self.h, self._stream()))

    def set_resign(self, threshold, disabled_permille):
        """F_RESIGN: resign threshold and per-mille share of no-resign calibration games (az_set_resign), stream-ordered:
        a captured graph of step() sees the new values on its next replay."""
        L.check(self.lib.az_set_resign(self.h, float(threshold), int(disabled_permille), self._stream()))

    def set_playout_cap(self, fast_playouts, full_permille):
        """F_PLAYOUT_CAP: simulations of a fast search and per-mille share of full searches (az_set_playout_cap),
        stream-ordered: a captured graph of step() sees the new values on its next replay."""
        L.check(self.lib.az_set_playout_cap(self.h, int(fast_playouts), int(full_permille), self._stream()))

    def set_forced_playouts(self, k):
        """F_FORCED_PLAYOUTS: k of the forced-playout floor sqrt(k * P * N) (az_set_forced_playouts; 0 forces nothing),
        stream-ordered: a captured graph of step() sees the new value on its next replay."""
        L.check(self.lib.az_set_forced_playouts(self.h, float(k), self._stream()))

    def set_positions(self, histories):
        """histories: list (len n_trees) of action lists, or None entries to leave a tree untouched."""
        n = self.n_trees
        max_len = max([len(h) for h in histories if h is not None] + [1])
        hist = np.zeros((n, max_len), dtype=np.int32)
        lens = np.full((n,), -1, dtype=np.int32)
        for i, h in enumerate(histories):
            if h is not None:
                lens[i] = len(h)
                hist[i, :len(h)] = h
        L.check(self.lib.az_set_positions(self.h, hist.ctypes.data, lens.ctypes.data, max_len, self._stream()))

    def command(self, update_root=None, reset_tree=None, begin=None):
        def arr(x, fill):
            if x is None:
                return None
            a = np.asarray(x, dtype=np.int32)
            assert a.shape == (self.n_trees,)
            return np.ascontiguousarray(a)
        u, r, b = arr(update_root, -1), arr(reset_tree, 0), arr(begin, 0)
        L.check(self.lib.az_command(self.h, None if u is None else u.ctypes.data,
                                    None if r is None else r.ctypes.data,
                                    None if b is None else b.ctypes.data, self._stream()))

    def status(self):
        n = self.n_trees
        out = torch.empty((4, n), dtype=torch.int32, device=self.device)
        L.check(self.lib.az_status(self.h, _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), self._stream()))
        o = out.cpu().numpy()
        return {"phase": o[0], "sims": o[1], "ply": o[2], "req_legal": o[3]}

    def phases(self):
        out = torch.empty((self.n_trees,), dtype=torch.int32, device=self.device)
        L.check(self.lib.az_status(self.h, _ptr(out), None, None, None, self._stream()))
        return out

    def request_info(self, max_depth=64):
        n = self.n_trees
        bb = torch.empty((n, 2), dtype=torch.int64, device=self.device)
        ply = torch.empty((n,), dtype=torch.int32, device=self.device)
        path = torch.full((n, max_depth), -1, dtype=torch.int32, device=self.device)
        depth = torch.empty((n,), dtype=torch.int32, device=self.device)
        L.check(self.lib.az_request_info(self.h, _ptr(bb), _ptr(ply), _ptr(path), _ptr(depth), max_depth,
                                         self._stream()))
        return {"bb": bb.cpu().numpy().view(np.uint64), "ply": ply.cpu().numpy(), "path": path.cpu().numpy(),
                "depth": depth.cpu().numpy()}

    def root_stats(self, offpolicy=True):
        n, m = self.n_trees, self.max_children
        dev = self.device
        root_n = torch.empty((n,), dtype=torch.int32, device=dev)
        root_q = torch.empty((n,), dtype=torch.float64, device=dev)
        nch = torch.empty((n,), dtype=torch.int32, device=dev)
        act = torch.empty((n, m), dtype=torch.int32, device=dev)
        cn = torch.empty((n, m), dtype=torch.int32, device=dev)
        cq = torch.empty((n, m), dtype=torch.float64, device=dev)
        cp = torch.empty((n, m), dtype=torch.float64, device=dev)
        a0c = torch.empty((n,), dtype=torch.float64, device=dev)
        off = torch.empty((n,), dtype=torch.float64, device=dev) if offpolicy else None
        L.check(self.lib.az_root_stats(self.h, _ptr(root_n), _ptr(root_q), _ptr(nch), _ptr(act), _ptr(cn), _ptr(cq),
                                       _ptr(cp), _ptr(a0c), _ptr(off), self._stream()))
        out = {"root_n": root_n, "root_q": root_q, "n_children": nch, "child_action": act, "child_n": cn,
               "child_q": cq, "child_p": cp, "v_a0c": a0c}
        if offpolicy:
            out["v_offpolicy"] = off
        return {k: v.cpu().numpy() for k, v in out.items()}

    def positions(self):
        n = self.n_trees
        bb = torch.empty((n, 2), dtype=torch.int64, device=self.device)
        ply = torch.empty((n,), dtype=torch.int32, device=self.device)
        term = torch.empty((n,), dtype=torch.int32, device=self.device)
        ret0 = torch.empty((n,), dtype=torch.float64, device=self.device)
        L.check(self.lib.az_positions(self.h, _ptr(bb), _ptr(ply), _ptr(term), _ptr(ret0), self._stream()))
        return {"bb": bb.cpu().numpy().view(np.uint64), "ply": ply.cpu().numpy(), "terminal": term.cpu().numpy(),
                "return0": ret0.cpu().numpy()}

    def drain_records(self):
        cap = int(self.cfg.record_capacity)
        if self._rec_host is None:
            self._rec_host = np.empty((cap,), dtype=self.rec_dtype)
        n = C.c_int64(0)
        L.check(self.lib.az_drain_records(self.h, self._rec_host.ctypes.data, cap, C.byref(n), self._stream()))
        return self._rec_host[:n.value].copy()

    def counters(self):
        out = np.zeros((len(L.CTR_NAMES),), dtype=np.uint64)
        L.check(self.lib.az_counters(self.h, out.ctypes.data, self._stream()))
        return {k: int(v) for k, v in zip(L.CTR_NAMES, out)}


def game_replay(game_name, histories, obs_format=L.OBS_F32_NCHW, device=0):
    """Stateless batched game ops (parity tests): replay histories on the device."""
    lib = L.load()
    gid, rows, cols = parse_game_name(game_name)
    n = len(histories)
    dev = torch.device("cuda", device)
    max_len = max([len(h) for h in histories] + [1])
    hist = np.zeros((n, max_len), dtype=np.int32)
    lens = np.zeros((n,), dtype=np.int32)
    for i, h in enumerate(histories):
        lens[i] = len(h)
        hist[i, :len(h)] = h
    return game_replay_dev(game_name, torch.from_numpy(hist).to(dev), torch.from_numpy(lens).to(dev), obs_format)


def game_replay_dev(game_name, hist, lens, obs_format=L.OBS_F32_NCHW):
    lib = L.load()
    gid, rows, cols = parse_game_name(game_name)
    n, max_len = hist.shape
    dev = hist.device
    maxc = 7 if gid == L.GAME_CONNECT_FOUR else 48
    bb = torch.empty((n, 2), dtype=torch.int64, device=dev)
    status = torch.empty((n,), dtype=torch.int32, device=dev)
    ret0 = torch.empty((n,), dtype=torch.float64, device=dev)
    nleg = torch.empty((n,), dtype=torch.int32, device=dev)
    legal = torch.empty((n, maxc), dtype=torch.int32, device=dev)
    if obs_format == L.OBS_BF16_NHWC:
        obs = torch.zeros((n, rows, cols, 4), dtype=torch.bfloat16, device=dev)
    else:
        obs = torch.zeros((n, 4, rows, cols), dtype=torch.float32, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    L.check(lib.az_game_replay(gid, rows, cols, n, _ptr(hist), _ptr(lens), max_len, _ptr(bb), _ptr(status),
                               _ptr(ret0), _ptr(nleg), _ptr(legal), _ptr(obs), obs_format, st))
    return {"bb": bb, "status": status, "return0": ret0, "n_legal": nleg, "legal": legal, "obs": obs}


def game_random_playouts(game_name, n, seed, max_plies, device=0):
    lib = L.load()
    gid, rows, cols = parse_game_name(game_name)
    dev = torch.device("cuda", device)
    hist = torch.zeros((n, max_plies), dtype=torch.int32, device=dev)
    lens = torch.zeros((n,), dtype=torch.int32, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    L.check(lib.az_game_random_playouts(gid, rows, cols, n, seed, max_plies, _ptr(hist), _ptr(lens), st))
    return hist, lens
