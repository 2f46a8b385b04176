"""Device-resident PUCT search / self-play pools over the C ABI.

Mirrors the C++ reference's search objects (cpp/self_play_client.cpp:369-493 ``MCTS``:
ctor / ``step`` / ``play``; :508-582 ``generate_game``) for G concurrent games at once, and the arena
(``Arena``, ``random_openings``) that plays two networks against each other with the same trees.
"""
import ctypes as C

import numpy as np

from . import _native
from ._native import AZ_FEATURES, AZ_LOGITS, AZ_MAX_MOVES, AzError, Position, check, lib
from .rules import pack_move, unpack_move

EVAL_FP32 = 0
EVAL_BF16 = 1
EVAL_F16 = 3
EVAL_EXTERNAL = 2


class PoolConfig(C.Structure):
    _fields_ = [("games", C.c_int32), ("visits", C.c_int32), ("max_plies", C.c_int32), ("noise", C.c_int32),
                ("auto_play", C.c_int32), ("eval_mode", C.c_int32), ("node_capacity", C.c_int32),
                ("steps_per_tick", C.c_int32), ("seed", C.c_uint64), ("start_fen", C.c_char * 64),
                ("speculate", C.c_int32), ("one_random_move", C.c_int32), ("reserved", C.c_int32 * 2)]


class PoolStats(C.Structure):
    _fields_ = [("ticks", C.c_uint64), ("steps", C.c_uint64), ("evals", C.c_uint64), ("terminal_steps", C.c_uint64),
                ("positions", C.c_uint64), ("games_finished", C.c_uint64), ("games_skipped", C.c_uint64),
                ("max_depth", C.c_uint64), ("kernel_launches", C.c_uint64), ("record_bytes", C.c_uint64),
                ("net_seconds", C.c_double),
                ("tree_seconds", C.c_double), ("levels", C.c_uint64), ("tick_seconds", C.c_double),
                ("timed_ticks", C.c_uint64), ("timed_evals", C.c_uint64)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


_vp = C.c_void_p
_native.register("az_pool_create", C.c_int, [_vp, C.POINTER(PoolConfig), C.POINTER(_vp)])
_native.register("az_pool_destroy", None, [_vp])
_native.register("az_pool_stats_get", C.c_int, [_vp, C.POINTER(PoolStats)])
_native.register("az_pool_set_root", C.c_int, [_vp, C.c_int, C.POINTER(Position)])
_native.register("az_pool_set_roots", C.c_int, [_vp, _vp])
_native.register("az_pool_set_visits", C.c_int, [_vp, C.c_int])
_native.register("az_pool_run", C.c_int, [_vp, C.c_int, C.POINTER(C.c_int32)])
_native.register("az_pool_collect", C.c_int, [_vp, _vp, C.POINTER(C.c_int32)])
_native.register("az_pool_provide", C.c_int, [_vp, _vp, _vp])
_native.register("az_pool_provide_n", C.c_int, [_vp, _vp, _vp, C.c_int32])
_native.register("az_pool_root", C.c_int, [_vp, C.c_int, C.POINTER(Position), C.POINTER(C.c_int32), _vp, _vp, _vp, _vp,
                                           C.POINTER(C.c_int32), C.POINTER(C.c_double)])
_native.register("az_pool_play", C.c_int, [_vp, C.c_int, C.c_uint16])
_native.register("az_pool_pv", C.c_int, [_vp, C.c_int, _vp, _vp, C.c_int, C.POINTER(C.c_int32)])
_native.register("az_selfplay_run", C.c_int, [_vp, C.c_char_p, C.c_int64, C.c_int64, C.c_double, C.POINTER(PoolStats)])
_native.register("az_selfplay_ticks", C.c_int, [_vp, C.c_char_p, C.c_int64, C.POINTER(PoolStats)])


class Pool:
    """G device-resident trees.  ``auto_play=False``: search mode (the caller plays moves);
    ``auto_play=True``: self-play generation (sample ~ visits, record, re-root, restart)."""

    def __init__(self, ctx, games, visits, eval_mode=EVAL_BF16, noise=False, auto_play=False, max_plies=400, seed=0,
                 start_fen="", node_capacity=0, steps_per_tick=0, speculate=0, one_random_move=False):
        self.ctx = ctx
        cfg = PoolConfig()
        cfg.games, cfg.visits, cfg.max_plies = int(games), int(visits), int(max_plies)
        cfg.noise, cfg.auto_play, cfg.eval_mode = int(bool(noise)), int(bool(auto_play)), int(eval_mode)
        cfg.node_capacity, cfg.steps_per_tick, cfg.seed = int(node_capacity), int(steps_per_tick), int(seed) & (2**64 - 1)
        cfg.start_fen = start_fen.encode()
        cfg.speculate = int(speculate)
        cfg.one_random_move = int(bool(one_random_move))
        self.cfg = cfg
        self.games = int(games)
        self._h = _vp()
        check(lib().az_pool_create(ctx.handle, C.byref(cfg), C.byref(self._h)))
        ctx.adopt(self)
        self._features = np.zeros((self.games, 7, 7, 4), dtype=np.float32)

    # ---- lifecycle ----
    def close(self):
        if self._h:
            lib().az_pool_destroy(self._h)
            self._h = _vp()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- search mode ----
    def set_root(self, game, position):
        check(lib().az_pool_set_root(self._h, int(game), C.byref(position)))

    def set_roots(self, positions):
        """All trees at once: ``positions`` is a structured array (rules.POSITION_DTYPE) or a list of Position."""
        from .rules import positions_array
        arr = positions_array(positions)
        if len(arr) != self.games:
            raise AzError(-1, "set_roots: %d positions for %d games" % (len(arr), self.games))
        check(lib().az_pool_set_roots(self._h, C.c_void_p(arr.ctypes.data)))

    def set_visits(self, visits):
        check(lib().az_pool_set_visits(self._h, int(visits)))

    def run(self, max_ticks=1 << 30):
        """Internal net: tick until every tree reached its visit target; returns True when idle."""
        idle = C.c_int32()
        check(lib().az_pool_run(self._h, int(max_ticks), C.byref(idle)))
        return bool(idle.value)

    def collect(self):
        """External evaluator: advance until blocked; returns float32 features [n,7,7,4] (n may be 0)."""
        n = C.c_int32()
        check(lib().az_pool_collect(self._h, C.c_void_p(self._features.ctypes.data), C.byref(n)))
        return self._features[:n.value]

    def provide(self, logits, values):
        logits = np.ascontiguousarray(logits, dtype=np.float32).reshape(-1, AZ_LOGITS)
        values = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
        if len(values) != len(logits):
            raise AzError(-1, "provide: %d logit rows but %d values" % (len(logits), len(values)))
        # the library copies one row per outstanding request: it is told how many rows these arrays really hold and
        # refuses a mismatch instead of reading past their end
        check(lib().az_pool_provide_n(self._h, C.c_void_p(logits.ctypes.data), C.c_void_p(values.ctypes.data), len(logits)))

    def run_external(self, evaluator):
        """Drive the pool with ``evaluator(features[n,7,7,4]) -> (logits[n,833], values[n])`` until idle."""
        while True:
            feats = self.collect()
            if len(feats) == 0:
                return
            logits, values = evaluator(feats)
            self.provide(logits, values)

    def root(self, game=0):
        """Root statistics in reference movegen order."""
        pos = Position()
        n = C.c_int32()
        rv = C.c_int32()
        val = C.c_double()
        moves = np.zeros(AZ_MAX_MOVES, dtype=np.uint16)
        visits = np.zeros(AZ_MAX_MOVES, dtype=np.int32)
        total = np.zeros(AZ_MAX_MOVES, dtype=np.float64)
        prior = np.zeros(AZ_MAX_MOVES, dtype=np.float64)
        check(lib().az_pool_root(self._h, int(game), C.byref(pos), C.byref(n), C.c_void_p(moves.ctypes.data),
                                 C.c_void_p(visits.ctypes.data), C.c_void_p(total.ctypes.data),
                                 C.c_void_p(prior.ctypes.data), C.byref(rv), C.byref(val)))
        k = n.value
        return {"position": pos, "moves": [unpack_move(m) for m in moves[:k]], "visits": visits[:k].tolist(),
                "total_score": total[:k].copy(), "prior": prior[:k].copy(), "root_visits": rv.value, "value": val.value}

    def principal_variation(self, game=0, max_len=64):
        """Most-visited line below the root: [(move, edge_visits), ...] (engine.py:331-336, best=True)."""
        moves = np.zeros(max_len, dtype=np.uint16)
        visits = np.zeros(max_len, dtype=np.int32)
        n = C.c_int32()
        check(lib().az_pool_pv(self._h, int(game), C.c_void_p(moves.ctypes.data), C.c_void_p(visits.ctypes.data), int(max_len),
                               C.byref(n)))
        return [(unpack_move(m), int(v)) for m, v in zip(moves[:n.value], visits[:n.value])]

    def play(self, game, move):
        """MCTS::play (self_play_client.cpp:475-492)."""
        check(lib().az_pool_play(self._h, int(game), pack_move(move)))

    # ---- self-play ----
    def selfplay(self, output_path, target_games=0, target_positions=0, max_seconds=0.0):
        stats = PoolStats()
        path = output_path.encode() if output_path else None
        check(lib().az_selfplay_run(self._h, path, int(target_games), int(target_positions), float(max_seconds),
                                    C.byref(stats)))
        return stats.as_dict()

    def selfplay_ticks(self, ticks, output_path=None):
        """Exactly ``ticks`` tree+net iterations; records go to ``output_path`` or stay on the device."""
        stats = PoolStats()
        path = output_path.encode() if output_path else None
        check(lib().az_selfplay_ticks(self._h, path, int(ticks), C.byref(stats)))
        return stats.as_dict()

    def stats(self):
        stats = PoolStats()
        check(lib().az_pool_stats_get(self._h, C.byref(stats)))
        return stats.as_dict()


class ArenaConfig(C.Structure):
    _fields_ = [("slots", C.c_int32), ("visits", C.c_int32 * 2), ("max_plies", C.c_int32), ("eval_mode", C.c_int32),
                ("node_capacity", C.c_int32), ("reserved", C.c_int32 * 2)]


_native.register("az_arena_create", C.c_int, [_vp, _vp, C.POINTER(ArenaConfig), C.POINTER(_vp)])
_native.register("az_arena_play", C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, C.POINTER(PoolStats)])


class Arena:
    """Network A (loaded in ``ctx_a``) against network B (``ctx_b``, may be ``ctx_a``) on the GPU, ``slots`` games at a time.
    Every opening is played twice, A moving first in the even game and B in the odd one; each move is the most visited root
    edge of the mover's search (no noise, no sampling)."""

    def __init__(self, ctx_a, ctx_b, slots, visits_a, visits_b, eval_mode=EVAL_BF16, max_plies=400, node_capacity=0):
        cfg = ArenaConfig()
        cfg.slots, cfg.max_plies, cfg.eval_mode, cfg.node_capacity = int(slots), int(max_plies), int(eval_mode), int(node_capacity)
        cfg.visits[0], cfg.visits[1] = int(visits_a), int(visits_b)
        self.cfg = cfg
        self.max_plies = int(max_plies) if int(max_plies) > 0 else 400
        self._h = _vp()
        check(lib().az_arena_create(ctx_a.handle, ctx_b.handle, C.byref(cfg), C.byref(self._h)))
        ctx_a.adopt(self)
        if ctx_b is not ctx_a:
            ctx_b.adopt(self)

    def close(self):
        if self._h:
            lib().az_pool_destroy(self._h)
            self._h = _vp()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def play(self, openings):
        """Plays the 2n games of n openings.  Returns a dict of per-game arrays: ``moves`` (list of move lists), ``plies``,
        ``result`` (1 x won, 2 o won, 0 max_plies reached), ``a_is_x`` (True where network A had x), plus ``stats``."""
        from .rules import positions_array
        arr = positions_array(openings)
        n = len(arr)
        moves = np.zeros((max(2 * n, 1), self.max_plies), dtype=np.uint16)
        plies = np.zeros(max(2 * n, 1), dtype=np.int32)
        result = np.zeros(max(2 * n, 1), dtype=np.int32)
        stats = PoolStats()
        check(lib().az_arena_play(self._h, C.c_void_p(arr.ctypes.data), n, C.c_void_p(moves.ctypes.data),
                                  C.c_void_p(plies.ctypes.data), C.c_void_p(result.ctypes.data), C.byref(stats)))
        games = np.arange(2 * n)
        a_first = games % 2 == 0
        x_first = arr["turn"][games >> 1] == 0
        return {"moves": [[unpack_move(m) for m in moves[i, :plies[i]]] for i in range(2 * n)], "plies": plies[:2 * n].copy(),
                "result": result[:2 * n].copy(), "a_is_x": a_first == x_first, "stats": stats.as_dict()}


def random_openings(ctx, n, plies, seed=0, start_fen=None):
    """``n`` distinct positions reached after ``plies`` uniformly random plies from ``start_fen`` (default: the self-play start
    with its four blockers), none of them decided, played on the device (rules.random_playouts).  A repeated opening would
    repeat its games exactly, so the positions are distinct.  Raises ValueError when random play does not reach n of them."""
    from .rules import START_FEN, positions_array, random_playouts, set_board
    start = set_board(start_fen or START_FEN)
    if plies == 0:
        if n != 1:
            raise ValueError("only one distinct opening after 0 plies")
        start.ply = 0
        return positions_array([start])
    out, seen = [], set()
    batch = max(2 * n, 64)
    for attempt in range(8):
        recs, n_plies, _ = random_playouts(ctx, start, batch, max_plies=plies + 1, seed=(int(seed) << 8) + attempt)
        for g in np.flatnonzero(n_plies > plies):        # a move was played from the position after `plies`: not decided
            r = recs[g, plies]
            key = (int(r["x"]), int(r["o"]))
            if key in seen:
                continue
            seen.add(key)
            out.append((0, (start.turn + plies) & 1, start.blockers, key))
            if len(out) == n:
                return np.array(out, dtype=positions_array([]).dtype)
        batch *= 2
    raise ValueError("random play reached only %d distinct undecided positions after %d plies, %d asked for" % (len(out), plies, n))
