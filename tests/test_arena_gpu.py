"""Arena pools (az_arena_create / az_arena_play): two networks play alternate moves of one game, `slots` games at a time.

The arena is checked move for move against a composition of existing entry points: one single-tree search pool per game and
player, the mover's pool run to its visit target, the first move of its principal variation played on both pools."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

AZ_ERR_ARG, AZ_ERR_STATE = -1, -3


@pytest.fixture(scope="module")
def ctx_pair(native):
    """Two contexts on one device, with different networks (different block counts on purpose)."""
    import ataxxzero_b200
    from ataxxzero_b200 import model, net
    a = ataxxzero_b200.Context(device=0, seed=1)
    b = ataxxzero_b200.Context(device=0, seed=2)
    net.load_weights(a, model.Network.random_init(seed=1))
    net.load_weights(b, model.Network.random_init(seed=2, blocks=6))
    yield a, b
    b.close()
    a.close()


@pytest.fixture(scope="module")
def openings6(ctx_pair):
    from ataxxzero_b200 import rules, search
    arr = search.random_openings(ctx_pair[0], 6, 4, seed=11)
    return rules.array_to_positions(arr)


def _single_tree_game(ctxs, opening, a_first, visits, mode, max_plies):
    """The oracle: existing single-tree search pools, one per player, driven from the host."""
    from ataxxzero_b200 import rules, search
    pools = [search.Pool(ctxs[k], 1, visits[k], eval_mode=mode) for k in (0, 1)]
    try:
        for p in pools:
            p.set_root(0, opening)
        pos, mover, moves = opening.clone(), 0 if a_first else 1, []
        while True:
            result = int(rules.result_batch(ctxs[0], [pos])[0])
            if result or len(moves) >= max_plies:
                return moves, result
            pools[mover].run()
            mv = pools[mover].principal_variation(0, 1)[0][0]
            for p in pools:
                p.play(0, mv)
            pos = rules.array_to_positions(rules.makemove_batch(ctxs[0], [pos], [mv]))[0]
            moves.append(mv)
            mover ^= 1
    finally:
        for p in pools:
            p.close()


_single_tree_cache = {}


def _single_tree_games(ctx_pair, openings6, mode, max_plies):
    """Oracle games of the 6 openings (12 games), A 48 visits, B 96 (computed once per mode and ply limit)."""
    key = (mode, max_plies)
    if key not in _single_tree_cache:
        _single_tree_cache[key] = [_single_tree_game(ctx_pair, openings6[i >> 1], i % 2 == 0, (48, 96), mode, max_plies) for i in range(12)]
    return _single_tree_cache[key]


def _compare(got, want):
    for i, (moves, result) in enumerate(want):
        assert got["moves"][i] == moves, "game %d: moves differ" % i
        assert int(got["plies"][i]) == len(moves), "game %d" % i
        assert int(got["result"][i]) == result, "game %d" % i


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("slots", [4, 12])
def test_arena_matches_single_tree_searches(ctx_pair, openings6, mode, slots):
    from ataxxzero_b200 import search
    m = {"fp32": search.EVAL_FP32, "bf16": search.EVAL_BF16}[mode]
    # 60 plies: the host-driven composition costs seconds per game and ply; whole games are checked against the CPU rules
    # by the mirror match below
    with search.Arena(ctx_pair[0], ctx_pair[1], slots, 48, 96, m, 60) as arena:
        got = arena.play(openings6)
    _compare(got, _single_tree_games(ctx_pair, openings6, m, 60))
    assert got["stats"]["positions"] == int(got["plies"].sum())
    want_x = [(i % 2 == 0) == (openings6[i >> 1].turn == 0) for i in range(12)]
    assert list(got["a_is_x"]) == want_x


def test_arena_max_plies_matches_single_tree_searches(ctx_pair, openings6):
    from ataxxzero_b200 import search
    with search.Arena(ctx_pair[0], ctx_pair[1], 4, 48, 96, search.EVAL_BF16, 30) as arena:
        got = arena.play(openings6)
    assert (got["result"] == 0).any() and (got["plies"] <= 30).all()
    _compare(got, _single_tree_games(ctx_pair, openings6, search.EVAL_BF16, 30))


@pytest.fixture(scope="module")
def mirror_match(ctx_pair):
    """One network against itself at a size that fills the GPU: 1024 slots, 1024 openings, 2048 games."""
    from ataxxzero_b200 import search
    openings = search.random_openings(ctx_pair[0], 1024, 6, seed=3)
    with search.Arena(ctx_pair[0], ctx_pair[0], 1024, 32, 32, search.EVAL_BF16, 400) as arena:
        out = arena.play(openings)
    return openings, out


def test_mirror_match_is_even(mirror_match):
    from ataxxzero_b200.cli import arena as cli
    openings, out = mirror_match
    assert len({(int(r["pieces"][0]), int(r["pieces"][1])) for r in openings}) == 1024
    for j in range(1024):
        assert out["moves"][2 * j] == out["moves"][2 * j + 1], "opening %d" % j
        assert out["result"][2 * j] == out["result"][2 * j + 1]
    s = cli.summarize(out["result"], out["a_is_x"])
    assert s["a_wins"] == s["b_wins"] and s["score"] == 0.5


def test_mirror_match_games_are_legal(mirror_match, oracle):
    from ataxxzero_b200 import rules
    openings, out = mirror_match
    for i in range(2048):
        q = oracle.set_board(rules.fen(rules.array_to_positions(openings[i >> 1 : (i >> 1) + 1])[0]))
        for mv in out["moves"][i]:
            assert oracle.legal_move(q, mv), "game %d" % i
            assert oracle.result(q) == 0
            q = oracle.makemove(q, mv)
        want = oracle.result(q)
        if want == 0:
            assert int(out["plies"][i]) == 400
        assert int(out["result"][i]) == want, "game %d" % i


def test_arena_argument_checks(ctx_pair, openings6):
    import ataxxzero_b200
    from ataxxzero_b200 import _native, rules, search
    lib = _native.lib()
    a, b = ctx_pair
    cfg = search.ArenaConfig()
    cfg.slots, cfg.max_plies, cfg.eval_mode = 2, 20, search.EVAL_BF16
    cfg.visits[0], cfg.visits[1] = 8, 8
    h = C.c_void_p()
    assert lib.az_arena_create(None, b.handle, C.byref(cfg), C.byref(h)) == AZ_ERR_ARG
    assert lib.az_arena_create(a.handle, None, C.byref(cfg), C.byref(h)) == AZ_ERR_ARG
    assert lib.az_arena_create(a.handle, b.handle, None, C.byref(h)) == AZ_ERR_ARG
    for bad in ((0, 8), (8, -1), (8, (1 << 22) + 1)):
        cfg.visits[0], cfg.visits[1] = bad
        assert lib.az_arena_create(a.handle, b.handle, C.byref(cfg), C.byref(h)) == AZ_ERR_ARG, bad
    cfg.visits[0], cfg.visits[1] = 8, 8
    if ataxxzero_b200.lib().az_device_count() > 1:
        with ataxxzero_b200.Context(device=1) as other:
            assert lib.az_arena_create(a.handle, other.handle, C.byref(cfg), C.byref(h)) == AZ_ERR_ARG
    with search.Arena(a, b, 2, 8, 8, search.EVAL_BF16, 20) as arena:
        arr = rules.positions_array(openings6)
        buf = [np.zeros(4 * 20, np.uint16), np.zeros(4, np.int32), np.zeros(4, np.int32)]
        ptrs = [C.c_void_p(x.ctypes.data) for x in buf]
        assert lib.az_arena_play(arena._h, C.c_void_p(arr.ctypes.data), 0, *ptrs, None) == AZ_ERR_ARG
        assert lib.az_arena_play(arena._h, None, 2, *ptrs, None) == AZ_ERR_ARG
        assert lib.az_arena_play(arena._h, C.c_void_p(arr.ctypes.data), 2, None, ptrs[1], ptrs[2], None) == AZ_ERR_ARG
        assert lib.az_arena_play(None, C.c_void_p(arr.ctypes.data), 2, *ptrs, None) == AZ_ERR_ARG
        gone = rules.set_board(rules.START_FEN)
        gone.pieces[1] = 0                                   # o has no pieces left: x has won
        decided = rules.positions_array([gone])
        assert lib.az_arena_play(arena._h, C.c_void_p(decided.ctypes.data), 1, *ptrs, None) == AZ_ERR_ARG
        assert lib.az_pool_run(arena._h, 1, None) == AZ_ERR_STATE
        assert lib.az_selfplay_ticks(arena._h, None, 1, None) == AZ_ERR_STATE
        assert lib.az_selfplay_run(arena._h, None, 1, 0, 0.0, None) == AZ_ERR_STATE
        out = arena.play(openings6[:2])                      # the pool and both contexts are still usable
        assert len(out["moves"]) == 4 and (out["plies"] > 0).all()
    with search.Pool(a, 1, 8) as pool:
        assert lib.az_arena_play(pool._h, C.c_void_p(arr.ctypes.data), 1, *ptrs, None) == AZ_ERR_STATE
        pool.set_root(0, rules.set_board(rules.START_FEN))
        assert pool.run()
