"""GPU self-play generation through the C ABI: JSON-lines records in the reference's format
(self_play_client.cpp:508-582,638-643), every game replayed move by move through the oracle,
plus the legacy 4-function contract of link.py driven like accelerated_generate_games.py:54-83."""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def replay_and_check(oracle, line, visits):
    from oracle.cpu import START_FEN
    game = json.loads(line)
    assert list(game.keys()) == ["boards", "dists", "moves", "result"]          # nlohmann emits sorted keys
    assert len(game["boards"]) == len(game["moves"]) == len(game["dists"]) >= 1
    assert game["result"] in (1, 2)
    p = oracle.set_board(START_FEN)
    for board, move, dist in zip(game["boards"], game["moves"], game["dists"]):
        assert oracle.result(p) == 0
        assert board == oracle.board_json(p)                                     # blockers serialise as 0 (App. B-1)
        legal = {oracle.move_string(m): m for m in oracle.movegen(p)}
        assert move in legal and move in dist
        assert set(dist) <= set(legal) and list(dist) == sorted(dist)
        total = sum(dist.values())
        assert abs(total - 1.0) < 1e-9
        counts = [w * max(visits, 1) for w in dist.values()]
        assert all(w > 0 for w in dist.values())
        p = oracle.makemove(p, legal[move])
    assert oracle.result(p) == game["result"] or len(game["moves"]) == 400
    return len(game["moves"])


def test_selfplay_records_replay_legally(tmp_path, ctx, oracle):
    from ataxxzero_b200 import model, net, search
    net.load_weights(ctx, model.Network.random_init(seed=0))
    out = str(tmp_path / "model-001-0.json")
    with search.Pool(ctx, 64, 40, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=7) as pool:
        stats = pool.selfplay(out, target_games=24, max_seconds=240)
    lines = open(out).read().splitlines()
    assert len(lines) >= 24 and stats["games_finished"] >= 24
    plies = [replay_and_check(oracle, ln, 40) for ln in lines]
    assert sum(plies) <= stats["positions"]
    assert stats["evals"] > 0 and stats["steps"] >= stats["evals"] - stats["positions"] - 64
    # append mode (std::ios_base::app, :691): a second run adds to the same file
    with search.Pool(ctx, 32, 20, eval_mode=search.EVAL_FP32, noise=True, auto_play=True, seed=8) as pool:
        pool.selfplay(out, target_games=4, max_seconds=240)
    assert len(open(out).read().splitlines()) >= len(lines) + 4


def test_selfplay_noise_changes_games_and_seed_reproduces(tmp_path, ctx):
    from ataxxzero_b200 import model, net, search
    net.load_weights(ctx, model.Network.random_init(seed=0))

    def run(seed, name):
        out = str(tmp_path / name)
        with search.Pool(ctx, 8, 30, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=seed) as pool:
            pool.selfplay_ticks(600, out)
        return sorted(open(out).read().splitlines()) if os.path.exists(out) else []
    a, b, c = run(1, "a.json"), run(1, "b.json"), run(2, "c.json")
    assert a and a == b            # same seed -> same games (Philox streams are per game slot)
    assert a != c


def test_capped_pool_replays_bit_for_bit(ctx, monkeypatch):
    """A capped pool -- the net serves only the first `cap` requests of a tick, the rest wait a tick -- replays exactly: which
    requests are served and how far each game gets in a tick follow from the seed, not from when the tree kernel's warps
    finish.  Same seed, same ticks: every root and every counter is the same, bit for bit."""
    from ataxxzero_b200 import model, net, search
    net.load_weights(ctx, model.Network.random_init(seed=0))
    monkeypatch.setenv("AZ_REQ_CAP", "160")         # read when the pool is created: far fewer than the 512 games request

    def run():
        with search.Pool(ctx, 512, 64, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=5) as pool:
            st = pool.selfplay_ticks(300)
            return st, [pool.root(g) for g in range(512)]
    (sa, ra), (sb, rb) = run(), run()
    assert sa["positions"] > 0 and sa["evals"] <= 160 * 300 + 512       # the cap bound: requests really were deferred
    for key in ("ticks", "steps", "evals", "terminal_steps", "positions", "games_finished", "max_depth", "levels"):
        assert sa[key] == sb[key], key
    for x, y in zip(ra, rb):
        assert x["position"].key() == y["position"].key() and x["position"].ply == y["position"].ply
        assert x["moves"] == y["moves"] and x["visits"] == y["visits"] and x["root_visits"] == y["root_visits"]
        assert [float(v).hex() for v in x["total_score"]] == [float(v).hex() for v in y["total_score"]]
        assert [float(v).hex() for v in x["prior"]] == [float(v).hex() for v in y["prior"]]


def test_visit_targets_respected(tmp_path, ctx, oracle):
    """Each recorded distribution is n/N with N >= visits at the moment the move was chosen."""
    from ataxxzero_b200 import model, net, search
    net.load_weights(ctx, model.Network.random_init(seed=0))
    out = str(tmp_path / "g.json")
    with search.Pool(ctx, 16, 64, eval_mode=search.EVAL_BF16, noise=False, auto_play=True, seed=3) as pool:
        pool.selfplay(out, target_games=4, max_seconds=240)
    for ln in open(out).read().splitlines():
        for dist in json.loads(ln)["dists"]:
            smallest = min(dist.values())
            n_total = round(1.0 / smallest) if smallest > 0 else 0
            # smallest weight is k/N for some integer k >= 1, so N >= 1/smallest only if k == 1; check weights are multiples of 1/N
            assert any(all(abs(w * N - round(w * N)) < 1e-6 for w in dist.values()) for N in range(64, 64 + 400))


def test_one_random_move_variant(tmp_path, ctx, oracle):
    """ONE_RANDOM_MOVE (self_play_client.cpp:24,515-552, compile-time off in the shipped build): records carry "random_ply"
    (keys stay sorted), the plies before it are sampled from the visit distribution, the ply AT it is any legal move -- also one
    the search never visited, which rebuilds the tree (MCTS::play miss, :477-483) -- the plies after it take the most visited move,
    and games that end at or before that ply are skipped (:632-637)."""
    from oracle.cpu import START_FEN
    from ataxxzero_b200 import model, net, search
    net.load_weights(ctx, model.Network.random_init(seed=0))
    out = str(tmp_path / "orm.json")
    with search.Pool(ctx, 256, 32, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=11, one_random_move=True) as pool:
        stats = pool.selfplay(out, target_games=120, max_seconds=120)
    assert stats["games_finished"] >= 120 and stats["games_skipped"] > 0          # random_ply ~ U{0..119}: many games end before it
    lines = open(out).read().splitlines()
    off_dist = after = 0
    for ln in lines:
        game = json.loads(ln)
        assert list(game.keys()) == ["boards", "dists", "moves", "random_ply", "result"]
        rp = game["random_ply"]
        assert 0 <= rp < 120 and rp + 1 < len(game["moves"])
        p = oracle.set_board(START_FEN)
        for ply, (board, move, dist) in enumerate(zip(game["boards"], game["moves"], game["dists"])):
            assert board == oracle.board_json(p) and oracle.result(p) == 0
            legal = {oracle.move_string(m): m for m in oracle.movegen(p)}
            assert move in legal and set(dist) <= set(legal)
            assert abs(sum(dist.values()) - 1.0) < 1e-9
            if ply == rp:
                off_dist += move not in dist
            else:
                assert move in dist
                if ply > rp:
                    assert dist[move] == max(dist.values())
                    after += 1
            p = oracle.makemove(p, legal[move])
        assert oracle.result(p) == game["result"]
    assert after > 0 and off_dist > 0          # with ~16..60 legal moves and 32 visits most random moves have no edge


def test_legacy_link_contract(tmp_path, ctx, oracle):
    """accelerated_generate_games.py's loop, verbatim, on top of ataxxzero_b200.link."""
    import ctypes
    from ataxxzero_b200 import link, model, net
    net.load_weights(ctx, model.Network.random_init(seed=0))
    out = str(tmp_path / "legacy.json")
    buffer_size = 16
    work_buffers = [np.zeros((buffer_size, 7, 7, 4), dtype=np.float32) for _ in (0, 1)]
    link.launch_threads(out.encode("utf-8"), 24, ctypes.c_void_p(work_buffers[0].ctypes.data),
                        ctypes.c_void_p(work_buffers[1].ctypes.data), buffer_size, buffer_size * 2)
    try:
        for _ in range(6000):
            i = link.get_workload()
            features = work_buffers[i]
            assert features[..., 0].min() == 1.0                       # plane 0 is all ones
            posteriors, values = net.forward(ctx, features, net.BF16)
            assert posteriors.dtype == np.float32 and posteriors.flags.c_contiguous
            link.complete_workload(i, ctypes.c_void_p(posteriors.ctypes.data), ctypes.c_void_p(values.ctypes.data))
            if os.path.exists(out) and os.path.getsize(out) > 0 and open(out).read().count("\n") >= 3:
                break
    finally:
        link.shutdown()
    lines = open(out).read().splitlines()
    assert len(lines) >= 3
    for ln in lines:
        replay_and_check(oracle, ln, 24)
    # shutdown clears the globals: a second launch must work (self_play_client.cpp:744-748)
    link.launch_threads(out.encode("utf-8"), 8, ctypes.c_void_p(work_buffers[0].ctypes.data),
                        ctypes.c_void_p(work_buffers[1].ctypes.data), buffer_size, buffer_size * 2)
    i = link.get_workload()
    assert i in (0, 1)
    link.shutdown()


def test_full_size_pool_properties(tmp_path, ctx, oracle):
    """BASELINE configs[3] per-GPU shard (2048 games x 800 visits, bf16 net, noise on) started from late-game positions so
    that games finish within the test: size-independent properties instead of a CPU re-run -- every finished record
    replays legally from its first board, every distribution is k/N with N >= 800 and sums to 1, counters add up."""
    import random
    from ataxxzero_b200 import model, net, rules, search
    from oracle.cpu import START_FEN
    net.load_weights(ctx, model.Network.random_init(seed=0))
    rng = random.Random(4)
    roots, start = [], oracle.set_board(START_FEN)
    while len(roots) < 2048:
        p = start
        for _ in range(rng.randrange(90, 170)):
            mv = oracle.movegen(p)
            if not mv or oracle.result(p):
                break
            p = oracle.makemove(p, rng.choice(mv))
        if oracle.result(p) == 0 and oracle.movegen(p):
            roots.append(p)
    arr = np.zeros(2048, dtype=rules.POSITION_DTYPE)
    for i, p in enumerate(roots):
        arr[i] = (p.ply, p.turn, p.blockers, (p.pieces[0], p.pieces[1]))
    out = str(tmp_path / "full.json")
    with search.Pool(ctx, 2048, 800, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=21) as pool:
        pool.set_roots(arr)
        stats = pool.selfplay(out, target_games=600, max_seconds=150)
    assert stats["games_finished"] >= 600 and stats["evals"] > 0
    assert stats["steps"] >= stats["terminal_steps"] and stats["max_depth"] < 1024
    lines = open(out).read().splitlines()
    assert len(lines) >= 600
    first_boards = {tuple(oracle.board_json(p)): p for p in roots}
    checked = 0
    for ln in lines:
        game = json.loads(ln)
        p = first_boards.get(tuple(game["boards"][0]))
        if p is None:                      # a game restarted from the standard opening after its slot's first game ended
            p = start
        for board, move, dist in zip(game["boards"], game["moves"], game["dists"]):
            assert board == oracle.board_json(p) and oracle.result(p) == 0
            legal = {oracle.move_string(m): m for m in oracle.movegen(p)}
            assert move in dist and set(dist) <= set(legal)
            assert abs(sum(dist.values()) - 1.0) < 1e-9
            smallest = min(dist.values())
            assert 0 < smallest and 1.0 / smallest < 5000          # k/N with 800 <= N (carried visits keep N near 800)
            p = oracle.makemove(p, legal[move])
            checked += 1
        assert oracle.result(p) == game["result"]
    assert checked >= 1000          # plies replayed
