"""The arena command line without a GPU: argument parsing, the score / Elo / interval arithmetic, PGN output."""
import argparse
import datetime
import math

import pytest


def test_parse_args_defaults_and_per_side_visits():
    from ataxxzero_b200.cli import arena
    a = arena.parse_args(["--network-a", "a.npy", "--network-b", "b.npy"])
    assert (a.visits_a, a.visits_b, a.openings, a.opening_plies, a.slots, a.mode, a.max_plies) == (400, 400, 256, 4, 1024, "bf16", 400)
    assert a.pgn_out is None and a.seed == 0 and a.device == 0
    a = arena.parse_args(["--network-a", "a", "--network-b", "b", "--visits", "64", "--visits-b", "256", "--mode", "f16",
                          "--openings", "10", "--opening-plies", "0", "--seed", "5", "--slots", "8", "--max-plies", "30",
                          "--pgn-out", "x.pgn", "--device", "1"])
    assert (a.visits_a, a.visits_b, a.mode, a.openings, a.opening_plies, a.seed, a.slots, a.max_plies, a.pgn_out, a.device) == (
        64, 256, "f16", 10, 0, 5, 8, 30, "x.pgn", 1)
    assert arena.MODES[a.mode] == 3
    for bad in (["--visits-a", "0"], ["--openings", "0"], ["--opening-plies", "-1"], ["--mode", "fp8"]):
        with pytest.raises(SystemExit):
            arena.parse_args(["--network-a", "a", "--network-b", "b"] + bad)
    with pytest.raises(SystemExit):
        arena.parse_args(["--network-a", "a"])


def test_score_elo_and_interval():
    from ataxxzero_b200.cli import arena
    # three openings.  Games (result, A had x):  opening 0: A wins as x, A wins as o -> 1.0
    #                                            opening 1: x wins with B, max plies  -> (0 + 0.5) / 2 = 0.25
    #                                            opening 2: o wins with A, x wins with A -> 1.0
    result = [1, 2, 1, 0, 2, 1]
    a_is_x = [True, False, False, True, False, True]
    s = arena.summarize(result, a_is_x)
    assert (s["games"], s["a_wins"], s["b_wins"], s["max_plies"]) == (6, 4, 1, 1)
    assert s["score"] == pytest.approx(0.75)
    assert s["elo"] == pytest.approx(-400 * math.log10(1 / 0.75 - 1))          # +190.85
    assert s["elo"] == pytest.approx(190.848, abs=1e-3)
    # pair scores 1, 0.25, 1: sample std 0.4330127, half width 1.96 * 0.4330127 / sqrt(3) = 0.49; the upper end is clipped at 1
    lo, hi = s["score_interval"]
    assert lo == pytest.approx(0.75 - 0.49, abs=1e-9) and hi == 1.0
    assert s["elo_interval"][0] == pytest.approx(-400 * math.log10(1 / 0.26 - 1)) and s["elo_interval"][1] == math.inf
    even = arena.summarize([1, 1, 2, 2], [True, False, True, False])
    assert even["score"] == 0.5 and even["elo"] == 0.0 and even["score_interval"] == (0.5, 0.5)
    one = arena.summarize([0, 0], [True, False])
    assert one["score"] == 0.5 and one["score_interval"] is None and one["elo_interval"] is None
    assert arena.elo(0.0) == -math.inf and arena.elo(1.0) == math.inf
    text = arena.format_summary(s, "new", "old")
    assert "new wins 4, old wins 1, 1 games reached the ply limit" in text and "+190.8" in text


def _game(**extra):
    game = {"moves": [("c", (1, 1)), ((0, 0), (2, 2))], "opening": [("c", (3, 3))], "start_time": 1.7e9, "end_time": 1.7e9 + 60,
            "white": ("engine", "one"), "black": ("two",), "result": 2, "final_score": (3, 5)}
    game.update(extra)
    return game


def test_pgn_without_start_fen_is_unchanged(tmp_path):
    from ataxxzero_b200.cli import uai_ringmaster
    path = tmp_path / "games.pgn"
    uai_ringmaster.write_game_to_pgn(argparse.Namespace(tc=1.5), str(path), _game(), round_index=3)
    start = datetime.datetime.fromtimestamp(1.7e9).isoformat()
    end = datetime.datetime.fromtimestamp(1.7e9 + 60).isoformat()
    date = datetime.datetime.now().strftime("%Y.%m.%d")
    want = ('[Event "?"]\n[Site "?"]\n[Date "%s"]\n[Round "3"]\n[White "engine one"]\n[Black "two"]\n[Opening "d4"]\n'
            '[GameStartTime "%s"]\n[GameEndTime "%s"]\n[Plycount "2"]\n[Result "0-1"]\n[FinalScore "3-5"]\n[TimeControl "+1.5"]\n'
            '\nb6 a7c5\n\n' % (date, start, end))
    assert path.read_text() == want


def test_pgn_with_start_fen(tmp_path):
    from ataxxzero_b200.cli import uai_ringmaster
    path = tmp_path / "games.pgn"
    fen = "x5o/7/3-3/2-1-2/3-3/7/o5x x"
    uai_ringmaster.write_game_to_pgn(argparse.Namespace(tc=1.0), str(path), _game(fen=fen, time_control="48/96 visits", result="invalid"))
    lines = path.read_text().splitlines()
    assert lines[5:8] == ['[Black "two"]', '[SetUp "1"]', '[FEN "%s"]' % fen]
    assert '[Result "1/2-1/2"]' in lines and '[TimeControl "48/96 visits"]' in lines


def test_pgn_games_of_an_arena_result():
    import numpy as np
    from ataxxzero_b200 import ataxx_rules, rules
    from ataxxzero_b200.cli import arena
    start = ataxx_rules.AtaxxState.from_fen(rules.START_FEN)
    opening = rules.positions_array([start.to_position()])
    first = ataxx_rules.AtaxxState.from_fen(rules.START_FEN)
    legal = [rules.from_reference_move(m) for m in first.legal_moves()]
    moves = [legal[0]]
    out = {"moves": [moves, moves], "result": np.array([0, 0]), "a_is_x": np.array([True, False]), "plies": np.array([1, 1])}
    games = arena.pgn_games(opening, out, "A", "B", 1.7e9, 1.7e9 + 1, (48, 96))
    assert [g["white"] for g in games] == [("A",), ("B",)] and [g["black"] for g in games] == [("B",), ("A",)]
    assert games[0]["fen"] == start.fen() and games[0]["result"] == "invalid" and games[0]["time_control"] == "48/96 visits"
    after = ataxx_rules.AtaxxState.from_fen(rules.START_FEN)
    after.move(rules.to_reference_move(moves[0]))
    assert games[0]["final_score"] == (after.board.count(1), after.board.count(2))
