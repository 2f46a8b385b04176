"""Match two networks on the GPU: ``python -m ataxxzero_b200.cli.arena --network-a new.npy --network-b old.npy``.

Both networks search with the device-resident PUCT trees of the self-play pool (search.Arena over az_arena_play): every
opening is played twice, once with each network moving first, and each move is the most visited root edge after the
mover's visit target.  The summary counts games that reach --max-plies as half a point each, as uai_ringmaster.py does,
and its 95 % interval is taken over opening pairs, because the two games of one opening are not independent."""
import argparse
import math
import time

import numpy as np

from .. import ataxx_rules

MODES = {"fp32": 0, "bf16": 1, "f16": 3}


def build_parser():
    parser = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    parser.add_argument("--network-a", metavar="PATH", required=True, help="Network A (.npy in the reference's model format).")
    parser.add_argument("--network-b", metavar="PATH", required=True, help="Network B.")
    parser.add_argument("--visits", metavar="N", type=int, default=400, help="Visits per move for both networks.")
    parser.add_argument("--visits-a", metavar="N", type=int, default=None, help="Visits per move of A (default: --visits).")
    parser.add_argument("--visits-b", metavar="N", type=int, default=None, help="Visits per move of B (default: --visits).")
    parser.add_argument("--openings", metavar="N", type=int, default=256, help="Distinct openings; each is played twice.")
    parser.add_argument("--opening-plies", metavar="K", type=int, default=4, help="Uniformly random plies that make an opening.")
    parser.add_argument("--seed", type=int, default=0, help="Seed of the random openings.")
    parser.add_argument("--slots", metavar="N", type=int, default=1024, help="Games played at once.")
    parser.add_argument("--mode", choices=sorted(MODES), default="bf16", help="Precision of both networks' forward pass.")
    parser.add_argument("--max-plies", metavar="N", type=int, default=400, help="A game that reaches N plies counts half a point each.")
    parser.add_argument("--device", type=int, default=0, help="CUDA device.")
    parser.add_argument("--pgn-out", metavar="PATH", default=None, help="PGN file the games are appended to.")
    return parser


def parse_args(argv=None):
    args = build_parser().parse_args(argv)
    args.visits_a = args.visits if args.visits_a is None else args.visits_a
    args.visits_b = args.visits if args.visits_b is None else args.visits_b
    if min(args.visits_a, args.visits_b, args.openings, args.slots, args.max_plies) < 1 or args.opening_plies < 0:
        raise SystemExit("visits, openings, slots and max-plies must be positive, opening-plies non-negative")
    return args


def elo(score):
    """Elo difference of a player that scores ``score`` (0..1) per game; +-inf at 1 and 0."""
    if score <= 0.0:
        return -math.inf
    if score >= 1.0:
        return math.inf
    return -400.0 * math.log10(1.0 / score - 1.0)


def summarize(result, a_is_x):
    """Tally of a match: ``result[i]`` (1 x won, 2 o won, 0 max plies) and ``a_is_x[i]`` of games 2j, 2j + 1 of opening j.
    A's score counts a game without a winner as half a point.  The 95 % interval is the normal interval of the mean over
    opening pairs (the two games of an opening share it, so they are one sample), mapped to Elo; None with one opening."""
    result = np.asarray(result)
    a_is_x = np.asarray(a_is_x, dtype=bool)
    a_won = ((result == 1) & a_is_x) | ((result == 2) & ~a_is_x)
    b_won = ((result == 1) & ~a_is_x) | ((result == 2) & a_is_x)
    points = a_won + 0.5 * (result == 0)
    pairs = points.reshape(-1, 2).mean(axis=1)
    score = float(pairs.mean())
    out = {"games": int(len(result)), "a_wins": int(a_won.sum()), "b_wins": int(b_won.sum()), "max_plies": int((result == 0).sum()),
           "score": score, "elo": elo(score), "score_interval": None, "elo_interval": None}
    if len(pairs) > 1:
        half = 1.96 * float(pairs.std(ddof=1)) / math.sqrt(len(pairs))
        lo, hi = max(score - half, 0.0), min(score + half, 1.0)
        out["score_interval"] = (lo, hi)
        out["elo_interval"] = (elo(lo), elo(hi))
    return out


def format_summary(s, name_a="A", name_b="B"):
    lines = ["%s wins %d, %s wins %d, %d games reached the ply limit (half a point each), %d games" % (
        name_a, s["a_wins"], name_b, s["b_wins"], s["max_plies"], s["games"]),
        "score of %s: %.4f   Elo difference %+.1f" % (name_a, s["score"], s["elo"])]
    if s["score_interval"] is not None:
        lines.append("95%% interval over opening pairs: score %.4f .. %.4f, Elo %+.1f .. %+.1f" % (s["score_interval"] + s["elo_interval"]))
    return "\n".join(lines)


def pgn_games(openings, out, name_a, name_b, start_time, end_time, visits):
    """The games of ``Arena.play`` as uai_ringmaster game dicts, each with the FEN of its opening."""
    from ..rules import array_to_positions, to_reference_move
    if isinstance(openings, np.ndarray):
        openings = array_to_positions(openings)
    games = []
    for i, moves in enumerate(out["moves"]):
        o = openings[i >> 1]
        state = ataxx_rules.AtaxxState.from_position(o)
        fen = state.fen()
        ref_moves = [to_reference_move(m) for m in moves]
        for m in ref_moves:
            state.move(m)
        x, o_name = (name_a, name_b) if out["a_is_x"][i] else (name_b, name_a)
        result = int(out["result"][i])
        games.append({"moves": ref_moves, "opening": [], "start_time": start_time, "end_time": end_time, "white": (x,), "black": (o_name,),
                      "result": result if result in (1, 2) else "invalid", "final_score": (state.board.count(1), state.board.count(2)),
                      "fen": fen, "time_control": "%d/%d visits" % tuple(visits)})
    return games


def main(argv=None):
    args = parse_args(argv)
    import ataxxzero_b200
    from .. import model, net, search
    from .uai_ringmaster import write_game_to_pgn
    ctx_a = ataxxzero_b200.Context(device=args.device)
    ctx_b = ataxxzero_b200.Context(device=args.device)
    try:
        net.load_weights(ctx_a, model.Network.load(args.network_a))
        net.load_weights(ctx_b, model.Network.load(args.network_b))
        openings = search.random_openings(ctx_a, args.openings, args.opening_plies, seed=args.seed)
        start = time.time()
        with search.Arena(ctx_a, ctx_b, args.slots, args.visits_a, args.visits_b, MODES[args.mode], args.max_plies) as arena:
            out = arena.play(openings)
        end = time.time()
    finally:
        ctx_a.close()
        ctx_b.close()
    summary = summarize(out["result"], out["a_is_x"])
    print(format_summary(summary, args.network_a, args.network_b))
    print("%d games, %d plies in %.1f s" % (summary["games"], int(out["plies"].sum()), end - start))
    if args.pgn_out:
        games = pgn_games(openings, out, args.network_a, args.network_b, start, end, (args.visits_a, args.visits_b))
        for k, game in enumerate(games):
            write_game_to_pgn(args, args.pgn_out, game, round_index=k + 1)
    return summary


if __name__ == "__main__":
    main()
