"""Match runner between UAI engines, with the flags of the reference's ``uai_ringmaster.py`` (uai_ringmaster.py:205-266):
round-robin (or ``--gauntlet``: the first engine against all others), every pairing played with both colours, moves
forwarded to both engines, wins tallied, games appended to a PGN file.  Used to compare engine strength, e.g. the
reference's ``uai_interface.py`` against ``python -m ataxxzero_b200.cli.uai_interface``.  Host-side orchestration only;
``--games N`` (not in the reference, which runs until killed) ends the tournament after N games."""
import argparse
import datetime
import itertools
import random
import shlex
import sys
import time

from .. import ataxx_rules
from .generate_games import UAIPlayer
from .uai_interface import uai_decode_move, uai_encode_move

OPENING_DEPTH = 0


def play_one_game(args, engine1, engine2, opening_moves):
    print('Game: "%s" vs "%s" with opening: [%s]' % (" ".join(engine1), " ".join(engine2), ", ".join(map(uai_encode_move, opening_moves))))
    game = {"moves": [], "opening": opening_moves, "start_time": time.time(), "white": engine1, "black": engine2}
    players = [UAIPlayer(engine1), UAIPlayer(engine2)]
    board = ataxx_rules.AtaxxState.initial()
    ply = 0
    try:
        while board.result() is None:
            counts = (board.board.count(1), board.board.count(2))
            if args.show_games:
                print("\n======= Player %i move.  [%3i plies] Score: %2i - %2i\n%s\n%s" % (ply % 2 + 1, ply, counts[0], counts[1], board.fen(), board))
            if ply < len(opening_moves):
                move = opening_moves[ply]
            elif len(board.legal_moves()) == 1:
                move, = board.legal_moves()                      # forced (a pass included)
            else:
                players[ply % 2].set_state(board)
                move = players[ply % 2].genmove(int(args.tc * 1000))
            if move not in board.legal_moves():
                raise ValueError("illegal move %s from %r at %s" % (uai_encode_move(move), players[ply % 2].cmd, board.fen()))
            board.move(move)
            game["moves"].append(move)
            ply += 1
            if args.max_plies is not None and ply > args.max_plies:
                break
    finally:
        for player in players:
            player.quit()
    game["result"] = board.result() if board.result() is not None else "invalid"
    game["end_time"] = time.time()
    game["final_score"] = (board.board.count(1), board.board.count(2))
    print("[%3i plies] Score: %2i - %2i" % ((ply,) + game["final_score"]))
    return game


def write_game_to_pgn(args, path, game, round_index=1):
    """Appends one game.  A game that starts from a set position carries its FEN ("fen": SetUp / FEN tags), and a game that
    was not played on the clock its own "time_control" text; games without these keys are written as before."""
    tags = [("Event", "?"), ("Site", "?"), ("Date", datetime.datetime.now().strftime("%Y.%m.%d")), ("Round", "%i" % round_index),
            ("White", " ".join(game["white"])), ("Black", " ".join(game["black"]))]
    if game.get("fen"):
        tags += [("SetUp", "1"), ("FEN", game["fen"])]
    tags += [("Opening", ", ".join(map(uai_encode_move, game["opening"]))),
            ("GameStartTime", datetime.datetime.fromtimestamp(game["start_time"]).isoformat()),
            ("GameEndTime", datetime.datetime.fromtimestamp(game["end_time"]).isoformat()),
            ("Plycount", "%i" % len(game["moves"])), ("Result", {1: "1-0", 2: "0-1", "invalid": "1/2-1/2"}[game["result"]]),
            ("FinalScore", "%i-%i" % game["final_score"]), ("TimeControl", game.get("time_control") or "+%r" % (args.tc,))]
    with open(path, "a+") as f:
        for key, value in tags:
            print('[%s "%s"]' % (key, value), file=f)
        print(file=f)
        print(" ".join(map(uai_encode_move, game["moves"])), file=f)
        print(file=f)


def get_opening(args):
    if args.opening is not None:
        return [uai_decode_move(m.strip()) for m in args.opening.split(",") if m.strip()]
    board, moves = ataxx_rules.AtaxxState.initial(), []
    for _ in range(OPENING_DEPTH):
        moves.append(random.choice(board.legal_moves()))
        board.move(moves[-1])
    return moves


def build_parser():
    parser = argparse.ArgumentParser()
    parser.add_argument("--engine", metavar="CMD", action="append", help="Engine command.")
    parser.add_argument("--show-games", action="store_true", help="Show the games while they're being generated.")
    parser.add_argument("--opening", metavar="MOVES", type=str, default=None, help="Comma separated sequence of moves for the opening.")
    parser.add_argument("--max-plies", metavar="N", type=int, default=None, help="Maximum number of plies in a game before it's aborted and rejected.")
    parser.add_argument("--pgn-out", metavar="PATH", type=str, default=None, help="PGN file path to accumulate games into. Writes in append mode.")
    parser.add_argument("--gauntlet", action="store_true", help="Just the first engine plays against all the other engines.")
    parser.add_argument("--tc", metavar="SEC", type=float, default=1.0, help="Seconds per move for all engines.")
    parser.add_argument("--games", metavar="N", type=int, default=None, help="Stop after N games (default: run until interrupted).")
    return parser


def main(argv=None):
    args = build_parser().parse_args(argv)
    print("Options:", args)
    engines = [tuple(shlex.split(cmd)) for cmd in (args.engine or [])]
    if len(engines) < 2:
        raise SystemExit("need at least two --engine commands")
    for i, engine in enumerate(engines):
        print("%4i: %s" % (i + 1, engine))
    wins = {engine: 0 for engine in engines}
    queue, played, annulled = [], 0, 0
    while args.games is None or played < args.games:
        if not queue:
            pairings = [(engines[0], e) for e in engines[1:]] if args.gauntlet else list(itertools.combinations(engines, 2))
            random.shuffle(pairings)
            for pairing in pairings:                     # every pairing both ways round, same opening
                opening = get_opening(args)
                queue += [(opening, pairing), (opening, pairing[::-1])]
        opening, pair = queue.pop()
        game = play_one_game(args, pair[0], pair[1], opening)
        played += 1
        if game["result"] in (1, 2):
            wins[pair[game["result"] - 1]] += 1
        else:
            wins[pair[0]] += 0.5
            wins[pair[1]] += 0.5
            annulled += 1
        print("Wins: %s (annulled: %i)" % (" - ".join(str(wins[e]) for e in engines), annulled))
        if args.pgn_out:
            write_game_to_pgn(args, args.pgn_out, game, round_index=played)
    return wins


if __name__ == "__main__":
    main()
