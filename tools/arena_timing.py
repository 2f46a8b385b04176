"""Arena timing on the GPU: games/s and plies/s of az_arena_play, the device memory its pool holds, and the wall time of the
single-tree composition (one search pool per game and player, driven from the host) next to the arena for the same games.

    python tools/arena_timing.py [--slots 2048 --visits 400 --max-plies 400 --compare-games 64 --compare-plies 400]

Prints the card's name and power limit with the numbers.  Two random-init networks (12 and 6 blocks) play each other."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown card"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=2048)
    ap.add_argument("--visits", type=int, default=400)
    ap.add_argument("--max-plies", type=int, default=400)
    ap.add_argument("--mode", type=int, default=1, help="0 fp32, 1 bf16, 3 f16")
    ap.add_argument("--compare-games", type=int, default=64, help="games of the single-tree comparison (0: skip it)")
    ap.add_argument("--compare-visits", type=int, default=48)
    ap.add_argument("--compare-plies", type=int, default=400)
    args = ap.parse_args()
    import torch
    import ataxxzero_b200
    from ataxxzero_b200 import model, net, search
    from test_arena_gpu import _single_tree_game
    from ataxxzero_b200.rules import array_to_positions
    print("card: %s" % card())
    a = ataxxzero_b200.Context(device=0, seed=1)
    b = ataxxzero_b200.Context(device=0, seed=2)
    net.load_weights(a, model.Network.random_init(seed=1))
    net.load_weights(b, model.Network.random_init(seed=2, blocks=6))
    openings = search.random_openings(a, args.slots // 2, 4, seed=7)
    free0 = torch.cuda.mem_get_info(0)[0]
    with search.Arena(a, b, args.slots, args.visits, args.visits, args.mode, args.max_plies) as arena:
        pool_bytes = free0 - torch.cuda.mem_get_info(0)[0]
        t0 = time.perf_counter()
        out = arena.play(openings)
        dt = time.perf_counter() - t0
    plies = int(out["plies"].sum())
    print("arena: %d slots, %d visits, mode %d, max_plies %d: %d games, %d plies in %.2f s: %.2f games/s, %.0f plies/s, %d ticks; "
          "pool device memory %.2f GiB (free memory before / after az_arena_create)" % (
              args.slots, args.visits, args.mode, args.max_plies, len(out["plies"]), plies, dt, len(out["plies"]) / dt, plies / dt,
              out["stats"]["ticks"], pool_bytes / 2 ** 30))
    if args.compare_games:
        n = args.compare_games // 2
        small = search.random_openings(a, n, 4, seed=9)
        v = (args.compare_visits, args.compare_visits)
        t0 = time.perf_counter()
        with search.Arena(a, b, args.compare_games, v[0], v[1], args.mode, args.compare_plies) as arena:
            got = arena.play(small)
        t_arena = time.perf_counter() - t0
        pos = array_to_positions(small)
        t0 = time.perf_counter()
        want = [_single_tree_game((a, b), pos[i >> 1], i % 2 == 0, v, args.mode, args.compare_plies) for i in range(2 * n)]
        t_single = time.perf_counter() - t0
        same = all(got["moves"][i] == w[0] and int(got["result"][i]) == w[1] for i, w in enumerate(want))
        print("%d games at %d visits, max_plies %d: single-tree composition %.1f s, az_arena_play %.2f s (%.0fx); same games: %s" % (
            2 * n, v[0], args.compare_plies, t_single, t_arena, t_single / t_arena, same))
    b.close()
    a.close()


if __name__ == "__main__":
    main()
