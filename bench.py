#!/usr/bin/env python
"""bench.py -- self-play positions/s of the B200-native hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's CPU pipeline
    python bench.py --dump-outputs DIR ...                          # our arm, plus the timed path's outputs as DIR/*.npy

Workload (config.workload): the per-GPU shard of BASELINE configs[3] -- 2048 concurrent self-play
games x 800 visits/move, random-init model-001 net (bf16 tensor-core mode), Dirichlet noise on,
moves sampled ~ visits, every game slot started from a seeded random-playout position (ply ~U[0,120])
so the pool is in a steady-state mix of game phases from the first timed tick.

A "step" is TICKS_PER_STEP ticks; one tick = one pass of the hot path over the whole pool: tree kernel
(consume evaluations, PUCT select/expand/backup, move selection + records) then the net kernel over
the <= 2048 requested leaves.  `value` = recorded plies of all ranks / device time (CUDA events on the
library's stream, max over ranks), nothing crosses PCIe in that region.  `e2e` = the same through the
public API with host inputs and outputs: every step re-uploads the weights from host memory and
az_selfplay_ticks() drains finished games to a JSON-lines file (records D2H + serialisation timed).
Games are independent, so ranks share nothing (weak scaling); NCCL only sums the counters at the end.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "selfplay_positions_per_sec"
UNIT = "positions/s"
GAMES_PER_GPU = 2048
VISITS = 800
TICKS_PER_STEP = 1024
FLOP_PER_EVAL = 347.49e6          # SURVEY 3.5 / 8(d): dense FLOPs of one forward pass
TREE_BYTES_PER_STEP = 13000.0     # SURVEY 8(d): algorithmic bytes of one MCTS step (select + backup + expand)
PERFT_OPS_PER_LEAF = 8.0          # SURVEY 8(d): ~4 64-bit = ~8 int32 ALU operations per counted leaf at depth >= 6


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ----------------------------------------------------------------------------------------------
# clocks: sample nvidia-smi DURING the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in open(self.path).read().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(smax), reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------------------------
# the reference's CPU pipeline (oracle/_ref/self_play_client.so + torch-CPU restatement of model.py)
# ----------------------------------------------------------------------------------------------
class ReferencePipeline:
    """accelerated_generate_games.py:24-83 verbatim, except that `engine.sess.run` (TensorFlow, not
    installable here) is the fp32 torch-CPU (oneDNN) restatement of model.py
    (oracle/net_torch.py, checked against the NumPy restatement).  All host cores: the client runs
    2*buffer_size worker threads, torch's intra-op pool uses the rest."""

    def __init__(self, visits, buffer_size=128):
        import ctypes
        import numpy as np
        import torch
        from oracle import cpu as ocpu, net_numpy, net_torch
        torch.set_num_threads(os.cpu_count() or 1)        # torchrun exports OMP_NUM_THREADS=1; the reference arm gets every core
        self.np, self.ctypes = np, ctypes
        self.kind = "reference" if os.path.exists(ocpu.REF_CLIENT_SO) else "port"
        self.visits, self.B = visits, buffer_size
        conv, bn = net_numpy.init_weights(seed=0)
        self.net = net_torch.TorchNet(conv, bn)            # fp32 torch-CPU (oneDNN) stand-in for TF's sess.run
        self.ocpu = ocpu
        self.evals_per_position = None
        self.epp_sample = ""
        self.out = None
        if self.kind == "reference":
            self.dll = ctypes.CDLL(ocpu.REF_CLIENT_SO)
            self.dll.get_workload.restype = ctypes.c_int
            self.out = tempfile.mktemp(suffix=".json")
            self.buffers = [np.zeros((buffer_size, 7, 7, 4), dtype=np.float32) for _ in (0, 1)]
            self.keep = []
            # the client announces itself on stdout (self_play_client.cpp:686-689); stdout is reserved for the JSON line
            # (and every finished game, :640): for the lifetime of the pipeline fd 1 points at stderr
            sys.stdout.flush()
            self.saved_stdout = os.dup(1)
            os.dup2(2, 1)
            self.dll.launch_threads(self.out.encode(), ctypes.c_int(visits), ctypes.c_void_p(self.buffers[0].ctypes.data),
                                    ctypes.c_void_p(self.buffers[1].ctypes.data), ctypes.c_int(buffer_size),
                                    ctypes.c_int(2 * buffer_size))

    def measure_evals_per_position(self):
        """Evaluations the REFERENCE's own search core needs per played move at this visit count (tree reuse carries
        visits over, adjudicated leaves need none): counted over ONE FULL GAME -- every ply from the opening to the
        end -- played by oracle/_ref/libref.so (reference lines 1-582 compiled here)."""
        if self.evals_per_position is None:
            if self.ocpu.Reference.available():
                ref, orc = self.ocpu.Reference(), self.ocpu.Oracle()
                plies, _, evals = ref.selfplay_greedy(self.ocpu.START_FEN, self.visits, 400, orc.probe_eval_ptr)
                self.evals_per_position = evals / max(len(plies), 1)
                self.epp_sample = "%d evaluations over the %d plies of one full reference game" % (evals, len(plies))
            else:
                orc = self.ocpu.Oracle()
                tree = orc.tree(orc.set_board(self.ocpu.START_FEN), "probe")
                n = 0
                while n < 400 and orc.result(tree.root_position()) == 0:
                    tree.search(self.visits)
                    d = tree.dist()
                    tree.play(max(d, key=lambda e: e[1])[0])
                    n += 1
                self.evals_per_position = tree.evals / max(n, 1)
                self.epp_sample = "%d evaluations over the %d plies of one full game of the oracle port" % (tree.evals, n)
        return self.evals_per_position

    def count_finished(self):
        """(games, plies) the client has appended to its output file so far"""
        games = plies = 0
        try:
            with open(self.out) as f:
                for ln in f:
                    if ln.strip():
                        games += 1
                        plies += len(json.loads(ln)["moves"])
        except (OSError, ValueError):
            pass
        return games, plies

    def run(self, seconds, evaluator=None):
        """Returns evaluations completed in ~`seconds` of wall time.  `evaluator(features) -> (policy, value)` replaces
        the torch-CPU net (used for the host-ceiling / GPU-evaluator variants of the baseline)."""
        np, ctypes = self.np, self.ctypes
        t0 = time.perf_counter()
        evals = 0
        forward = evaluator or self.net.forward
        if self.kind == "reference":
            while time.perf_counter() - t0 < seconds:
                i = self.dll.get_workload()
                policy, value = forward(self.buffers[i])
                policy = np.ascontiguousarray(policy, dtype=np.float32)
                value = np.ascontiguousarray(value, dtype=np.float32)
                self.keep = (self.keep + [(policy, value)])[-6:]
                self.dll.complete_workload(ctypes.c_int(i), ctypes.c_void_p(policy.ctypes.data), ctypes.c_void_p(value.ctypes.data))
                evals += self.B
        else:       # port: our C restatement of the search, one game at a time, same NumPy net
            orc = self.ocpu.Oracle()

            def ev(f):
                p, v = self.net.forward(f.reshape(1, 7, 7, 4))
                return p.reshape(-1), float(v[0, 0])
            tree = orc.tree(orc.set_board(self.ocpu.START_FEN), py_eval=ev)
            while time.perf_counter() - t0 < seconds:
                tree.step()
            evals = tree.evals
        return evals, time.perf_counter() - t0

    def close(self):
        if self.kind == "reference":
            self.dll.shutdown()
            self.ctypes.CDLL(None).fflush(None)
            os.dup2(self.saved_stdout, 1)
            os.close(self.saved_stdout)
            try:
                os.unlink(self.out)
            except OSError:
                pass


def counted_variant(visits, seconds, evaluator, buffer_size=8):
    """The reference client with few enough worker threads (2 x buffer_size) that whole games FINISH inside the sample:
    positions are then counted from its own output file (len(moves) of every line) instead of derived from evaluations.
    In-flight games at the end of the window are lost, so this is a lower bound that cross-checks the derived figure."""
    pipe = ReferencePipeline(visits, buffer_size)
    try:
        if pipe.kind != "reference":
            return None
        t0 = time.perf_counter()
        evals, _ = pipe.run(seconds, evaluator=evaluator)
        dt = time.perf_counter() - t0
        games, plies = pipe.count_finished()
    finally:
        pipe.close()
    return {"threads": 2 * buffer_size, "seconds": dt, "games_finished": games, "positions_counted": plies,
            "positions_per_s_counted": plies / dt, "leaf_evals_per_s": evals / dt,
            "evals_per_counted_position": (evals / plies) if plies else None}


def reference_sample(seconds, visits=VISITS, gpu_evaluator=None):
    pipe = ReferencePipeline(visits)
    variants = {}
    try:
        epp = pipe.measure_evals_per_position()
        pipe.run(min(2.0, seconds / 4))                     # warm the thread pool / BLAS
        evals, dt = pipe.run(seconds)
        if pipe.kind == "reference":
            # BASELINE.md's two other views of the reference: its host side with a free evaluator (the ceiling of the
            # thread pool + hash-map trees), and the reference client fed by OUR GPU net through its own legacy ABI
            zeros = (pipe.np.zeros((pipe.B, 7, 7, 17), dtype=pipe.np.float32), pipe.np.zeros((pipe.B, 1), dtype=pipe.np.float32))
            e0, t0 = pipe.run(4.0, evaluator=lambda f: zeros)
            variants["zero_cost_evaluator_host_ceiling"] = {"leaf_evals_per_s": e0 / t0, "positions_per_s": e0 / t0 / epp}
            if gpu_evaluator is not None:
                e1, t1 = pipe.run(4.0, evaluator=gpu_evaluator)
                variants["reference_client_with_our_gpu_net"] = {"leaf_evals_per_s": e1 / t1, "positions_per_s": e1 / t1 / epp}
    finally:
        pipe.close()
    if pipe.kind == "reference" and gpu_evaluator is not None:
        # in a fresh process: the reference client keeps fill levels / the current buffer in globals that shutdown() does not
        # reset (self_play_client.cpp:597-598,740-749), so a second launch with another buffer size trips its own assert
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "counted", "--visits", str(visits)],
                                 capture_output=True, text=True, timeout=120)
            variants["reference_client_with_our_gpu_net_counted"] = json.loads(out.stdout.strip().splitlines()[-1])
        except Exception as exc:
            variants["reference_client_with_our_gpu_net_counted"] = {"error": repr(exc)}
    cores = os.cpu_count() or 1
    return {"value": evals / dt / epp, "unit": UNIT, "cores": cores, "kind": pipe.kind, "variants": variants,
            "evals_per_position": epp, "evals_per_position_sample": pipe.epp_sample,
            "positions_note": "a reference game needs ~%.0f evaluations per ply x ~185 plies: with 256 concurrent games none finishes "
                              "inside a bounded sample, so positions/s = leaf-evals/s / (evaluations per ply counted over one full "
                              "reference game); the *_counted variant runs 16 worker threads so that games do finish and counts "
                              "len(moves) from the client's output file" % epp,
            "sample": "%.0f s of %s + torch-CPU fp32 net (TensorFlow absent), %d-visit searches, buffer 128 / 256 threads: "
                      "%.0f leaf-evals/s / %.0f evals per played move (%s)"
                      % (dt, "oracle/_ref/self_play_client.so" if pipe.kind == "reference" else "oracle C port", visits,
                         evals / dt, epp, pipe.epp_sample)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    k, w = max(args.steps, 1), max(args.warmup, 0)
    step_s = max(2.0, min(10.0, 150.0 / (k + w)))
    pipe = ReferencePipeline(VISITS)
    try:
        epp = pipe.measure_evals_per_position()
        for _ in range(w):
            pipe.run(step_s)
        evals, dt = 0, 0.0
        for _ in range(k):
            e, t = pipe.run(step_s)
            evals, dt = evals + e, dt + t
    finally:
        pipe.close()
    value = evals / dt / epp
    cores = os.cpu_count() or 1
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": k, "warmup": w,
            "ms_per_step": dt / k * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": "selfplay %d-visit MCTS, reference CPU pipeline (buffer 128 / 256 threads)" % VISITS,
                       "visits": VISITS, "buffer_size": 128, "step": "%.1f s sample" % step_s},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": pipe.kind,
                             "sample": "%d x %.1f s; %.0f leaf-evals/s / %.0f evals per played move (%s)" % (k, step_s, evals / dt, epp, pipe.epp_sample)},
            "positions_note": "no reference game finishes inside the sample (%.0f evaluations per ply x ~185 plies x 256 concurrent "
                              "games): positions = leaf evaluations / evaluations per ply, counted over one full reference game" % epp,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def synthetic_roots(ctx, n, seed):
    """n start positions from seeded random playouts (ply ~U[0,120]) played with the GPU rule kernels."""
    import random
    import numpy as np
    from ataxxzero_b200 import rules
    rng = random.Random(seed)
    arr = rules.positions_array([rules.set_board(rules.START_FEN)] * n)
    target = np.array([rng.randrange(0, 121) for _ in range(n)])
    for ply in range(120):
        res = rules.result_batch(ctx, arr)
        idx = np.nonzero((target > ply) & (res == 0))[0]
        if len(idx) == 0:
            break
        lists = rules.movegen_batch(ctx, arr[idx])
        keep, moves = [], []
        for i, mv in zip(idx, lists):
            if not mv:
                continue
            m = rng.choice(mv)
            keep.append(i)
            moves.append(m)
        if not keep:
            break
        nxt = rules.makemove_batch(ctx, arr[keep], moves)
        ok = rules.result_batch(ctx, nxt) == 0          # never start a game slot on a finished position
        keep = np.array(keep)
        arr[keep[ok]] = nxt[ok]
    return arr


DUMP_GAMES = 2048                 # roots written by --dump-outputs: 2048 games x 256 move slots x 24 bytes = 12.6 MB


def dump_outputs(directory, pool, counters):
    """--dump-outputs: the state the timed steps leave in the pool, one .npy per array.  For every game: the root position
    (ply, turn, blockers, x, o), the per-move root statistics in movegen order (packed move, visits, total score, prior;
    -1 / 0 past the game's move count), the root's visits and value; plus the counters of the timed region.  The game
    records that selfplay_ticks hands its caller are not dumped: the timed steps keep them on the device, and the root state
    stands in for them at a fixed size.  Pools of more than DUMP_GAMES games write the same seeded sample of them every run;
    under torchrun only rank 0 writes.

    The same arguments give the same files: the pool replays its games exactly from the seed (which requests a tick's net
    launch serves, and how far a game gets in a tick, do not depend on timing), so two builds compare array for array."""
    import numpy as np
    from ataxxzero_b200 import rules
    from ataxxzero_b200._native import AZ_MAX_MOVES
    games = pool.games
    idx = np.arange(games)
    if games > DUMP_GAMES:
        idx = np.sort(np.random.default_rng(0).choice(games, DUMP_GAMES, replace=False))
    n = len(idx)
    out = {"game_index": idx.astype(np.float64), "root_position": np.zeros((n, 5)),
           "root_moves": np.full((n, AZ_MAX_MOVES), -1.0, np.float32), "root_edge_visits": np.zeros((n, AZ_MAX_MOVES), np.float32),
           "root_total_score": np.zeros((n, AZ_MAX_MOVES)), "root_prior": np.zeros((n, AZ_MAX_MOVES)),
           "root_visits": np.zeros(n), "root_value": np.zeros(n)}
    for row, g in enumerate(idx):
        r = pool.root(int(g))
        p, k = r["position"], len(r["moves"])
        out["root_position"][row] = (p.ply, p.turn, p.blockers, p.pieces[0], p.pieces[1])    # bitboards < 2^49: exact in float64
        out["root_moves"][row, :k] = [rules.pack_move(m) for m in r["moves"]]
        out["root_edge_visits"][row, :k] = r["visits"]
        out["root_total_score"][row, :k] = r["total_score"]
        out["root_prior"][row, :k] = r["prior"]
        out["root_visits"][row], out["root_value"][row] = r["root_visits"], r["value"]
    names = ("ticks", "steps", "evals", "terminal_steps", "positions", "games_finished", "games_skipped")
    out["timed_counters"] = np.array([counters[name] for name in names], np.float64)      # in the order of `names`
    os.makedirs(directory, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(directory, name + ".npy"), arr)


def run_ours(args):
    import numpy as np
    import torch
    import ataxxzero_b200 as az
    from ataxxzero_b200 import model, net, rules, search

    from ataxxzero_b200 import dist as azdist
    rank, local_rank, world = azdist.env_rank()
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        # NCCL may print its version banner on stdout while the communicator comes up; stdout carries only the JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            azdist.init("nccl")               # counters only: the games themselves never cross ranks
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()

    def allreduce(x, op="sum"):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM if op == "sum" else dist.ReduceOp.MAX)
        return float(t.item())

    k, w = args.steps, max(args.warmup, 3)
    games, visits, ticks = args.games, args.visits, args.ticks_per_step
    ctx = az.Context(device=local_rank, seed=azdist.rank_seed(1000, rank))
    network = model.Network.random_init(seed=0)          # "model-001": the reference's init distributions
    packed = network.packed()
    net.load_weights(ctx, network)
    pool = search.Pool(ctx, games, visits, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=1000 + rank)
    pool.set_roots(synthetic_roots(ctx, games, seed=rank))
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    for _ in range(w):
        pool.selfplay_ticks(ticks)

    # ---- device-resident timed region ----
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    ctx.sync()
    s0 = pool.stats()
    sampler.start()
    ev0.record(stream)
    for _ in range(k):
        pool.selfplay_ticks(ticks)
    ev1.record(stream)
    ctx.sync()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    barrier()
    s1 = pool.stats()
    ms = allreduce(ev0.elapsed_time(ev1), "max")
    d = {key: s1[key] - s0[key] for key in s1}
    positions = allreduce(d["positions"])
    evals = allreduce(d["evals"])
    steps = allreduce(d["steps"])
    value = positions / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pool, d)

    # ---- roofline of the dominant kernel (net), from CUDA events around its launches ----
    pk, pk_kind = peaks()
    # net_seconds / tree_seconds: CUDA events around every k_tree_tick and k_net_pair launch of the event-carrying ticks -- a
    # contiguous window of 256 ticks out of every 1024 (a timing event between two kernels costs ~3 us of GPU time, so the other
    # ticks run without) -- summed; timed_evals = the evaluations exactly those net launches served, counted on the device
    net_s = max(d["net_seconds"], 1e-9)
    timed = max(d.get("timed_ticks", 0), 1)
    timed_evals = d.get("timed_evals", 0)
    achieved = timed_evals * FLOP_PER_EVAL / net_s / 1e12
    peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0)))
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_net_pair"]["dram_bytes_per_launch"]
    except Exception:
        traffic = None
    roofline = {"bound": "tensor", "kernel": "k_net_pair (bf16 tcgen05 cta_group::2 tower on CTA pairs)", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_note": "dram__bytes_read+write per launch from profiles/ (ncu --set full); the weights stream from L2",
                "flop_per_launch": timed_evals / timed * FLOP_PER_EVAL,
                "peak_kind": "%s bf16_tflops_sustained (kernel timed inside a long step)" % pk_kind,
                "net_share_of_step": d["net_seconds"] / max(d["net_seconds"] + d["tree_seconds"], 1e-9),
                "tree_ms_per_tick": d["tree_seconds"] / timed * 1e3, "net_ms_per_tick": d["net_seconds"] / timed * 1e3,
                "launches_timed": int(3 * timed), "evals_timed": int(timed_evals),
                "timing": "CUDA events around every k_tree_tick (with the k_order_requests behind it) and k_net_pair launch of %d ticks (contiguous 256-tick windows, one per 1024 "
                          "ticks of the timed region), summed; the evaluations of exactly those net launches are counted on the device; "
                          "ticks outside the windows carry no events (an event between two kernels costs ~3 us)" % timed}
    # tree kernel: HBM roofline on SURVEY 8(d)'s algorithmic bytes of the reference algorithm (13 KB per MCTS step: every
    # child's P/W/n at every level of the selection path, the backup, 833 logits, the new node)
    tree_s = max(d["tree_seconds"], 1e-9)
    steps_per_launch = d["steps"] / max(d["ticks"], 1)            # MCTS steps per tree launch, mean over the whole timed region
    tree_bytes = steps_per_launch * timed * TREE_BYTES_PER_STEP      # ... times the launches that carried events
    hbm_peak = float(pk.get("hbm_gbs", 6550.0))
    try:
        tree_traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["k_tree_tick"]["dram_bytes_per_launch"]
    except Exception:
        tree_traffic = None
    roofline["kernels"] = {
        "k_tree_tick": {"bound": "hbm", "achieved": tree_bytes / tree_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": tree_bytes / tree_s / 1e9 / hbm_peak, "traffic": tree_traffic,
                        "algorithmic_bytes_per_step": TREE_BYTES_PER_STEP, "steps_per_launch": steps_per_launch,
                        "levels_per_step": d.get("levels", 0) / max(d["steps"], 1),
                        "us_per_level_per_game": tree_s * 1e6 / timed / max(d.get("levels", 0) / max(d["ticks"], 1) / games, 1e-9),
                        "note": "latency-bound by design: one warp per game walks a dependent chain of tree levels; the compact node "
                                "layout reads far fewer bytes than the reference algorithm's 13 KB per step"}}

    # ---- end to end: host weights in, JSON game records out, every step ----
    out_path = azdist.rank_output_path(os.path.join(tempfile.gettempdir(), "az_bench_model-001.json"), rank, max(world, 2))
    if os.path.exists(out_path):
        os.unlink(out_path)
    barrier()
    ctx.sync()
    e0 = pool.stats()
    t0 = time.perf_counter()
    pinned = torch.from_numpy(packed).pin_memory()       # the step's input lives in pinned host memory
    pinned_np = pinned.numpy()
    for _ in range(k):
        net.load_packed(ctx, pinned_np, network.filters, network.blocks)   # H2D: the weights of the .npy, every step
        pool.selfplay_ticks(ticks, out_path)             # D2H: finished games -> JSON lines on the host
    ctx.sync()
    e2e_s = allreduce(time.perf_counter() - t0, "max")
    e1 = pool.stats()
    barrier()
    e2e_positions = allreduce(e1["positions"] - e0["positions"])
    e2e_evals = allreduce(e1["evals"] - e0["evals"])
    record_bytes = e1["record_bytes"] - e0["record_bytes"]
    try:
        json_bytes = os.path.getsize(out_path)
        os.unlink(out_path)
    except OSError:
        json_bytes = 0
    e2e = {"value": e2e_positions / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(packed.nbytes),
           "d2h_bytes_per_step": int(record_bytes / k), "json_bytes_per_step": int(json_bytes / k),
           "leaf_evals_per_s": e2e_evals / e2e_s,
           "api": "net.load_packed (pinned host weights) + Pool.selfplay_ticks(ticks, path) -> az_net_load / az_selfplay_ticks"}

    # ---- BASELINE configs[4]: single-tree search (replicas only, rank 0) + leaf-batch latency of the net kernel ----
    single = {}
    if rank == 0 and not args.no_single_tree:
        golden = os.path.join(ROOT, "tests", "golden", "mcts_golden.json")
        fen = json.load(open(golden))["midgame_fen"] if os.path.exists(golden) else rules.START_FEN
        single = {"fen": fen, "visits": args.single_tree_visits, "runs": {}}
        root_ref = None
        for spec in (0, 4, 16):       # 0 = one leaf per net round trip; k = the k likeliest children of every new node ride along
            with search.Pool(ctx, 1, 64, eval_mode=search.EVAL_BF16, node_capacity=args.single_tree_visits + 64, steps_per_tick=64,
                             speculate=spec) as tree:
                tree.set_root(0, rules.set_board(fen))
                tree.run()                                   # warm-up: 64 visits
                tree.set_visits(args.single_tree_visits)
                st0 = tree.stats()
                t0 = time.perf_counter()
                tree.run()
                dt = time.perf_counter() - t0
                st = tree.stats()
                root = tree.root(0)
                if root_ref is None:
                    root_ref = root
                same = root["visits"] == root_ref["visits"] and [float(x).hex() for x in root["total_score"]] == [float(x).hex() for x in root_ref["total_score"]]
                single["runs"]["speculate_%d" % spec] = {
                    "visits_per_s": (args.single_tree_visits - 64) / dt, "ticks": st["ticks"] - st0["ticks"],
                    "visits_per_tick": (args.single_tree_visits - 64) / max(st["ticks"] - st0["ticks"], 1),
                    "us_per_tick": dt * 1e6 / max(st["ticks"] - st0["ticks"], 1),
                    "root_identical_to_one_leaf_per_tick": bool(same)}
        best = max(single["runs"].values(), key=lambda r: r["visits_per_s"])
        single["visits_per_s"] = best["visits_per_s"]
        single["mode"] = ("bit-exact sequential PUCT, no virtual loss; speculate_k: the k highest-prior children of every consumed node are "
                          "evaluated in the same batch and linked from a per-tree cache when the search reaches them (engine.py:387-392)")
        lat = {}
        feats = np.zeros((128, 7, 7, 4), dtype=np.float32)
        feats[..., 0] = 1.0
        for b in (1, 8, 32, 128):
            samples = []
            for _ in range(200):
                t0 = time.perf_counter()
                net.forward(ctx, feats[:b], net.BF16)
                samples.append((time.perf_counter() - t0) * 1e6)
            samples.sort()
            lat["batch%d" % b] = {"p50_us": samples[len(samples) // 2], "p99_us": samples[int(0.99 * len(samples))]}
        single["leaf_batch_latency_host_to_host"] = lat

    # ---- BASELINE configs[2]: 256 concurrent games x 400 visits on one B200 (>= 10 k recorded positions after warm-up) ----
    config3 = {}
    if rank == 0 and not args.no_single_tree:
        with search.Pool(ctx, 256, 400, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=3000) as small:
            small.set_roots(synthetic_roots(ctx, 256, seed=77))
            small.selfplay_ticks(2048)                   # warm-up
            c0 = small.stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ctx.sync()
            e0.record(stream)
            done = 0
            while done < 64 * 1024:
                small.selfplay_ticks(4096)
                done += 4096
                if small.stats()["positions"] - c0["positions"] >= 10000:
                    break
            e1.record(stream)
            ctx.sync()
            c1 = small.stats()
            cms = e0.elapsed_time(e1)
            cd = {key: c1[key] - c0[key] for key in c1}
            config3 = {"games": 256, "visits": 400, "positions": cd["positions"], "positions_per_s": cd["positions"] / (cms * 1e-3),
                       "leaf_evals_per_s": cd["evals"] / (cms * 1e-3), "ms_per_tick": cms / max(cd["ticks"], 1),
                       "tree_ms_per_tick": cd["tree_seconds"] / max(cd.get("timed_ticks", 0), 1) * 1e3,
                       "net_ms_per_tick": cd["net_seconds"] / max(cd.get("timed_ticks", 0), 1) * 1e3}

    # ---- SURVEY 8f-4: the reference's optimisation step (train.py defaults: minibatch 512, 128 filters x 12 blocks) ----
    train_step = {}
    if rank == 0 and world == 1 and not args.no_single_tree:
        from ataxxzero_b200 import trainer as aztrainer
        rng = np.random.default_rng(11)
        feats = np.zeros((512, 7, 7, 4), np.int8)
        feats[..., 0] = 1
        who = rng.integers(0, 3, size=(512, 7, 7))
        feats[..., 1], feats[..., 2] = who == 1, who == 2
        pol = rng.random((512, 7, 7, 17)).astype(np.float32) ** 8
        pol /= pol.reshape(512, -1).sum(1).reshape(512, 1, 1, 1)
        val = rng.choice([-1.0, 1.0], size=(512, 1)).astype(np.float32)
        tr = aztrainer.Trainer(ctx, model.Network.random_init(seed=1), max_batch=512)
        for _ in range(3):
            tr.train(feats, pol, val, learning_rate=1e-3)
        l0, dev_ms, t0 = tr.launches, 0.0, time.perf_counter()
        for _ in range(30):
            tr.train(feats, pol, val, learning_rate=1e-3)
            dev_ms += tr.last_step_ms
        wall = (time.perf_counter() - t0) / 30
        n_launch = (tr.launches - l0) // 30
        tr.close()
        flop = 3 * 512 * FLOP_PER_EVAL                   # forward + data gradient + weight gradient (algorithmic)
        train_step = {"minibatch": 512, "network": "128 filters x 12 blocks", "ms_per_step_e2e": wall * 1e3, "ms_per_step_device": dev_ms / 30,
                      "samples_per_s_e2e": 512 / wall, "gpu_launches_per_step": n_launch,
                      "tensor_tflops": flop / (dev_ms / 30 * 1e-3) / 1e12, "frac_of_bf16_peak": flop / (dev_ms / 30 * 1e-3) / 1e12 / peak,
                      "note": "host minibatch in, losses out per step (e2e); device = CUDA events around the step's kernels; operands bf16, fp32 accumulate / master weights"}

    # ---- BASELINE configs[0]: uniformly random play, 2000 games, on the device (records copied back to the host) ----
    start = rules.set_board(rules.OPEN_FEN)
    rules.random_playouts(ctx, start, 2000, 400, seed=1)
    t0 = time.perf_counter()
    _, n_plies, _ = rules.random_playouts(ctx, start, 2000, 400, seed=2)
    random_play = {"games": 2000, "positions": int(n_plies.sum()), "positions_per_s": float(n_plies.sum()) / (time.perf_counter() - t0)}

    # ---- secondary metric of BASELINE.json: perft Mnodes/s (device time incl. frontier expansion) ----
    perft = {}
    for depth in (7, 8):
        p = rules.set_board(rules.OPEN_FEN)
        rules.perft(ctx, p, depth)
        t0 = time.perf_counter()
        nodes = rules.perft(ctx, p, depth)
        dt = time.perf_counter() - t0
        perft["depth%d" % depth] = {"nodes": nodes, "mnodes_per_s": nodes / dt / 1e6}
    try:        # integer-ALU roofline of the perft walk kernel: algorithmic int32 ops per leaf x leaves/s against the measured
        # issue peak of the integer pipe (tools/micro/int_alu_peak.cu, same pool), plus the ncu pipe utilisation (profiles/)
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        perft["k_walk_alu_pipe_pct_of_peak_ncu"] = tj["k_walk"]["alu_pipe_pct_of_peak_active"]
        int_peak = float(tj["int_alu_peak"]["iadd3_tops"])
        ach = perft["depth8"]["mnodes_per_s"] * 1e6 * PERFT_OPS_PER_LEAF / 1e12
        roofline["kernels"]["k_walk (perft depth 8)"] = {
            "bound": "int_alu", "achieved": ach, "peak": int_peak, "unit": "Tops/s (int32)", "frac": ach / int_peak,
            "ops_per_leaf": PERFT_OPS_PER_LEAF, "traffic": tj["k_walk"].get("dram_bytes_per_launch"),
            "note": "ops per leaf is SURVEY 8(d)'s algorithmic estimate; peak = measured IADD3 issue rate; wall clock incl. frontier expansion"}
    except Exception:
        pass

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": k, "warmup": w,
            "ms_per_step": ms / k, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "selfplay %d games/GPU x %d visits (BASELINE configs[3] per-GPU shard), random-init model-001"
                                   % (games, visits),
                       "games_per_gpu": games, "visits": visits, "ticks_per_step": ticks, "noise": True,
                       "start": "seeded random-playout positions, ply~U[0,120]",
                       "l2": "working set (node pool + records, several GB per GPU) is far larger than the 126 MB L2; no flush needed",
                       "parallelism": "games sharded across ranks, no data-path collective"},
            "e2e": e2e, "roofline": roofline, "clocks": clocks, "gpu_launches": int(d["kernel_launches"]),
            "extra": {"leaf_evals_per_s": evals / (ms * 1e-3), "mcts_steps_per_s": steps / (ms * 1e-3),
                      "evals_per_position": evals / max(positions, 1), "max_depth": s1["max_depth"], "perft": perft,
                      "single_tree": single, "config3_256x400": config3, "random_play": random_play, "train_step": train_step}}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        pool.close()
        try:
            line["cpu_baseline"] = reference_sample(args.cpu_seconds, visits,
                                                    gpu_evaluator=lambda f: net.forward(ctx, f, net.BF16))
            # second metric of BASELINE.json: the reference's own movegen/makemove (oracle/_ref/perft_ref) on the host cores
            from oracle import cpu as ocpu
            if os.path.exists(ocpu.REF_PERFT):
                cores = os.cpu_count() or 1
                n1, s1 = ocpu.ref_perft(ocpu.OPEN_FEN, 6, 1)
                nN, sN = ocpu.ref_perft(ocpu.OPEN_FEN, 7, cores)
                line["cpu_baseline"]["perft"] = {"kind": "reference", "depth6_1thread_mnodes_per_s": n1 / s1 / 1e6,
                                                 "depth7_%dthreads_mnodes_per_s" % cores: nN / sN / 1e6, "nodes": [n1, nN]}
            # the honest comparisons with the reference's own SEARCH ENGINE (BASELINE.md): the unmodified client fed by our GPU
            # net through its legacy ABI, and its host side alone with a zero-cost evaluator
            var = line["cpu_baseline"].get("variants", {})
            if var.get("reference_client_with_our_gpu_net"):
                line["vs_reference_client_gpu_net"] = e2e["leaf_evals_per_s"] / var["reference_client_with_our_gpu_net"]["leaf_evals_per_s"]
            if var.get("zero_cost_evaluator_host_ceiling"):
                line["vs_reference_host_ceiling"] = e2e["leaf_evals_per_s"] / var["zero_cost_evaluator_host_ceiling"]["leaf_evals_per_s"]
            line["vs_reference_note"] = ("e2e leaf evaluations/s of this arm (search + net + records, host in / host out) / leaf evaluations/s of "
                                         "the unmodified reference client on the box's host cores: fed by OUR GPU net through its own legacy ABI, "
                                         "and with a zero-cost evaluator (its thread pool + hash-map trees alone).  Leaf evaluations are what both "
                                         "pipelines count exactly; positions/s = that / evaluations per ply, the same factor for the same games.  "
                                         "The --impl reference arm additionally pays for an fp32 conv net on the host cores")
        except Exception as exc:        # the baseline is reported, never the product path
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable",
                                    "sample": "failed: %r" % (exc,)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def positive_int(text):
    value = int(text)
    if value < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % value)
    return value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=4, help="timed steps of TICKS_PER_STEP ticks each")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "counted"])
    ap.add_argument("--games", type=int, default=GAMES_PER_GPU)
    ap.add_argument("--visits", type=int, default=VISITS)
    ap.add_argument("--ticks-per-step", type=int, default=TICKS_PER_STEP)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-single-tree", action="store_true")
    ap.add_argument("--single-tree-visits", type=int, default=100000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed (see dump_outputs) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "counted":         # helper of the cpu_baseline leg (see reference_sample)
        import ataxxzero_b200 as az
        from ataxxzero_b200 import model, net
        ctx = az.Context(device=0, seed=1)
        net.load_weights(ctx, model.Network.random_init(seed=0))
        res = counted_variant(args.visits, 12.0, lambda f: net.forward(ctx, f, net.BF16))
        print(json.dumps(res), flush=True)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
