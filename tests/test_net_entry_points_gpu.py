"""The net kernels' entry points that the search calls, checked directly at multi-wave batch sizes.

tests/test_net_gpu.py and tests/test_net_pair_tiles_gpu.py check the plain forward pass from host feature planes.  The search
runs three other passes of the same kernels, and this file checks each of them against that plain pass, bit for bit, and
against the fp64 restatement of model.py (oracle/net_numpy.py):
  * position input: the net encodes az_position[] itself (AZ_IN_POS), under both variants of k_net_pair (one and two tiles
    per CTA) and in the three modes, with the board count also read from device memory;
  * the speculative cache pass (k_net_pair's one-tile CACHE kind): logits null, the values, the softmax numerators
    exp((double)logit) and their strictly sequential sums scattered through an output map into a cache table, whose trash
    row takes dropped requests;
  * the symmetry ensemble (az_net_forward_sym8, k_net_pair's one-tile SYM8 kind): each CTA evaluates one position at a time
    in 4 passes of 2 images, several positions per CTA.

S is the device's SM count (148 on a B200) and R = 4 * S a full round of boards: one pass of every CTA of either kernel
variant.  Sizes around R, 2R and 3R make CTAs walk a second and third unit, and leave partial units at the tail.

Positions are random walks from the C++ start position, from the empty board and from positions with blockers, played to
the end of the game, so both sides are to move and late endgames and finished games are included.  Their feature planes
come from the C oracle (oracle.features) and must equal the library's own encoding (rules.features_batch).

Bounds against the fp64 oracle, on a fixed sample of boards of each batch (the head and tail of every batch and random rows;
the fp64 oracle takes ~15 ms of host time per board).  At random init they are test_net_gpu.py's: 1e-5 in FP32, 2e-2 in BF16,
3e-4 in F16.  At trained scale (oracle.net_numpy.trained_scale_weights, logits of standard deviation 2) they are
test_bf16_at_trained_scale's: BF16 max 3 % of the largest logit and rms 2.5 % of the logits' deviation, values 0.15; F16
2e-2; FP32 1e-5 of full scale and 5e-5 on values.  Measured on a B200 (1000 W power limit):
  * random init, the largest |error| over the sampled boards of every size and variant (the same in both variants):
    FP32 logits 1.5e-7, values 1.9e-8; BF16 logits 8.6e-4, values 8.8e-5; F16 logits 9.6e-5, values 1.2e-5.
  * trained scale, position input at R + 1 boards (largest logit 11.1): BF16 logits 0.138 (1.24 % of full scale), rms
    1.38 % of the logits' deviation, values 0.044; F16 logits 1.87e-2, values 9.6e-3; FP32 logits 2.5e-5, values 7.5e-6.
  * symmetry ensemble, random init: FP32 logits 5.1e-8, values 7.1e-9; BF16 6.0e-4 and 2.9e-5;
    F16 5.0e-5 and 3.9e-6.  At trained scale (largest ensemble logit 4.9), BF16: logits 0.093 (1.89 %), rms 0.72 %,
    values 5.0e-3.
"""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FP32_TOL, BF16_TOL, F16_TOL = 1e-5, 2e-2, 3e-4
SENTINEL = -7.0

# k_net_pair with two or one tiles per CTA; the variant is read when weights load
POS_VARIANTS = {
    "pair2": {"AZ_NET_PAIR_TILES": "2"},
    "pair1": {"AZ_NET_PAIR_TILES": "1"},
}


def _with_env(env, fn):
    """runs fn(ctx) in a fresh context whose weights are loaded under `env` (the kernel choice is read when weights load)"""
    import ataxxzero_b200 as az
    saved = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        with az.Context(0) as c:
            return fn(c)
    finally:
        for k, v in saved.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def _pool_forward():
    """az_net_forward_pool_dev: the call the self-play pool makes (az_pool.cu launch_net); a test hook, not in the header"""
    from ataxxzero_b200 import _native
    fn = _native.lib().az_net_forward_pool_dev
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5
    return fn


def _dp(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _debug_exp(ctx, x):
    """the tree kernel's own exp_d (az_tree.cu) of every float in x, as float64"""
    from ataxxzero_b200 import _native
    lib = _native.lib()
    lib.az_debug_exp.restype = C.c_int
    lib.az_debug_exp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    x = np.ascontiguousarray(x, dtype=np.float32).reshape(-1)
    out = np.empty((len(x), 2), np.float64)
    _native.check(lib.az_debug_exp(ctx.handle, C.c_void_p(x.ctypes.data), len(x), C.c_void_p(out.ctypes.data)))
    return out[:, 1]


@pytest.fixture(scope="module")
def sms():
    """The SM count the library sizes its launches with (ctx->sm_count comes from the same device property)."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def network():
    from ataxxzero_b200 import model
    from oracle import net_numpy
    nw = model.Network.random_init(seed=0)
    nw.bn = net_numpy.randomize_bn(nw.bn, seed=1)
    return nw


@pytest.fixture(scope="module")
def oracle64(network, positions):
    return Oracle64(network, positions[1])


@pytest.fixture(scope="module")
def sym_oracle():
    return {}


@pytest.fixture(scope="module")
def trained():
    from ataxxzero_b200 import model
    from oracle import net_numpy
    return model.Network(*net_numpy.trained_scale_weights(seed=0, logit_std=2.0))


WALK_STARTS = [
    "x5o/7/3-3/2-1-2/3-3/7/o5x x",           # the C++ start position
    "x5o/7/3-3/2-1-2/3-3/7/o5x o",           # ... with o to move
    "x5o/7/7/7/7/7/o5x x",                   # no blockers
    "x-1o3/--5/7/7/7/7/7 x",                 # blockers next to x
    "-1-1-1-/x5o/-1-1-1-/7/-1-1-1-/o5x/-1-1-1- o",     # many blockers
]


@pytest.fixture(scope="module")
def positions(ctx, oracle, sms):
    """(az_position structured array, oracle feature planes [N,7,7,4]) for N = max(2048, 6S + 5) positions: every position
    of random walks from WALK_STARTS to the end of the game, shuffled, with the edge positions of test_rules_gpu in front"""
    from ataxxzero_b200 import rules
    from test_rules_gpu import EDGE_FENS
    need = max(2048, 6 * sms + 5)
    rng = np.random.default_rng(2024)
    walked = []
    for walk in range(10 ** 6):
        if len(walked) >= 8 * need:
            break
        p = oracle.set_board(WALK_STARTS[walk % len(WALK_STARTS)])
        walked.append(p)
        for _ in range(400):
            moves = oracle.movegen(p)
            if oracle.result(p) != 0 or not moves:
                break
            p = oracle.makemove(p, moves[rng.integers(len(moves))])
            walked.append(p)
    order = rng.permutation(len(walked))[:need - len(EDGE_FENS)]
    pos = [oracle.set_board(f) for f in EDGE_FENS] + [walked[i] for i in order]
    arr = rules.positions_array(pos)
    assert set(arr["turn"]) == {0, 1} and (arr["blockers"] != 0).mean() > 0.3
    assert (arr["ply"] > 60).sum() > need // 4                     # late endgames
    planes = np.stack([oracle.features(p) for p in pos]).astype(np.float32)
    assert planes[..., 3].any() and np.array_equal(planes, rules.features_batch(ctx, arr))
    return arr, planes


def _device_positions(arr):
    import torch
    return torch.from_numpy(arr.view(np.uint8).copy()).cuda()


def _sample(n, rng, k=6):
    """the boards of a batch of n compared with the fp64 oracle: head, tail, and k random rows"""
    return np.unique(np.concatenate([np.arange(min(n, k)), np.arange(max(n - k, 0), n), rng.integers(0, n, k)]))


class Oracle64:
    """fp64 restatement outputs per board index, computed once per network and board"""

    def __init__(self, nw, planes):
        self.nw, self.planes, self.p, self.v = nw, planes, {}, {}

    def get(self, idx):
        from oracle import net_numpy
        todo = [int(i) for i in idx if int(i) not in self.p]
        if todo:
            p, v = net_numpy.forward(self.planes[todo], self.nw.conv, self.nw.bn, dtype=np.float64)
            for j, i in enumerate(todo):
                self.p[i], self.v[i] = p[j], v[j]
        return np.stack([self.p[int(i)] for i in idx]), np.stack([self.v[int(i)] for i in idx])


def _within(mode, got_p, got_v, want_p, want_v, worst):
    from ataxxzero_b200 import net
    tol = {net.FP32: FP32_TOL, net.BF16: BF16_TOL, net.F16: F16_TOL}[mode]
    ep, ev = float(np.abs(got_p - want_p).max()), float(np.abs(got_v - want_v).max())
    worst[mode] = max(worst.get(mode, (0, 0))[0], ep), max(worst.get(mode, (0, 0))[1], ev)
    assert ep < tol and ev < tol, (mode, ep, ev)


def _trained_within(mode, got_p, got_v, want_p, want_v, label):
    from ataxxzero_b200 import net
    full = float(np.abs(want_p).max())
    assert full > 2.0                                                  # the regime the bounds are about
    err = np.abs(got_p - want_p)
    ev = float(np.abs(got_v - want_v).max())
    print("%s mode %d: logits max %.3e (%.2f %% of %.2f), rms %.2f %% of std, values %.3e" % (
        label, mode, err.max(), 100 * err.max() / full, full, 100 * np.sqrt((err ** 2).mean()) / want_p.std(), ev))
    if mode == net.BF16:
        assert err.max() < 0.03 * full and np.sqrt((err ** 2).mean()) < 0.025 * want_p.std() and ev < 0.15
    elif mode == net.F16:
        assert err.max() < BF16_TOL and ev < BF16_TOL
    else:
        assert err.max() < FP32_TOL * max(full, 1.0) and ev < 5 * FP32_TOL


# ------------------------------------------------------------------------------------------------------------------------
# 1. position input
# ------------------------------------------------------------------------------------------------------------------------
def _run_pos(c, d_pos, n, mode, count=None, tiles=0):
    import torch
    logits = torch.full((n, 833), SENTINEL, device="cuda")
    values = torch.full((n,), SENTINEL, device="cuda")
    d_count = None if count is None else torch.tensor([count], dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()            # the fills run on torch's stream, the net on the context's own non-blocking stream
    from ataxxzero_b200 import _native
    _native.check(_pool_forward()(c.handle, _dp(d_pos), n, _dp(d_count), mode, tiles, _dp(logits), _dp(values), None, None, None))
    c.sync()
    return logits.cpu().numpy().reshape(n, 7, 7, 17), values.cpu().numpy()


@pytest.mark.parametrize("variant", list(POS_VARIANTS))
def test_position_input_matches_planes(variant, network, positions, oracle64, sms):
    """az_position[] in, the net encodes the planes itself (AZ_IN_POS): bit for bit the plain pass on the oracle's planes,
    within the fp64 bounds, and with the count read from device memory it computes the rows below it and writes none past it"""
    from ataxxzero_b200 import net
    arr, planes = positions
    R = 4 * sms
    sizes = (1, 7, R - 1, R, R + 1, 3 * R, 2048)
    counted = ((2048, 1777), (3 * R, 2 * R + 3), (7, 1))
    worst = {}

    def run(c):
        net.load_weights(c, network)
        d_pos = _device_positions(arr)
        for n in sizes:
            idx = _sample(n, np.random.default_rng(n))
            want_p, want_v = oracle64.get(idx)
            for mode in (net.FP32, net.BF16, net.F16):
                got_p, got_v = _run_pos(c, d_pos, n, mode)
                ref_p, ref_v = net.forward(c, planes[:n], mode)
                assert np.array_equal(got_p, ref_p) and np.array_equal(got_v, ref_v[:, 0]), (variant, n, mode)
                _within(mode, got_p[idx], got_v[idx], want_p, want_v[:, 0], worst)
                for cn, count in counted:
                    if cn != n:
                        continue
                    cp, cv = _run_pos(c, d_pos, n, mode, count=count)
                    assert (cp[count:] == SENTINEL).all() and (cv[count:] == SENTINEL).all(), (variant, n, count, mode)
                    assert np.array_equal(cp[:count], got_p[:count]) and np.array_equal(cv[:count], got_v[:count]), (variant, n, count, mode)
    _with_env(POS_VARIANTS[variant], run)
    print("position input %s: max |err| vs fp64 (logits, values) per mode: %r" % (variant, worst))


def test_position_input_at_trained_scale(trained, positions, sms):
    from ataxxzero_b200 import net
    arr, planes = positions
    n = 4 * sms + 1
    idx = _sample(n, np.random.default_rng(12), k=12)
    want_p, want_v = Oracle64(trained, planes).get(idx)

    def run(c):
        net.load_weights(c, trained)
        d_pos = _device_positions(arr)
        for mode in (net.FP32, net.BF16, net.F16):
            got_p, got_v = _run_pos(c, d_pos, n, mode)
            ref_p, ref_v = net.forward(c, planes[:n], mode)
            assert np.array_equal(got_p, ref_p) and np.array_equal(got_v, ref_v[:, 0]), mode
            _trained_within(mode, got_p[idx], got_v[idx], want_p, want_v[:, 0], "position input, trained scale")
    _with_env({}, run)


# ------------------------------------------------------------------------------------------------------------------------
# 2. the speculative cache pass
# ------------------------------------------------------------------------------------------------------------------------
def _check_cache_pass(c, arr, planes, n, count, mode, tiles, rng):
    """one cache pass of n requests, count of them live, scattered through a random injective map into a 2n + 1 row table
    whose last row is the trash row (about 5 % of the requests point there, as dropped requests do)"""
    import torch
    from ataxxzero_b200 import _native, net
    rows = 2 * n + 1
    trash = 2 * n
    out_map = rng.permutation(2 * n)[:n].astype(np.int32)
    drop = rng.random(n) < 0.05
    if n >= 3:
        drop[n // 2] = True
    out_map[drop] = trash
    d_pos = _device_positions(arr[:n])
    d_map = torch.from_numpy(out_map).cuda()
    d_count = torch.tensor([count], dtype=torch.int32, device="cuda")
    exps = torch.full((rows, 833), SENTINEL, dtype=torch.float64, device="cuda")
    totals = torch.full((rows,), SENTINEL, dtype=torch.float64, device="cuda")
    values = torch.full((rows,), SENTINEL, device="cuda")
    torch.cuda.synchronize()
    _native.check(_pool_forward()(c.handle, _dp(d_pos), n, _dp(d_count), mode, tiles, None, _dp(values), _dp(exps), _dp(totals),
                                  _dp(d_map)))
    c.sync()
    exps, totals, values = exps.cpu().numpy(), totals.cpu().numpy(), values.cpu().numpy()
    ref_p, ref_v = net.forward(c, planes[:n], mode)
    live = np.arange(count)
    kept = live[out_map[live] != trash]
    m = out_map[kept]
    key = (n, count, mode, tiles)
    assert np.array_equal(values[m], ref_v[kept, 0]), key
    want_e = _debug_exp(c, ref_p[kept].reshape(len(kept), 833)).reshape(len(kept), 833) if len(kept) else np.zeros((0, 833))
    assert np.array_equal(exps[m].view(np.uint64), want_e.view(np.uint64)), key
    # the reference's `total += exp(...)` over i = 0..832, strictly in order (np.cumsum adds one term at a time)
    want_t = np.cumsum(exps[m], axis=1)[:, -1] if len(m) else np.zeros(0)
    assert np.array_equal(totals[m].view(np.uint64), want_t.view(np.uint64)), key
    untouched = np.ones(rows, bool)
    untouched[out_map[live]] = False
    assert (values[untouched] == SENTINEL).all() and (totals[untouched] == SENTINEL).all(), key
    assert (exps[untouched] == SENTINEL).all(), key
    return int(drop[:count].sum())


CACHE_SIZES = ("1", "3", "R-1", "R+1", "2R+3")


@pytest.mark.parametrize("size", CACHE_SIZES)
def test_speculative_cache_pass(size, network, positions, sms):
    """values, softmax numerators and their sequential totals scattered through out_map: bit for bit the plain pass's values,
    the tree kernel's exp_d of its logits, and the host's in-order float64 sum; rows no live request maps to keep their
    sentinel.  At 2R + 3 boards every CTA sums a second unit in its helper warp while its epilogue runs the next one."""
    from ataxxzero_b200 import net
    arr, planes = positions
    R = 4 * sms
    n = {"1": 1, "3": 3, "R-1": R - 1, "R+1": R + 1, "2R+3": 2 * R + 3}[size]
    rng = np.random.default_rng(13 + n)

    def run(c):
        import torch
        import ataxxzero_b200 as az
        from ataxxzero_b200 import _native
        net.load_weights(c, network)
        dropped = 0
        for count in ((n, n - 2) if n > 2 else (n,)):
            for mode in (net.BF16, net.F16):
                dropped += _check_cache_pass(c, arr, planes, n, count, mode, 1, rng)
        assert dropped > 0 or n < 3             # from 3 requests on, one of them always points at the trash row
        d_pos = _device_positions(arr[:4])
        buf = torch.zeros(16 * 833, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        with pytest.raises(az.AzError):          # FP32 has no softmax numerators
            _native.check(_pool_forward()(c.handle, _dp(d_pos), 4, None, net.FP32, 1, None, _dp(buf), _dp(buf), _dp(buf), None))
    _with_env({}, run)


def test_speculative_cache_pass_at_trained_scale(trained, positions, sms):
    from ataxxzero_b200 import net
    arr, planes = positions

    def run(c):
        net.load_weights(c, trained)
        n = 4 * sms + 1
        for mode in (net.BF16, net.F16):
            _check_cache_pass(c, arr, planes, n, n - 2, mode, 2, np.random.default_rng(14))
    _with_env({}, run)


# ------------------------------------------------------------------------------------------------------------------------
# 3. the symmetry ensemble
# ------------------------------------------------------------------------------------------------------------------------
def _sym(t, s):
    """net.apply_symmetry on axes 1 and 2 of a batch"""
    if s & 1:
        t = t[:, ::-1, :]
    if s & 2:
        t = t[:, :, ::-1]
    if s & 4:
        t = np.swapaxes(t, 1, 2)
    return t


def _sym8_reference(c, planes, mode):
    """the 8 images through one plain forward, each undone, then the kernels' order: policy summed image by image 0..7,
    value ((v0+v1)+(v2+v3))+((v4+v5)+(v6+v7)), both times 0.125, in float32"""
    from ataxxzero_b200 import net
    n = len(planes)
    images = np.stack([np.ascontiguousarray(_sym(planes, s)) for s in range(8)], axis=1)
    p8, v8 = net.forward(c, images.reshape(8 * n, 7, 7, 4), mode)
    p8, v = p8.reshape(n, 8, 7, 7, 17), v8.reshape(n, 8)
    acc = np.ascontiguousarray(_sym(p8[:, 0], net.inverse_symmetry[0]))
    for s in range(1, 8):
        acc = acc + _sym(p8[:, s], net.inverse_symmetry[s])
    pv = ((v[:, 0] + v[:, 1]) + (v[:, 2] + v[:, 3])) + ((v[:, 4] + v[:, 5]) + (v[:, 6] + v[:, 7]))
    return acc * np.float32(0.125), pv * np.float32(0.125)


def _sym8_oracle(nw, planes, idx):
    from ataxxzero_b200 import net
    from oracle import net_numpy
    images = np.stack([np.ascontiguousarray(net.apply_symmetry(planes[b], s)) for b in idx for s in range(8)])
    w8, wv8 = net_numpy.forward(images, nw.conv, nw.bn, dtype=np.float64)
    w8, wv8 = w8.reshape(len(idx), 8, 7, 7, 17), wv8.reshape(len(idx), 8)
    want = np.stack([np.mean([net.apply_symmetry(w8[j, s], net.inverse_symmetry[s]) for s in range(8)], axis=0)
                     for j in range(len(idx))])
    return want, wv8.mean(axis=1)


SYM_SIZES = ("1", "2", "2S-1", "2S+1", "6S+5")


@pytest.mark.parametrize("size", SYM_SIZES)
@pytest.mark.parametrize("mode_name", ("BF16", "F16", "FP32"))
def test_symmetry_ensemble(mode_name, size, network, positions, sym_oracle, sms):
    """az_net_forward_sym8 bit for bit against its definition over the plain pass, and within the fp64 bounds of the ensemble
    mean.  The 2S one-tile CTAs each evaluate one position at a time: one CTA of the only pair has no position (1), both have
    one (2), the last pair has one CTA without a position (2S - 1), CTAs evaluate one or two (2S + 1) and up to four (6S + 5)."""
    from ataxxzero_b200 import net
    mode = getattr(net, mode_name)
    run_id = "%s-%s" % (mode_name, size)
    arr, planes = positions
    n = {"1": 1, "2": 2, "2S-1": 2 * sms - 1, "2S+1": 2 * sms + 1, "6S+5": 6 * sms + 5}[size]
    ora_idx = np.unique([0, n // 2, n - 1])
    if n not in sym_oracle:
        sym_oracle[n] = _sym8_oracle(network, planes, ora_idx)
    want_p, want_v = sym_oracle[n]
    worst = {}

    def run(c):
        net.load_weights(c, network)
        got_p, got_v = net.evaluate_symmetric(c, planes[:n], mode)
        ref_p, ref_v = _sym8_reference(c, planes[:n], mode)
        bad = np.nonzero(~((got_p == ref_p).all(axis=(1, 2, 3)) & (got_v == ref_v)))[0]
        assert len(bad) == 0, (run_id, n, "positions differing from the reference", bad[:16], len(bad))
        _within(mode, got_p[ora_idx], got_v[ora_idx], want_p, want_v, worst)
    _with_env({}, run)
    print("symmetry ensemble %s: max |err| vs fp64 (logits, values): %r" % (run_id, worst))


def test_symmetry_ensemble_at_trained_scale(trained, positions, sms):
    from ataxxzero_b200 import net
    arr, planes = positions
    n = 2 * sms + 1
    idx = np.array([0, 1, n // 2, n - 1])
    want_p, want_v = _sym8_oracle(trained, planes, idx)

    def run(c):
        net.load_weights(c, trained)
        got_p, got_v = net.evaluate_symmetric(c, planes[:n], net.BF16)
        ref_p, ref_v = _sym8_reference(c, planes[:n], net.BF16)
        assert np.array_equal(got_p, ref_p) and np.array_equal(got_v, ref_v)
        _trained_within(net.BF16, got_p[idx], got_v[idx], want_p, want_v, "symmetry ensemble, trained scale")
    _with_env({}, run)
