"""The two-tile CTA-pair net kernel (k_net_pair<2>, the default for batches of a full round) against the one-tile kernel
(k_net_pair<1>) and the single-CTA kernel (k_net_tc): same operand images, same chunk order, fp32 accumulation per tile, so the
outputs must be identical bit for bit -- at every batch size, with the board count read from device memory as the self-play pool
launches it, and over a whole capped self-play run."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VARIANTS = ({"AZ_NET_PAIR_TILES": "2"}, {"AZ_NET_PAIR_TILES": "1"}, {"AZ_NET_PAIR": "0"})


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


@pytest.fixture(scope="module")
def network():
    from ataxxzero_b200 import model
    from oracle import net_numpy
    nw = model.Network.random_init(seed=0)
    nw.bn = net_numpy.randomize_bn(nw.bn, seed=1)
    return nw


def test_tiles_agree_bitwise_across_batch_sizes(network):
    from ataxxzero_b200 import net
    from oracle import net_numpy
    sizes = (1, 7, 592, 1776, 2048)
    feats = {n: net_numpy.random_features(n, seed=100 + n) for n in sizes}

    def run(c):
        net.load_weights(c, network)
        return {(n, m): net.forward(c, feats[n], m) for n in sizes for m in (net.BF16, net.F16)}
    outs = [_with_env(env, run) for env in VARIANTS]
    for key in outs[0]:
        for other in outs[1:]:
            assert np.array_equal(outs[0][key][0], other[key][0]) and np.array_equal(outs[0][key][1], other[key][1]), key


def test_tiles_agree_with_device_count(network):
    """n = the request buffer, the kernel reads min(*d_count, n) when it starts: the two-tile kernel (chosen by n) serves
    counts that are not a multiple of its 8-board pair unit exactly like the others, and writes nothing past the count"""
    import torch
    from ataxxzero_b200 import _native, net
    from oracle import net_numpy
    lib = _native.lib()
    fn = lib.az_net_forward_counted_dev
    fn.restype, fn.argtypes = C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    n = 1776
    feats = torch.from_numpy(net_numpy.random_features(n, seed=7).reshape(n, 196).copy()).cuda()
    counts = (1776, 1775, 1001, 600, 13, 1)

    def run(c):
        net.load_weights(c, network)
        res = {}
        for count in counts:
            for mode in (net.BF16, net.F16):
                d_count = torch.tensor([count], dtype=torch.int32, device="cuda")
                logits = torch.full((n, 833), -7.0, device="cuda")
                values = torch.full((n,), -7.0, device="cuda")
                torch.cuda.synchronize()          # the fills run on torch's stream, the net on the context's non-blocking stream
                _native.check(fn(c.handle, C.c_void_p(feats.data_ptr()), n, C.c_void_p(d_count.data_ptr()), mode,
                                 C.c_void_p(logits.data_ptr()), C.c_void_p(values.data_ptr())))
                c.sync()
                res[(count, mode)] = (logits.cpu().numpy(), values.cpu().numpy())
        return res
    outs = [_with_env(env, run) for env in VARIANTS]
    for (count, mode), (lg, v) in outs[0].items():
        assert (lg[count:] == -7.0).all() and (v[count:] == -7.0).all(), (count, mode)
        for other in outs[1:]:
            assert np.array_equal(lg, other[(count, mode)][0]) and np.array_equal(v, other[(count, mode)][1]), (count, mode)


def test_capped_selfplay_identical_across_tiles():
    """a capped 512-game self-play pool, a few hundred ticks under each kernel: every root and counter bit for bit"""
    from ataxxzero_b200 import model, search

    def run(c):
        from ataxxzero_b200 import net
        net.load_weights(c, model.Network.random_init(seed=0))
        with search.Pool(c, 512, 64, eval_mode=search.EVAL_BF16, noise=True, auto_play=True, seed=5) as pool:
            st = pool.selfplay_ticks(300)
            return st, [pool.root(g) for g in range(512)]
    # AZ_REQ_CAP is read when the pool is created: far fewer than the 512 games request, so requests are deferred
    runs = [_with_env(dict(env, AZ_REQ_CAP="160"), run) for env in VARIANTS]
    sa, ra = runs[0]
    assert sa["positions"] > 0
    for sb, rb in runs[1:]:
        for key in ("ticks", "steps", "evals", "terminal_steps", "positions", "games_finished", "max_depth", "levels"):
            assert sa[key] == sb[key], key
        for x, y in zip(ra, rb):
            assert x["position"].key() == y["position"].key() and x["position"].ply == y["position"].ply
            assert x["moves"] == y["moves"] and x["visits"] == y["visits"] and x["root_visits"] == y["root_visits"]
            assert [float(v).hex() for v in x["total_score"]] == [float(v).hex() for v in y["total_score"]]
            assert [float(v).hex() for v in x["prior"]] == [float(v).hex() for v in y["prior"]]
