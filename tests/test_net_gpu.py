"""GPU parity of the network forward pass (through the C ABI) against the NumPy restatement of
model.py (oracle/net_numpy.py).  Tolerances are north_star's: 1e-5 in fp32 mode, 2e-2 abs in bf16."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2


@pytest.fixture(scope="module")
def nets(ctx):
    from ataxxzero_b200 import model, net
    from oracle import net_numpy
    network = model.Network.random_init(seed=0)
    network.bn = net_numpy.randomize_bn(network.bn, seed=1)      # exercise the BN folding
    net.load_weights(ctx, network)
    return network


def _features(n, seed):
    from oracle import net_numpy
    return net_numpy.random_features(n, seed=seed)


def test_fp32_mode_matches_restatement(ctx, nets):
    from ataxxzero_b200 import net
    from oracle import net_numpy
    feats = _features(37, 3)                       # odd count: exercises a half-empty CTA
    want_p, want_v = net_numpy.forward(feats, nets.conv, nets.bn, dtype=np.float64)
    got_p, got_v = net.forward(ctx, feats, net.FP32)
    assert got_p.shape == (37, 7, 7, 17) and got_v.shape == (37, 1)
    assert np.abs(got_p - want_p).max() < FP32_TOL
    assert np.abs(got_v - want_v).max() < FP32_TOL
    # and against the fp32 restatement (what TF itself would have computed in)
    p32, v32 = net_numpy.forward(feats[:8], nets.conv, nets.bn, dtype=np.float32)
    assert np.abs(got_p[:8] - p32).max() < FP32_TOL
    assert np.abs(got_v[:8] - v32).max() < FP32_TOL


def test_tc_tower_layer_by_layer(ctx, nets):
    """Debug hook: the tensor-core tower after 1, 2, 3 and all conv layers against the restatement
    evaluated with the same bf16-rounded, BN-folded operands (tight) -- localises layout bugs."""
    import ctypes as C
    from ataxxzero_b200 import _native
    from oracle import net_numpy
    lib = _native.lib()
    lib.az_net_debug_tower.restype = C.c_int
    lib.az_net_debug_tower.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    feats = _features(6, 5)
    for layers in (1, 2, 3, 5, 25):
        out = np.zeros((6, 49, 128), dtype=np.float32)
        _native.check(lib.az_net_debug_tower(ctx.handle, C.c_void_p(feats.ctypes.data), 6, layers,
                                             C.c_void_p(out.ctypes.data)))
        want = tower_reference(feats, nets, layers)
        err = np.abs(out.reshape(6, 7, 7, 128) - want).max()
        scale = np.abs(want).max()
        assert err < 3e-2 * max(scale, 1.0), "after %d conv layers: max err %g (scale %g)" % (layers, err, scale)


def tower_reference(feats, nets, layers):
    """fp64 tower with bf16-rounded folded weights and bf16-rounded activations between layers."""
    import torch
    from oracle import net_numpy

    def bf16(a):
        return torch.from_numpy(np.asarray(a, dtype=np.float32)).to(torch.bfloat16).to(torch.float64).numpy()

    x = bf16(feats)
    res = None
    for l in range(layers):
        w = np.asarray(nets.conv[l], dtype=np.float64)
        scale = 1.0 / np.sqrt(np.asarray(nets.bn[2 * l + 1], dtype=np.float64) + 1e-3)
        shift = -np.asarray(nets.bn[2 * l], dtype=np.float64) * scale
        wq = bf16((w * scale).astype(np.float32))
        y = net_numpy._conv_same(x, wq) + shift.astype(np.float32).astype(np.float64)
        second = l > 0 and l % 2 == 0
        if second:
            y = y + res
        y = np.maximum(y, 0)
        if l == 0 or second:
            res = y.astype(np.float32).astype(np.float64)
        out = y
        x = bf16(y.astype(np.float32))
    return out


def test_bf16_mode_within_tolerance(ctx, nets):
    from ataxxzero_b200 import net
    from oracle import net_numpy
    feats = _features(301, 7)                      # many units, ragged tail
    want_p, want_v = net_numpy.forward(feats, nets.conv, nets.bn, dtype=np.float64)
    got_p, got_v = net.forward(ctx, feats, net.BF16)
    assert np.isfinite(got_p).all() and np.isfinite(got_v).all()
    assert np.abs(got_p - want_p).max() < BF16_TOL
    assert np.abs(got_v - want_v).max() < BF16_TOL


def test_bf16_at_trained_scale(ctx, nets):
    """Calibrated batch-norm statistics, logits of standard deviation 2 (|logit| up to ~9), saturating values: the regime
    of a TRAINED net, where the random-init tests above are loose.  An 8-bit mantissa cannot hold north_star's 2e-2
    absolute on logits of magnitude 9: every operand is rounded to 2^-9 relative, ~50 roundings deep, and the measured
    error is what that predicts -- 1.4 % rms of the logit scale, growing as sqrt(depth) (profiles/r02_net_error.txt, per
    layer).  So at this scale the bf16 bound is RELATIVE (the absolute 2e-2 is kept for logits of the benchmark's scale,
    test_bf16_mode_within_tolerance); the fp16-operand mode (test_f16_mode_keeps_2e2_at_trained_scale) keeps 2e-2
    absolute here, and the fp32 mode keeps 1e-5 of full scale (float32 itself is 1e-5 from fp64 at this magnitude)."""
    from ataxxzero_b200 import model, net
    from oracle import net_numpy
    conv, bn = net_numpy.trained_scale_weights(seed=0, logit_std=2.0)
    net.load_weights(ctx, model.Network(conv, bn))
    try:
        feats = _features(24, 21)
        want_p, want_v = net_numpy.forward(feats, conv, bn, dtype=np.float64)
        full = np.abs(want_p).max()
        assert full > 5.0 and np.abs(want_v).max() > 0.99            # the regime the test is about
        got_p, got_v = net.forward(ctx, feats, net.BF16)
        err = np.abs(got_p - want_p)
        assert err.max() < 0.03 * full                                # measured 1.5 %
        assert np.sqrt((err ** 2).mean()) < 0.025 * want_p.std()      # measured 1.4 %
        assert np.abs(got_v - want_v).max() < 0.15                    # measured 0.08 (where tanh is steep)
        # the priors the search actually consumes: softmax over the legal-move-sized logit vector moves by a few percent
        sm = lambda z: np.exp(z - z.max(axis=(1, 2, 3), keepdims=True)) / np.exp(z - z.max(axis=(1, 2, 3), keepdims=True)).sum(axis=(1, 2, 3), keepdims=True)
        assert np.abs(sm(got_p.astype(np.float64)) - sm(want_p)).max() < 0.02
        p32, v32 = net.forward(ctx, feats, net.FP32)
        assert np.abs(p32 - want_p).max() < FP32_TOL * max(full, 1.0) and np.abs(v32 - want_v).max() < 5 * FP32_TOL
    finally:
        net.load_weights(ctx, nets)


def test_f16_mode_keeps_2e2_at_trained_scale(ctx, nets):
    """AZ_NET_F16: same tcgen05 kernel, IEEE-half operands (11-bit mantissa).  north_star's 2e-2 absolute holds for
    trained-scale logits (|logit| up to ~9) and saturating values, and at the benchmark's scale the error drops ~8x."""
    from ataxxzero_b200 import model, net
    from oracle import net_numpy
    conv, bn = net_numpy.trained_scale_weights(seed=0, logit_std=2.0)
    net.load_weights(ctx, model.Network(conv, bn))
    try:
        feats = _features(24, 21)
        want_p, want_v = net_numpy.forward(feats, conv, bn, dtype=np.float64)
        got_p, got_v = net.forward(ctx, feats, net.F16)
        assert np.isfinite(got_p).all() and np.isfinite(got_v).all()
        assert np.abs(got_p - want_p).max() < BF16_TOL
        assert np.abs(got_v - want_v).max() < BF16_TOL
        bp, _ = net.forward(ctx, feats, net.BF16)
        assert np.abs(got_p - want_p).max() < 0.25 * np.abs(bp - want_p).max()
    finally:
        net.load_weights(ctx, nets)
    feats = _features(64, 23)
    want_p, want_v = net_numpy.forward(feats, nets.conv, nets.bn, dtype=np.float64)
    got_p, got_v = net.forward(ctx, feats, net.F16)
    assert np.abs(got_p - want_p).max() < 3e-4 and np.abs(got_v - want_v).max() < 3e-4
    # and a search pool can run on it
    from ataxxzero_b200 import rules, search
    with search.Pool(ctx, 2, 40, eval_mode=search.EVAL_F16) as pool:
        pool.run()
        assert pool.root(0)["root_visits"] >= 40


def test_modes_agree_and_batch_invariance(ctx, nets):
    from ataxxzero_b200 import net
    feats = _features(64, 9)
    p_all, v_all = net.forward(ctx, feats, net.BF16)
    p_one, v_one = net.forward(ctx, feats[17:18], net.BF16)
    assert np.array_equal(p_all[17:18], p_one) and np.array_equal(v_all[17:18], v_one)   # position in batch is irrelevant
    p32, v32 = net.forward(ctx, feats, net.FP32)
    assert np.abs(p_all - p32).max() < BF16_TOL and np.abs(v_all - v32).max() < BF16_TOL


def test_int8_wire_format_and_rpc_contract(ctx, nets):
    from ataxxzero_b200 import net
    feats = _features(5, 11)
    p_f, v_f = net.forward(ctx, feats, net.FP32)
    p_i, v_i = net.forward(ctx, feats.astype(np.int8), net.FP32)
    assert np.array_equal(p_f, p_i) and np.array_equal(v_f, v_i)
    blob, value = net.network_rpc(ctx, feats[0].astype(np.int8).tobytes(), net.FP32)
    assert len(blob) == 3332 and isinstance(value, float)            # gpu_server.py:52-56
    assert np.array_equal(np.frombuffer(blob, dtype=np.float32).reshape(7, 7, 17), p_f[0])


def test_weight_file_roundtrip(tmp_path, ctx, nets):
    """model.py:179-196 layout: a saved file reloads to identical outputs."""
    from ataxxzero_b200 import model, net
    path = str(tmp_path / "model-001.npy")
    nets.save(path)
    raw = np.load(path, allow_pickle=True)
    assert raw.shape == (2,) and len(raw[0]) == 29 and len(raw[1]) == 50
    again = model.Network.load(path)
    feats = _features(4, 13)
    a = net.forward(ctx, feats, net.FP32)
    net.load_weights(ctx, again)
    b = net.forward(ctx, feats, net.FP32)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    net.load_weights(ctx, nets)


def test_errors(ctx, nets):
    import ataxxzero_b200 as az
    from ataxxzero_b200 import net
    with pytest.raises(az.AzError):
        net.forward(ctx, np.zeros((2, 7, 7, 3), dtype=np.float32))
    with pytest.raises(az.AzError):
        net.forward(ctx, _features(2, 1), mode=7)
    with az.Context(0) as fresh:
        with pytest.raises(az.AzError):
            net.forward(fresh, _features(2, 1))      # no weights loaded


def test_symmetry_ensembled_evaluation(ctx, nets):
    """nn_evals.evaluate (nn_evals.py:48-62): the GPU expand / reduce kernels against the NumPy composition of the same
    steps over our own forward pass (exact up to float32 summation order), and against the fp64 restatement."""
    from ataxxzero_b200 import net
    from oracle import net_numpy
    feats = _features(5, 9)
    for mode, tol in ((net.FP32, FP32_TOL), (net.BF16, BF16_TOL)):
        got_p, got_v = net.evaluate_symmetric(ctx, feats, mode)
        assert got_p.shape == (5, 7, 7, 17) and got_v.shape == (5,)
        for b in range(5):
            images = np.stack([np.ascontiguousarray(net.apply_symmetry(feats[b], s)) for s in range(8)])
            p8, v8 = net.forward(ctx, images, mode)
            back = [net.apply_symmetry(p8[s], net.inverse_symmetry[s]) for s in range(8)]
            assert np.abs(got_p[b] - np.mean(back, axis=0)).max() < 1e-6
            assert abs(got_v[b] - np.mean(v8)) < 1e-6
            w8, wv8 = net_numpy.forward(images, nets.conv, nets.bn, dtype=np.float64)
            want = np.mean([net.apply_symmetry(w8[s], net.inverse_symmetry[s]) for s in range(8)], axis=0)
            assert np.abs(got_p[b] - want).max() < tol and abs(got_v[b] - np.mean(wv8)) < tol
    p0, v0 = net.evaluate_symmetric(ctx, np.zeros((0, 7, 7, 4), dtype=np.float32))
    assert len(p0) == 0 and len(v0) == 0
