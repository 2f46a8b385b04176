"""The hand-written training step (csrc/az_train.cu behind ataxxzero_b200/trainer.py) against the fp32 PyTorch restatement of
the reference's training graph (tests/torch_train_reference.py; model.py:35-101).

Operands are bf16 (8 mantissa bits) with fp32 accumulation, so the comparison is by tolerance, stated per quantity:
  * forward conv outputs / activations: relative L2 error <= 2e-2 per layer (measured 2e-3 .. 6e-3 over 5 layers);
  * losses of the step: |policy| <= 2e-3, |value| <= 5e-3, regularisation relative 1e-5 (fp32 either side);
  * gradients: cosine similarity >= 0.98 and norm ratio within 3 % per tensor.  At random init with random targets a weight
    gradient is a sum of ~n*49 terms of mixed sign that cancels to ~1/50 of its terms' size, which amplifies the operands'
    0.4 % rounding to a few percent of the (small) sum: measured 5..9 % relative L2 error = cosine 0.996.  The yardstick is
    measured in the same test: PyTorch's own bf16 autocast differs from its fp32 gradients by 6..11 % on these tensors, and
    every weight gradient of ours must be no further from fp32 than 1.25 x that;
  * 30 optimiser steps on a fixed batch: the loss trajectory follows PyTorch's within 2e-3 at every step.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def synthetic_batch(n, seed):
    rng = np.random.default_rng(seed)
    feats = np.zeros((n, 7, 7, 4), np.int8)
    feats[..., 0] = 1
    who = rng.integers(0, 3, size=(n, 7, 7))
    feats[..., 1] = who == 1
    feats[..., 2] = who == 2
    pol = rng.random((n, 7, 7, 17)).astype(np.float32) ** 8
    pol /= pol.reshape(n, -1).sum(1).reshape(n, 1, 1, 1)
    val = rng.choice([-1.0, 1.0], size=(n, 1)).astype(np.float32)
    return feats, pol, val


def rel(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def cosine(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(a @ b / max(np.linalg.norm(a) * np.linalg.norm(b), 1e-30))


def torch_setup(network, blocks, lr):
    import torch
    import torch_train_reference as ref
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    net = ref.build_torch_network(128, blocks).to(dev)
    ref.load_into(net, network)
    net.train()
    return ref, net, torch.optim.SGD(net.parameters(), lr=lr, momentum=0.9), dev


@pytest.mark.parametrize("blocks,n", [(2, 64), (1, 37), (0, 2)])
def test_one_step_matches_fp32_restatement(ctx, blocks, n):
    """Forward tensors, the three loss terms, every gradient tensor and the updated weights of ONE step; n = 37 leaves half a
    tile empty (odd batch) and leaves the weight-gradient kernel fewer tiles than ranges; (0, 2) is the smallest legal call: a
    tower of the input conv alone, a batch of two boards."""
    import torch
    from ataxxzero_b200 import model, trainer
    lr, lam = 0.01, 1e-4
    network = model.Network.random_init(seed=5, blocks=blocks)
    ref, net, opt, dev = torch_setup(network, blocks, lr)
    tr = trainer.Trainer(ctx, network, max_batch=64)
    batch = synthetic_batch(n, 1)
    x, pol, val = ref.to_torch_batch(batch, dev)
    pl, vl, reg, zs, acts = ref.loss_terms_retained(net, x, pol, val)
    opt.zero_grad()
    (pl + vl + reg).backward()

    ours = tr.train(*batch, learning_rate=lr)
    assert abs(ours[0] - float(pl)) < 2e-3 and abs(ours[1] - float(vl)) < 5e-3 and abs(ours[2] - float(reg)) < 1e-5 * float(reg) + 1e-7
    # yardstick for the gradient comparison: the SAME PyTorch graph under bf16 autocast against its own fp32 gradients, i.e.
    # what bf16 operand rounding alone does to these (heavily cancelling) sums
    import copy
    net16 = copy.deepcopy(net)
    for p_ in net16.parameters():
        p_.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16):
        p16, v16, r16, _, acts16 = ref.loss_terms_retained(net16, x, pol, val)
    (p16.float() + v16.float() + r16.float()).backward()
    layers = 1 + 2 * blocks
    for l in range(layers):
        assert rel(tr.debug_read("z", l, n), zs[l].detach().permute(0, 2, 3, 1).cpu().numpy()) < 2e-2, l
        assert rel(tr.debug_read("act", l + 1, n), acts[l].detach().permute(0, 2, 3, 1).cpu().numpy()) < 2e-2, l
    # d_h after the step: the gradient with respect to layer 0's output (heads, then every data gradient and skip on the way down)
    d_h, d_ref = tr.debug_read("d_h", 0, n), acts[0].grad.permute(0, 2, 3, 1).cpu().numpy()
    assert cosine(d_h, d_ref) > 0.98 and abs(np.linalg.norm(d_h) / np.linalg.norm(d_ref) - 1) < 0.03
    assert rel(d_h, d_ref) < 1.25 * rel(acts16[0].grad.float().permute(0, 2, 3, 1).cpu().numpy(), d_ref) + 1e-3, rel(d_h, d_ref)
    for l in range(layers):
        w = net.convs[l].weight
        g_ref = (w.grad - lam * w).detach().permute(2, 3, 1, 0).cpu().numpy()          # TF order [kx][ky][cin][cout], L2 term removed
        g = tr.debug_read("grad_conv", l)
        if l == 0:
            assert not g[:, :, 4:, :].any()                                              # padded input channels stay exactly zero
            g = g[:, :, :4, :]
        assert cosine(g, g_ref) > 0.98 and abs(np.linalg.norm(g) / np.linalg.norm(g_ref) - 1) < 0.03, l
        autocast_err = rel(net16.convs[l].weight.grad.float().cpu().numpy(), w.grad.cpu().numpy())
        assert rel(g, g_ref) < 1.25 * autocast_err + 1e-3, (l, rel(g, g_ref), autocast_err)   # no further from fp32 than PyTorch's own bf16
        for name, p in (("grad_gamma", net.bns[l].weight), ("grad_beta", net.bns[l].bias)):
            assert cosine(tr.debug_read(name, l), (p.grad - lam * p).detach().cpu().numpy()) > 0.98, (name, l)
    gh = tr.debug_read("grad_heads")
    assert rel(gh[:128 * 17].reshape(128, 17), (net.policy.weight.grad - lam * net.policy.weight).detach().reshape(17, 128).t().cpu().numpy()) < 2e-2
    assert rel(gh[128 * 17:128 * 18], (net.value.weight.grad - lam * net.value.weight).detach().reshape(128).cpu().numpy()) < 3e-2
    assert rel(gh[128 * 18:128 * 18 + 49], (net.fc_w.grad - lam * net.fc_w).detach().reshape(49).cpu().numpy()) < 3e-2
    assert rel(gh[-1:], (net.fc_b.grad - lam * net.fc_b).detach().cpu().numpy()) < 1e-2
    opt.step()
    for l in range(layers):
        w_ref = net.convs[l].weight.detach().permute(2, 3, 1, 0).cpu().numpy()
        w = tr.debug_read("conv", l)
        assert rel(w[:, :, :4, :] if l == 0 else w, w_ref) < 5e-3, l
    top = layers - 1
    mv = tr.debug_read("moving", top)                                                   # update ops: decay 0.99, unbiased variance
    assert rel(mv[0], net.bns[top].running_mean.cpu().numpy()) < 2e-2 and rel(mv[1], net.bns[top].running_var.cpu().numpy()) < 1e-3
    tr.close()


def test_fixed_batch_run_follows_fp32_trajectory_and_export_round_trips(ctx, tmp_path):
    """30 momentum steps on one batch: the loss curve follows PyTorch's; the exported .npy feeds the inference kernels, whose
    fp32 forward reproduces the trainer's eval-mode outputs when gamma = 1 / beta = 0 (fresh load, no step taken)."""
    from ataxxzero_b200 import model, net as aznet, trainer
    blocks, n, lr = 2, 64, 0.01
    network = model.Network.random_init(seed=7, blocks=blocks)
    ref, net, opt, dev = torch_setup(network, blocks, lr)
    tr = trainer.Trainer(ctx, network, max_batch=n)
    batch = synthetic_batch(n, 3)
    # eval mode before any step == the library's own inference on the same weights
    pe, ve, logits, values = tr.losses(*batch, outputs=True)
    aznet.load_weights(ctx, network)
    lg, vv = aznet.forward(ctx, batch[0].astype(np.float32), mode=aznet.FP32)
    assert np.abs(logits - lg.reshape(logits.shape)).max() < 2e-2 and np.abs(values.reshape(-1) - vv.reshape(-1)).max() < 2e-2
    xb = ref.to_torch_batch(batch, dev)
    ours, theirs = [], []
    for _ in range(30):
        lo = tr.train(*batch, learning_rate=lr)
        p2, v2, r2 = ref.loss_terms(net, *xb)
        opt.zero_grad()
        (p2 + v2 + r2).backward()
        opt.step()
        ours.append(lo[0] + lo[1])
        theirs.append(float(p2.detach() + v2.detach()))
    assert np.abs(np.array(ours) - np.array(theirs)).max() < 2e-3, (ours, theirs)
    assert ours[-1] < ours[0] - 0.5
    # eval-mode losses use the moving statistics (is_training = False), any batch size, odd sizes and slices included
    big = synthetic_batch(150, 4)
    p_all, v_all = tr.losses(*big)
    parts = [tr.losses(big[0][a:b], big[1][a:b], big[2][a:b]) for a, b in ((0, 64), (64, 128), (128, 150))]
    want_p = (parts[0][0] * 64 + parts[1][0] * 64 + parts[2][0] * 22) / 150
    assert abs(p_all - want_p) < 1e-4 and np.isfinite(v_all)
    out = tr.network()
    path = tmp_path / "model-002.npy"
    model.save_model(out, str(path))
    back = model.Network.load(str(path))
    assert back.blocks == blocks and all(np.array_equal(a, b) for a, b in zip(back.conv, out.conv))
    assert not np.array_equal(back.conv[1], network.conv[1]) and not np.array_equal(back.bn[0], network.bn[0])
    tr.close()


def test_resident_games_step_equals_host_minibatch_step(ctx):
    """az_trainer_step_picks (games on the device, extraction + step back to back) == az_samples_extract to the host followed
    by az_trainer_step on the same picks."""
    from conftest import load_golden
    from ataxxzero_b200 import AzError, model, train_data, trainer
    entries = load_golden("train_samples_golden.json")["entries"]
    packed = train_data.pack_entries(entries)
    network = model.Network.random_init(seed=3, blocks=1)
    a, b = trainer.Trainer(ctx, network, max_batch=64), trainer.Trainer(ctx, network, max_batch=64)
    a.set_games(packed)
    w0 = network.conv[1]
    rng = np.random.default_rng(2)
    for step in range(3):
        offsets, meta = train_data.draw_arrays(packed, 64, rng)
        la = a.train_picks(offsets, meta, learning_rate=0.01)
        feats = np.zeros((64, 7, 7, 4), np.int8)
        pol = np.zeros((64, 7, 7, 17), np.float32)
        val = np.zeros((64, 1), np.float32)
        _native = train_data._native
        _native.check(_native.lib().az_samples_extract(ctx.handle, train_data._vp(packed.words.ctypes.data), packed.words.size, train_data._vp(offsets.ctypes.data),
                                                       train_data._vp(meta.ctypes.data), 64, train_data._vp(feats.ctypes.data), train_data._vp(pol.ctypes.data),
                                                       train_data._vp(val.ctypes.data)))
        lb = b.train(feats, pol, val, learning_rate=0.01)
        # the same weights and inputs at step 0: only the order of the fp32 / fp64 atomic sums differs between two runs of a
        # step (DESIGN 3g: like the reference's TensorFlow step it is not bit-reproducible); after that the two trainers'
        # weights drift apart by that rounding, amplified by the momentum updates (observed: 1.2e-5 relative at step 2)
        assert np.allclose(la, lb, rtol=1e-5 if step == 0 else 5e-4, atol=1e-6), (step, la, lb)
        wa, wb = a.debug_read("conv", 1), b.debug_read("conv", 1)
        if step < 2:
            assert np.allclose(wa, wb, rtol=2e-3, atol=1e-5), step
    # by the third step one rounding flip in those sums can move a few hundred of this layer's weights by up to 8e-5, and it
    # does so between two trainers on the SAME path as often (measured on a B200 at 1000 W: in 2 of 6 runs one of three
    # trainers flipped, by 0.6 - 0.75 % of the layer's update): past that point the two paths are held to taking the same
    # update, not to the same rounding.  The 2 % bound is 2.7x the largest flip of those six runs, no more data than that.
    assert np.linalg.norm(wa - wb) < 2e-2 * np.linalg.norm(wb - w0), (np.linalg.norm(wa - wb), np.linalg.norm(wb - w0))
    bad = offsets.copy()
    bad[5] = packed.words.size                                 # outside the table
    with pytest.raises(AzError):
        a.train_picks(bad, meta, learning_rate=0.01)
    with pytest.raises(AzError):
        b.train_picks(offsets, meta, learning_rate=0.01)       # no games loaded
    a.close()
    b.close()


def test_full_size_step_and_argument_checks(ctx):
    """The reference's shape (128 filters x 12 blocks, minibatch 512): finite losses that fall over a few steps; bad calls fail."""
    from ataxxzero_b200 import AzError, model, trainer
    network = model.Network.random_init(seed=1)
    tr = trainer.Trainer(ctx, network, max_batch=512)
    batch = synthetic_batch(512, 9)
    first = tr.train(*batch, learning_rate=0.01)
    for _ in range(10):
        last = tr.train(*batch, learning_rate=0.01)
    assert all(np.isfinite(first)) and last[0] + last[1] < first[0] + first[1]
    assert tr.launches > 0
    with pytest.raises(AzError):
        tr.train(batch[0][:1], batch[1][:1], batch[2][:1], learning_rate=0.01)          # a batch-norm batch of one board
    big = synthetic_batch(514, 2)
    with pytest.raises(AzError):
        tr.train(*big, learning_rate=0.01)                                               # beyond max_batch
    with pytest.raises(AzError):
        tr.train(*batch, learning_rate=float("nan"))
    with pytest.raises(ValueError):
        trainer.Trainer(ctx, model.Network.random_init(seed=1, filters=64, blocks=1))
    tr.close()
    # a minibatch that fills the GPU several times over (501 tiles: the 2-tile conv variant with an odd tile count, 48 ranges
    # of 10-11 tiles in the weight-gradient kernel)
    wide = trainer.Trainer(ctx, model.Network.random_init(seed=2, blocks=2), max_batch=1024)
    big = synthetic_batch(1001, 5)
    first = wide.train(*big, learning_rate=0.01)
    for _ in range(8):
        last = wide.train(*big, learning_rate=0.01)
    assert all(np.isfinite(last)) and last[0] + last[1] < first[0] + first[1]
    wide.close()


def test_context_close_takes_its_pools_and_trainers_along(native):
    """Objects created on a context hold pointers into it: closing the context first (an exception unwinding past a fixture,
    interpreter shutdown order) must close them, not leave them to touch freed memory when they are collected later."""
    import gc
    import ataxxzero_b200
    from ataxxzero_b200 import model, search, trainer
    c = ataxxzero_b200.Context(device=0, seed=3)
    tr = trainer.Trainer(c, model.Network.random_init(seed=1, blocks=1), max_batch=8)
    pool = search.Pool(c, 2, 16, eval_mode=search.EVAL_EXTERNAL)
    c.close()
    assert not tr._h and not pool._h
    with pytest.raises(ataxxzero_b200.AzError):
        tr.train(*synthetic_batch(8, 1), learning_rate=0.01)
    del tr, pool
    gc.collect()
