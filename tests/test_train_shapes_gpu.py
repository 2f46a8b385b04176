"""The training step (csrc/az_train.cu) at the batch sizes where its kernels change code path, and at the shape it trains at.

tests/test_train_gpu.py compares one step tensor by tensor with the fp32 PyTorch restatement at 2..64 boards.  Every kernel
of the step takes another path once the batch grows past that (S = the device's SM count, 148 on a B200):
  * k_conv<2> (two tiles per CTA) runs the forward conv and the data gradient from 2*S + 1 boards on; with an odd tile count
    the last CTA owns a tile past the end;
  * k_heads walks several boards per block from 2*S + 1 boards on, summing the head weight gradients in registers, and a
    block's second board can be the empty half of the last tile;
  * k_wgrad gives a row range more than one tile from 97 boards on, and its 3-stage ring wraps from 289 boards on;
  * the elementwise batch-norm kernels loop over several tiles per block from 129 boards on.
This file checks those paths: one step against fp32 at 2S, 2S + 1, 12 blocks x 512 and 1001 boards; bit-for-bit agreement
of eval-mode outputs across the conv variants, the elementwise chunking and the position of a board in its batch; exact
zeros in the empty half of the last tile; a short trajectory at 12 x 512.

Bounds of the one-step comparison.  The yardstick is the same PyTorch graph under bf16 autocast, measured against its own
fp32 result in the same test: for every compared tensor, our relative L2 distance from fp32 must be at most 1.25 x
autocast's + 1e-3, and below a fixed ceiling: forward tensors (z, act) 2e-2, updated weights 5e-3, moving mean 2e-2 and
variance 1e-3, policy / value loss 2e-3 / 5e-3, gradients cosine >= 0.98 and norm within 3 % (25 layers: 0.95 and 5 %).
Measured on a B200 (1000 W power limit), S = 148:
  * 2 blocks at 296, 297 and 1001 boards: z / act 1.7e-3 (layer 0) .. 5.7e-3 (layer 4), 0.64 .. 0.72 x autocast; gradients
    3.9e-4 .. 0.11 relative L2, cosine >= 0.9936, norms within 1.6 %; d_h 8.9e-2 (autocast 0.11); losses within 2.5e-5;
    updated weights <= 3.7e-4, moving mean <= 1.7e-3, variance <= 1.8e-7.  The same as at 64 boards (test_train_gpu.py).
  * 12 blocks x 512 boards: z / act grow with depth from 1.7e-3 (layer 0) to 1.7e-2 (layer 24), autocast's from 2.4e-3 to
    2.6e-2 -- each layer adds the rounding of its bf16 operands to what it inherits, and ours stays 0.64 .. 0.72 x autocast's
    at every depth.  Gradients grow the same way down the data-gradient chain: grad_conv 5.8e-2 at layer 24 (autocast 7.6e-2)
    to 0.22 at layer 0 (autocast 0.28), d_h 0.23 (autocast 0.28); every gradient tensor 0.15 .. 1.02 x autocast's distance.
    That is 24 data-gradient convs, each rounding its dz to bf16 and summing 1152 products of mixed sign; at random init the
    sums cancel to a small fraction of their terms, which magnifies the rounding.  Autocast's own cosine falls to 0.945 and
    its norms stray by up to 4.7 %; ours, cosine >= 0.966 and norms within 3.5 %.  So at 25 layers the gradient ceiling is
    cosine 0.95 and norm 5 %, just outside what bf16 rounding alone does there, and the 1.25 x autocast rule is unchanged.
    Losses within 1.1e-4, updated weights <= 3.4e-3 (autocast 4.2e-3), moving mean <= 2.0e-3, variance <= 1.6e-6.
  * grad_fc_b, one scalar, is held to autocast's distance on grad_fc_w (see the test): measured 3.9e-4 .. 1.5e-2.
"""
import copy

import numpy as np
import pytest

from test_train_gpu import cosine, rel, synthetic_batch, torch_setup

pytestmark = pytest.mark.gpu

LR, LAM = 0.01, 1e-4


@pytest.fixture(scope="module")
def sms():
    """The SM count the library sizes its launches with (ctx->sm_count comes from the same device property)."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def nhwc(t):
    return t.detach().float().permute(0, 2, 3, 1).cpu().numpy()


def tf_conv(t):
    return t.detach().float().permute(2, 3, 1, 0).cpu().numpy()


class Checks:
    """Collects every comparison of a test, prints the table (pytest -s shows it) and fails once, naming every miss.
    cos_min / norm_tol: the hard ceiling on gradients (cosine with fp32, norm ratio)."""

    def __init__(self, title, cos_min, norm_tol):
        self.title, self.cos_min, self.norm_tol, self.lines, self.misses = title, cos_min, norm_tol, [], []

    def forward(self, name, ours, want, auto, ceiling=2e-2):
        e, a = rel(ours, want), rel(auto, want)
        self._add(name, "rel %.2e  autocast %.2e" % (e, a), e <= 1.25 * a + 1e-3 and e <= ceiling)

    def grad(self, name, ours, want, auto, yardstick=None):
        """yardstick: autocast's distance to hold ours to, when not this tensor's own (a single number)."""
        e, a, c = rel(ours, want), rel(auto, want) if yardstick is None else yardstick, cosine(ours, want)
        ratio = np.linalg.norm(ours) / max(np.linalg.norm(want), 1e-30)
        self._add(name, "rel %.2e  autocast %.2e  cos %.5f (autocast %.5f)  norm %.4f (autocast %.4f)" % (
            e, a, c, cosine(auto, want), ratio, np.linalg.norm(auto) / max(np.linalg.norm(want), 1e-30)),
                  e <= 1.25 * a + 1e-3 and c >= self.cos_min and abs(ratio - 1) <= self.norm_tol)

    def value(self, name, ours, want, bound):
        e = abs(ours - want)
        self._add(name, "ours %.6f  fp32 %.6f  diff %.2e  bound %.1e" % (ours, want, e, bound), e <= bound)

    def _add(self, name, text, ok):
        self.lines.append("%-28s %s%s" % (name, text, "" if ok else "   <-- FAIL"))
        if not ok:
            self.misses.append(name)

    def finish(self):
        print("\n== %s\n%s" % (self.title, "\n".join(self.lines)))
        assert not self.misses, "%s: %d comparisons out of bounds: %s\n%s" % (self.title, len(self.misses), ", ".join(self.misses),
                                                                               "\n".join(l for l in self.lines if "FAIL" in l))


SHAPES = [pytest.param(2, lambda s: 2 * s, id="2blocks-2S"),             # k_conv<1> at its largest, several tiles per elementwise block
          pytest.param(2, lambda s: 2 * s + 1, id="2blocks-2S+1"),       # k_conv<2>, odd tile count, head block ending on the empty board
          pytest.param(12, lambda s: 512, id="12blocks-512"),            # the production shape: 5-6 tiles per wgrad range, the ring wraps
          pytest.param(2, lambda s: 1001, id="2blocks-1001")]            # 501 tiles, 3-4 boards per head block


@pytest.mark.parametrize("blocks,size", SHAPES)
def test_one_step_at_switching_shapes(ctx, sms, blocks, size):
    """One step against the fp32 restatement, constructed like test_one_step_matches_fp32_restatement: the three losses,
    every layer's conv output z and activation, d_h (the gradient with respect to layer 0's output, the end of the data-
    gradient chain), every gradient tensor, and after the update every layer's weights and moving statistics."""
    import torch
    from ataxxzero_b200 import model, trainer
    n = size(sms)
    network = model.Network.random_init(seed=5, blocks=blocks)
    ref, net, opt, dev = torch_setup(network, blocks, LR)
    net16 = copy.deepcopy(net)                               # before any forward: its moving statistics start where net's do
    opt16 = torch.optim.SGD(net16.parameters(), lr=LR, momentum=0.9)
    tr = trainer.Trainer(ctx, network, max_batch=n)
    batch = synthetic_batch(n, 1)
    x, pol, val = ref.to_torch_batch(batch, dev)
    pl, vl, reg, zs, acts = ref.loss_terms_retained(net, x, pol, val)
    opt.zero_grad()
    (pl + vl + reg).backward()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        p16, v16, r16, zs16, acts16 = ref.loss_terms_retained(net16, x, pol, val)
    opt16.zero_grad()
    (p16.float() + v16.float() + r16.float()).backward()
    ours = tr.train(*batch, learning_rate=LR)

    # 25 layers: the gradient ceiling moves with the rounding the data-gradient chain accumulates (module docstring)
    ck = Checks("one step, %d blocks x %d boards (S = %d)" % (blocks, n, sms), *((0.98, 0.03) if blocks <= 2 else (0.95, 0.05)))
    ck.value("policy loss", ours[0], pl.item(), min(1.25 * abs(p16.item() - pl.item()) + 1e-3, 2e-3))
    ck.value("value loss", ours[1], vl.item(), min(1.25 * abs(v16.item() - vl.item()) + 1e-3, 5e-3))
    ck.value("regularisation", ours[2], reg.item(), 1e-5 * reg.item() + 1e-7)
    layers = 1 + 2 * blocks
    for l in range(layers):
        ck.forward("z[%d]" % l, tr.debug_read("z", l, n), nhwc(zs[l]), nhwc(zs16[l]))
        ck.forward("act[%d]" % (l + 1), tr.debug_read("act", l + 1, n), nhwc(acts[l]), nhwc(acts16[l]))
    ck.grad("d_h", tr.debug_read("d_h", 0, n), nhwc(acts[0].grad), nhwc(acts16[0].grad))
    for l in range(layers):
        w, w16 = net.convs[l].weight, net16.convs[l].weight
        g = tr.debug_read("grad_conv", l)
        if l == 0:
            assert not g[:, :, 4:, :].any()                                      # padded input channels stay exactly zero
            g = g[:, :, :4, :]
        ck.grad("grad_conv[%d]" % l, g, tf_conv(w.grad - LAM * w), tf_conv(w16.grad - LAM * w16))
        for name, p, p16_ in (("grad_gamma", net.bns[l].weight, net16.bns[l].weight), ("grad_beta", net.bns[l].bias, net16.bns[l].bias)):
            ck.grad("%s[%d]" % (name, l), tr.debug_read(name, l), (p.grad - LAM * p).detach().cpu().numpy(),
                    (p16_.grad - LAM * p16_).detach().float().cpu().numpy())
    gh = tr.debug_read("grad_heads")

    def head(m):
        return [(m.policy.weight.grad - LAM * m.policy.weight).detach().reshape(17, 128).t().cpu().numpy(),
                (m.value.weight.grad - LAM * m.value.weight).detach().reshape(128).cpu().numpy(),
                (m.fc_w.grad - LAM * m.fc_w).detach().reshape(49).cpu().numpy(),
                (m.fc_b.grad - LAM * m.fc_b).detach().cpu().numpy()]
    parts = [gh[:128 * 17].reshape(128, 17), gh[128 * 17:128 * 18], gh[128 * 18:128 * 18 + 49], gh[-1:]]
    for name, o, want, auto in zip(("grad_policy", "grad_value", "grad_fc_w"), parts, head(net), head(net16)):
        ck.grad(name, o, want, auto)
    # the fc_b gradient is ONE number, sum over boards of d loss / d (value pre-activation), which cancels to a fraction of its
    # terms: its distance from fp32 is one draw of rounding noise, and autocast's one draw is no yardstick for it (measured
    # ratios 0.45 .. 8 across the shapes here).  It is held to autocast's error on the 49 fc_w gradients, sums of the same terms.
    ck.grad("grad_fc_b", parts[3], head(net)[3], head(net16)[3], yardstick=max(rel(head(net16)[3], head(net)[3]), rel(head(net16)[2], head(net)[2])))
    opt.step()
    opt16.step()
    for l in range(layers):
        w = tr.debug_read("conv", l)
        ck.forward("conv[%d] updated" % l, w[:, :, :4, :] if l == 0 else w, tf_conv(net.convs[l].weight), tf_conv(net16.convs[l].weight), 5e-3)
        mv = tr.debug_read("moving", l)
        bn, bn16 = net.bns[l], net16.bns[l]
        ck.forward("moving mean[%d]" % l, mv[0], bn.running_mean.cpu().numpy(), bn16.running_mean.cpu().numpy())
        ck.forward("moving var[%d]" % l, mv[1], bn.running_var.cpu().numpy(), bn16.running_var.cpu().numpy(), 1e-3)
    tr.close()
    ck.finish()


def bn_network(blocks, seed):
    """A random network with non-trivial moving statistics, so that eval-mode batch-norm is not the identity."""
    from ataxxzero_b200 import model
    from oracle import net_numpy
    network = model.Network.random_init(seed=seed, blocks=blocks)
    return model.Network(network.conv, net_numpy.randomize_bn(network.bn, seed=seed))


def make_trainer(ctx, monkeypatch, network, max_batch, conv_tiles=None, ew_chunks=None):
    """A trainer with the AZ_TRAIN_CONV_TILES / AZ_TRAIN_EW_CHUNKS knobs set (None: unset, the library's choice); they are
    read when the trainer is created."""
    from ataxxzero_b200 import trainer
    for var, v in (("AZ_TRAIN_CONV_TILES", conv_tiles), ("AZ_TRAIN_EW_CHUNKS", ew_chunks)):
        if v is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(v))
    return trainer.Trainer(ctx, network, max_batch=max_batch)


@pytest.mark.parametrize("size", [pytest.param(lambda s: 2 * s + 1, id="2S+1"), pytest.param(lambda s: 64, id="64")])
def test_conv_variants_agree_bit_for_bit(ctx, sms, monkeypatch, size):
    """Both conv variants read the same input tile and weight image and accumulate each tile's 72 MMAs in the same order,
    so their results are the same bits.  In eval mode nothing between the input and the logits is summed with atomics
    (moving statistics, no batch statistics), so the logits and values must be identical; in training mode so must layer
    0's conv output (the layers above it normalise with fp64 atomic batch sums, whose order is free)."""
    n = size(sms)
    network = bn_network(2, 11)
    batch = synthetic_batch(n, 12)
    out = {}
    for tiles in (1, 2):
        tr = make_trainer(ctx, monkeypatch, network, n, conv_tiles=tiles)
        _, _, logits, values = tr.losses(*batch, outputs=True)
        tr.train(*batch, learning_rate=LR)
        out[tiles] = (logits, values, tr.debug_read("z", 0, n))
        tr.close()
    assert np.isfinite(out[1][0]).all() and np.abs(out[1][0]).max() > 0
    for what, a, b in zip(("logits", "values", "training z[0]"), out[1], out[2]):
        assert np.array_equal(a, b), (what, n, int((a != b).sum()), float(np.abs(a - b).max()))


def test_elementwise_chunking_agrees_bit_for_bit(ctx, sms, monkeypatch):
    """AZ_TRAIN_EW_CHUNKS sets how many blocks per channel group the elementwise batch-norm kernels use; each element is
    computed by exactly one thread whatever the chunking, so eval-mode outputs at 2S + 1 boards must be the same bits for the
    default (64: several tiles per block), 1 (one block walks every tile) and 7 (uneven strides)."""
    n = 2 * sms + 1
    network = bn_network(2, 13)
    batch = synthetic_batch(n, 14)
    out = []
    for chunks in (None, 1, 7):
        tr = make_trainer(ctx, monkeypatch, network, n, ew_chunks=chunks)
        out.append(tr.losses(*batch, outputs=True)[2:])
        tr.close()
    for chunks, (logits, values) in zip((1, 7), out[1:]):
        assert np.array_equal(logits, out[0][0]) and np.array_equal(values, out[0][1]), (chunks, int((logits != out[0][0]).sum()))


def test_board_result_does_not_depend_on_its_batch(ctx, sms, monkeypatch):
    """A board's eval-mode logits and value are the same bits whether it is computed inside a batch of 2S + 1 boards (k_conv<2>,
    several boards per head block) or in a batch of two (k_conv<1>, one tile), in either half of a tile: the rows of
    neighbouring boards never meet under a tap shift (the padding row and column of the 8 x 8 frame are zero).  Also the
    eval-mode forward at 2S + 1 boards against the library's fp32 inference kernel on the same network."""
    from ataxxzero_b200 import net as aznet
    n = 2 * sms + 1
    network = bn_network(2, 15)
    feats, pol, val = synthetic_batch(n, 16)
    tr = make_trainer(ctx, monkeypatch, network, n)
    _, _, logits, values = tr.losses(feats, pol, val, outputs=True)
    other = synthetic_batch(2, 17)
    for b in (0, 1, sms, 2 * sms - 1, 2 * sms):                   # first / second half, the middle, the half-empty last tile
        for pos in (0, 1):
            f2, p2, v2 = (a.copy() for a in other)
            f2[pos], p2[pos], v2[pos] = feats[b], pol[b], val[b]
            _, _, lg2, vv2 = tr.losses(f2, p2, v2, outputs=True)
            assert np.array_equal(lg2[pos], logits[b]) and np.array_equal(vv2[pos], values[b]), (b, pos, float(np.abs(lg2[pos] - logits[b]).max()))
    tr.close()
    aznet.load_weights(ctx, network)
    lg, vv = aznet.forward(ctx, feats.astype(np.float32), mode=aznet.FP32)
    assert np.abs(logits - lg.reshape(logits.shape)).max() < 2e-2 and np.abs(values.reshape(-1) - vv.reshape(-1)).max() < 2e-2


@pytest.mark.parametrize("conv_tiles", [1, 2])
def test_empty_half_of_last_tile_stays_zero(ctx, sms, monkeypatch, conv_tiles):
    """With an odd batch the second board of the last tile is not part of it.  k_stage_input, the conv epilogue's row mask,
    k_bn_apply's live mask, the k_heads zero fill and k_bn_bwd_apply all keep it at exactly zero -- if it leaked, the batch
    statistics of the real boards would pick up a ghost board.  The trainer first steps on a full batch of n + 1 boards, so
    that board n holds real data before the odd step has to clear it."""
    n = 2 * sms + 1
    blocks = 2
    network = bn_network(blocks, 19)
    tr = make_trainer(ctx, monkeypatch, network, n + 1, conv_tiles=conv_tiles)
    tr.train(*synthetic_batch(n + 1, 20), learning_rate=LR)
    tr.train(*synthetic_batch(n, 21), learning_rate=LR)
    layers = 1 + 2 * blocks
    reads = [("z", l) for l in range(layers)] + [("act", l) for l in range(layers + 1)] + [("d_h", 0)]
    for what, l in reads:
        t = tr.debug_read(what, l, n + 1)
        assert np.abs(t[n - 1]).max() > 0, (what, l)                  # the last real board is not zero
        assert not t[n].any(), (what, l, int(np.count_nonzero(t[n])), float(np.abs(t[n]).max()))
    tr.close()


def test_short_production_trajectory(ctx):
    """5 momentum steps on one batch at 12 blocks x 512 boards, lr 0.01: the native policy + value loss follows PyTorch's fp32
    trajectory at every step, as closely as PyTorch's own bf16 autocast trajectory does.  An update that is right in
    direction but wrong in size somewhere deep in the tower shows up here as a drift that grows step by step.
    Measured on a B200 (1000 W): losses 7.966 -> 6.846; ours from fp32 2.2e-4, 5.5e-4, 1.7e-3 .. 1.9e-3, 5.1e-3 .. 5.7e-3,
    2.5e-3 .. 2.6e-3 (two runs), bf16 autocast from fp32 2.0e-4, 5e-5, 2.1e-4, 4.3e-3, 2.0e-3.  Both stray most at step 3,
    in the same direction: the trajectory itself is that sensitive to rounding there.  Bound: at every step, 1.25 x the
    largest distance of the bf16 trajectory + the 2e-3 of the 30-step check at 2 blocks x 64 boards = 7.4e-3.  A wgrad
    range that drops a tile, or head gradients from one board per block, drift by 0.018 .. 0.07 at step 1
    and 0.04 .. 0.23 by step 4."""
    import torch
    from ataxxzero_b200 import model, trainer
    blocks, n, steps = 12, 512, 5
    network = model.Network.random_init(seed=7, blocks=blocks)
    ref, net, opt, dev = torch_setup(network, blocks, LR)
    net16 = copy.deepcopy(net)
    opt16 = torch.optim.SGD(net16.parameters(), lr=LR, momentum=0.9)
    tr = trainer.Trainer(ctx, network, max_batch=n)
    batch = synthetic_batch(n, 3)
    xb = ref.to_torch_batch(batch, dev)
    ours, fp32, bf16 = [], [], []
    for _ in range(steps):
        lo = tr.train(*batch, learning_rate=LR)
        ours.append(lo[0] + lo[1])
        for m, o, out, cast in ((net, opt, fp32, False), (net16, opt16, bf16, True)):
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=cast):
                p2, v2, r2 = ref.loss_terms(m, *xb)
            o.zero_grad()
            (p2.float() + v2.float() + r2.float()).backward()
            o.step()
            out.append(float(p2.detach().float() + v2.detach().float()))
    tr.close()
    ours, fp32, bf16 = np.array(ours), np.array(fp32), np.array(bf16)
    print("\n== trajectory 12 x 512\nours  %s\nfp32  %s\nbf16  %s" % tuple(" ".join("%.5f" % v for v in a) for a in (ours, fp32, bf16)))
    assert ours[-1] < ours[0] - 0.1, ours
    assert (np.abs(ours - fp32) <= 1.25 * np.abs(bf16 - fp32).max() + 2e-3).all(), (ours - fp32, bf16 - fp32)
