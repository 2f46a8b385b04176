"""Stage-by-stage comparison of the hand-written training step (csrc/az_train.cu) with the fp32 PyTorch restatement
(tests/torch_train_reference.py): conv outputs, activations, losses, every gradient, updated weights.  GPU box only."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import ataxxzero_b200 as az
from ataxxzero_b200 import model, trainer
import torch_train_reference as ref

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
BLOCKS = int(sys.argv[1]) if len(sys.argv) > 1 else 2
N = int(sys.argv[2]) if len(sys.argv) > 2 else 64
LR = 0.01


def rel(a, b):
    a = np.asarray(a, np.float64).ravel(); b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


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


ctx = az.Context(0)
network = model.Network.random_init(seed=5, blocks=BLOCKS)
tr = trainer.Trainer(ctx, network, max_batch=max(N, 2))
dev = torch.device("cuda", 0)
net = ref.build_torch_network(128, BLOCKS).to(dev)
ref.load_into(net, network)
net.train()
opt = torch.optim.SGD(net.parameters(), lr=LR, momentum=0.9)
batch = synthetic_batch(N, 1)
x, pol, val = ref.to_torch_batch(batch, dev)

# torch forward with intermediates (zs[l] conv output, acts[l] output activation of layer l; acts[0].grad = d loss / d layer 0's output)
pl, vl, reg, zs, acts = ref.loss_terms_retained(net, x, pol, val)
opt.zero_grad()
(pl + vl + reg).backward()

losses = tr.train(*batch, learning_rate=LR)
print("losses ours %s torch (%.6f, %.6f, %.6f)" % (losses, float(pl), float(vl), float(reg)))
L = 1 + 2 * BLOCKS
for l in range(L):
    z_ours = tr.debug_read("z", l, N)
    z_ref = zs[l].detach().permute(0, 2, 3, 1).cpu().numpy()
    a_ours = tr.debug_read("act", l + 1, N)
    a_ref = acts[l].detach().permute(0, 2, 3, 1).cpu().numpy()
    print("layer %2d  z rel %.2e  act rel %.2e" % (l, rel(z_ours, z_ref), rel(a_ours, a_ref)))
d_ours = tr.debug_read("d_h", 0, N)                                            # after the step: d loss / d (layer 0's output)
d_ref = acts[0].grad.permute(0, 2, 3, 1).cpu().numpy()
print("d_h (layer 0 output grad) rel %.2e  cosine %.6f  norm ours %.3e ref %.3e" % (
    rel(d_ours, d_ref), float(d_ours.ravel() @ d_ref.ravel() / (np.linalg.norm(d_ours) * np.linalg.norm(d_ref))), np.linalg.norm(d_ours), np.linalg.norm(d_ref)))
lam = 1e-4
for l in reversed(range(L)):
    g_ours = tr.debug_read("grad_conv", l)
    w = net.convs[l].weight
    g_ref = (w.grad - lam * w).detach().permute(2, 3, 1, 0).cpu().numpy()      # [kx][ky][cin][cout], L2 term removed
    if l == 0:
        g_ours = g_ours[:, :, :4, :]
    gg = tr.debug_read("grad_gamma", l); gb = tr.debug_read("grad_beta", l)
    gg_ref = (net.bns[l].weight.grad - lam * net.bns[l].weight).detach().cpu().numpy()
    gb_ref = (net.bns[l].bias.grad - lam * net.bns[l].bias).detach().cpu().numpy()
    print("layer %2d  grad_conv rel %.2e (norm ours %.3e ref %.3e)  grad_gamma rel %.2e  grad_beta rel %.2e" % (
        l, rel(g_ours, g_ref), np.linalg.norm(g_ours), np.linalg.norm(g_ref), rel(gg, gg_ref), rel(gb, gb_ref)))
gh = tr.debug_read("grad_heads")
gp_ref = (net.policy.weight.grad - lam * net.policy.weight).detach().reshape(17, 128).t().cpu().numpy()
gv_ref = (net.value.weight.grad - lam * net.value.weight).detach().reshape(128).cpu().numpy()
gw_ref = (net.fc_w.grad - lam * net.fc_w).detach().reshape(49).cpu().numpy()
gb_ref = (net.fc_b.grad - lam * net.fc_b).detach().cpu().numpy()
print("heads: grad_policy rel %.2e  grad_value rel %.2e  grad_fc_w rel %.2e  grad_fc_b rel %.2e" % (
    rel(gh[:128 * 17].reshape(128, 17), gp_ref), rel(gh[128 * 17:128 * 18], gv_ref), rel(gh[128 * 18:128 * 18 + 49], gw_ref), rel(gh[-1:], gb_ref)))
# how large is bf16 operand rounding by itself?  the SAME PyTorch graph under bf16 autocast against its own fp32 gradients
import copy
net16 = copy.deepcopy(net)
for p_ in net16.parameters():
    p_.grad = None
with torch.autocast("cuda", dtype=torch.bfloat16):
    p16, v16, r16 = ref.loss_terms(net16, x, pol, val)
(p16.float() + v16.float() + r16.float()).backward()
print("PyTorch bf16 autocast vs its own fp32 gradients (operand rounding alone): " + "  ".join(
    "layer %d %.2e" % (l, rel(net16.convs[l].weight.grad.float().cpu().numpy(), net.convs[l].weight.grad.cpu().numpy())) for l in reversed(range(L))))
opt.step()
for l in (0, 1, L - 1):
    w_ours = tr.debug_read("conv", l)
    w_ref = net.convs[l].weight.detach().permute(2, 3, 1, 0).cpu().numpy()
    if l == 0:
        w_ours = w_ours[:, :, :4, :]
    print("layer %2d  updated weights rel %.2e" % (l, rel(w_ours, w_ref)))
mv = tr.debug_read("moving", 1)
print("moving mean rel %.2e var rel %.2e" % (rel(mv[0], net.bns[1].running_mean.cpu().numpy()), rel(mv[1], net.bns[1].running_var.cpu().numpy())))

# a short run on a fixed batch: both must drive the loss down the same way
hist_o, hist_t = [], []
for step in range(30):
    lo = tr.train(*batch, learning_rate=LR)
    p2, v2, r2 = ref.loss_terms(net, x, pol, val)
    opt.zero_grad(); (p2 + v2 + r2).backward(); opt.step()
    hist_o.append(lo[0] + lo[1]); hist_t.append(float(p2 + v2))
print("fixed-batch run  ours:", " ".join("%.4f" % v for v in hist_o[::5]))
print("fixed-batch run torch:", " ".join("%.4f" % v for v in hist_t[::5]))
# eval mode agrees with the inference kernels of the library on the exported network
net_e = tr.network()
pe, ve, lg, vals = tr.losses(*batch, outputs=True)
from ataxxzero_b200 import net as aznet
aznet.load_weights(ctx, net_e)
lg2, v2 = aznet.forward(ctx, batch[0].astype(np.float32), mode=aznet.FP32)
print("eval vs fp32 inference kernel: logits max abs %.2e values max abs %.2e (gamma/beta are dropped on export: expect a gap after training)" % (
    np.abs(lg - lg2.reshape(lg.shape)).max(), np.abs(vals.reshape(-1) - v2.reshape(-1)).max()))

# timing
for n_t, blocks_t in ((512, 12),):
    network_t = model.Network.random_init(seed=1, blocks=blocks_t)
    trt = trainer.Trainer(ctx, network_t, max_batch=n_t)
    bt = synthetic_batch(n_t, 2)
    for _ in range(3): trt.train(*bt, learning_rate=1e-3)
    t0 = time.perf_counter(); l0 = trt.launches
    for _ in range(20): trt.train(*bt, learning_rate=1e-3)
    dt = (time.perf_counter() - t0) / 20
    print("native step %d x %d blocks: %.3f ms/step (%.0f samples/s, %d launches/step)" % (n_t, blocks_t, dt * 1e3, n_t / dt, (trt.launches - l0) // 20))
    nett = ref.build_torch_network(128, blocks_t).to(dev); ref.load_into(nett, network_t); nett.train()
    optt = torch.optim.SGD(nett.parameters(), lr=1e-3, momentum=0.9)
    xb = ref.to_torch_batch(bt, dev)
    def tstep():
        p2, v2, r2 = ref.loss_terms(nett, *xb); optt.zero_grad(); (p2 + v2 + r2).backward(); optt.step()
    for _ in range(3): tstep()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(10): tstep()
    torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 10
    print("torch fp32 eager step: %.3f ms/step (%.0f samples/s)" % (dt * 1e3, n_t / dt))
