"""fp32 PyTorch restatement of the reference's training graph (model.py:35-101) -- TEST INFRASTRUCTURE: the checker the
hand-written training step (ataxxzero_b200/csrc/az_train.cu) is compared with.  Nothing under ataxxzero_b200/ imports it."""
import numpy as np

from ataxxzero_b200 import model as azmodel


def build_torch_network(filters, blocks):
    import torch
    import torch.nn as nn

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            def conv(cin, cout, k):
                return nn.Conv2d(cin, cout, k, padding=k // 2, bias=False)
            def bn():
                return nn.BatchNorm2d(filters, eps=1e-3, momentum=0.01)     # tf momentum 0.99
            self.convs = nn.ModuleList([conv(4, filters, 3)] + [conv(filters, filters, 3) for _ in range(2 * blocks)])
            self.bns = nn.ModuleList([bn() for _ in range(1 + 2 * blocks)])
            self.policy = conv(filters, azmodel.MOVE_TYPES, 1)
            self.value = conv(filters, 1, 1)
            self.fc_w = nn.Parameter(torch.zeros(49, 1))
            self.fc_b = nn.Parameter(torch.full((1,), 0.01))

        def forward(self, x):                      # x: [B, 4, 7(x), 7(y)] float
            import torch.nn.functional as F
            h = F.relu(self.bns[0](self.convs[0](x)))
            for b in range((len(self.convs) - 1) // 2):
                y = F.relu(self.bns[1 + 2 * b](self.convs[1 + 2 * b](h)))
                y = self.bns[2 + 2 * b](self.convs[2 + 2 * b](y))
                h = F.relu(y + h)
            logits = self.policy(h).permute(0, 2, 3, 1).reshape(len(x), -1)          # [B, 7*7*17], index 119x + 17y + plane
            v = self.value(h).permute(0, 2, 3, 1).reshape(len(x), 49)                # x-major, like tf.reshape of NHWC
            return logits, torch.tanh(v @ self.fc_w + self.fc_b)

    return Net()


def load_into(net, network):
    """model.Network (TF layout [kh(x), kw(y), Cin, Cout]) -> torch modules (NCHW with H = x, W = y)."""
    import torch
    with torch.no_grad():
        convs = list(net.convs) + [net.policy, net.value]
        for module, w in zip(convs, network.conv[:len(convs)]):
            module.weight.copy_(torch.from_numpy(np.ascontiguousarray(w.transpose(3, 2, 0, 1))))
        net.fc_w.copy_(torch.from_numpy(network.conv[-2]))
        net.fc_b.copy_(torch.from_numpy(network.conv[-1]))
        for i, bn in enumerate(net.bns):
            bn.running_mean.copy_(torch.from_numpy(network.bn[2 * i]))
            bn.running_var.copy_(torch.from_numpy(network.bn[2 * i + 1]))


def export(net):
    """torch modules -> model.Network: conv / FC weights + batch-norm moving statistics (gamma / beta are not saved).
    torch accumulates the UNBIASED batch variance in running_var where TF's moving_variance takes the biased one; with
    minibatch * 49 >= 25 000 samples per channel the factor n / (n - 1) is below 1.00005 and is exported as is."""
    convs = list(net.convs) + [net.policy, net.value]
    conv = [m.weight.detach().cpu().numpy().transpose(2, 3, 1, 0).copy() for m in convs]
    conv += [net.fc_w.detach().cpu().numpy().copy(), net.fc_b.detach().cpu().numpy().copy()]
    bn = []
    for m in net.bns:
        bn += [m.running_mean.detach().cpu().numpy().copy(), m.running_var.detach().cpu().numpy().copy()]
    return azmodel.Network(conv, bn)


def loss_terms(net, features, policies, values):
    """(policy_loss, value_loss, regularization) exactly as model.py:81-96 defines them."""
    import torch
    logits, out = net(features)
    log_sm = torch.log_softmax(logits, dim=1)
    policy_loss = -(policies.reshape(len(features), -1) * log_sm).sum(dim=1).mean()
    value_loss = ((values - out) ** 2).mean()
    reg = 0.0001 * sum(0.5 * (p ** 2).sum() for p in net.parameters())               # l2_regularizer(scale) = scale * l2_loss
    return policy_loss, value_loss, reg


def loss_terms_retained(net, features, policies, values):
    """loss_terms written out layer by layer, keeping what the native step's debug_read can be compared with:
    returns (policy_loss, value_loss, reg, zs, acts) where zs[l] is layer l's conv output and acts[l] its output activation
    (after the residual add and ReLU; acts[-1] is the tower output).  Every acts[l] retains its gradient, so after backward
    acts[0].grad is the gradient with respect to layer 0's output."""
    import torch
    import torch.nn.functional as F
    zs, acts = [], []

    def conv_bn(i, inp):
        z = net.convs[i](inp)
        zs.append(z)
        return net.bns[i](z)

    def keep(a):
        a.retain_grad()
        acts.append(a)
        return a
    h = keep(F.relu(conv_bn(0, features)))
    for b in range((len(net.convs) - 1) // 2):
        y = keep(F.relu(conv_bn(1 + 2 * b, h)))
        h = keep(F.relu(conv_bn(2 + 2 * b, y) + h))
    n = len(features)
    logits = net.policy(h).permute(0, 2, 3, 1).reshape(n, -1)
    out = torch.tanh(net.value(h).permute(0, 2, 3, 1).reshape(n, 49) @ net.fc_w + net.fc_b)
    policy_loss = -(policies.reshape(n, -1) * torch.log_softmax(logits, dim=1)).sum(dim=1).mean()
    value_loss = ((values - out) ** 2).mean()
    reg = 0.0001 * sum(0.5 * (p ** 2).sum() for p in net.parameters())
    return policy_loss, value_loss, reg, zs, acts


def to_torch_batch(batch, device):
    import torch
    feats, pol, val = batch
    x = torch.from_numpy(np.ascontiguousarray(feats.astype(np.float32).transpose(0, 3, 1, 2))).to(device)    # [B,x,y,c] -> [B,c,x,y]
    return x, torch.from_numpy(pol).to(device), torch.from_numpy(val.astype(np.float32)).to(device)


def host_minibatch_fn(entries):
    """NumPy twin of az_samples_extract behind train_data.draw's picks: lets the CPU tests pin the sampling + encoding rules
    (train.py:43-77) against the reference goldens without a GPU."""
    from ataxxzero_b200 import train_data
    packed = train_data.pack_entries(entries)

    def host(size, rng):
        picks = train_data.draw(packed, size, rng)
        feats = np.zeros((size, 7, 7, 4), np.int8)
        pol = np.zeros((size, 7, 7, 17), np.float32)
        val = np.zeros((size, 1), np.float32)
        from ataxxzero_b200.engine import add_move_to_heatmap
        from ataxxzero_b200.rules import to_reference_move, unpack_move
        for i, (g, ply, sym) in enumerate(picks):
            entry = entries[g]
            to_move = 1 if ply % 2 == 0 else 2
            def tr(xy):
                x, y = xy
                if sym & 1: x = 6 - x
                if sym & 2: y = 6 - y
                return (y, x) if sym & 4 else (x, y)
            for idx, v in enumerate(entry["boards"][ply]):
                x, y = tr((idx % 7, idx // 7))
                feats[i, x, y, 0] = 1
                if v:
                    feats[i, x, y, 1 if v == to_move else 2] = 1
            off = packed.offsets[g][ply]
            w = packed.words
            n_e = int(w[off + 4] >> 16) if packed.has_dists[g] else 1
            for e in range(n_e):
                if packed.has_dists[g]:
                    mv, p = int(w[off + 6 + 2 * e]) & 0xffff, float(np.uint32(w[off + 7 + 2 * e]).view(np.float32))
                else:
                    mv, p = int(w[off + 4]) & 0xffff, 1.0
                start, end = to_reference_move(unpack_move(mv))
                move = ("c", tr(end)) if start == "c" else (tr(start), tr(end))
                add_move_to_heatmap(pol[i], move, np.float32(p))
            val[i, 0] = 1.0 if entry["result"] == to_move else -1.0
        return feats, pol, val
    return host
