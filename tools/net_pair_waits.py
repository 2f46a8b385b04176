"""Where k_net_pair's issuing thread waits, from clock64() stamps taken in the kernel (az_net_pair_profile).

    python tools/net_pair_waits.py [boards ...]          # default 1776 2048

For every leader CTA the issuer records how long it waits on weights (B_FULL), on the first and second input-channel part of a
layer's activations (B_ACT 0/1), on the staged input planes (B_IN), and the "gap" from each accumulator commit to the moment the
next layer's first part is ready -- the stretch in which the pair has no MMA queued.  Shares are of the issuer's span (setup to
last accumulator).  The tensor pipe of an SM serves both CTA pairs resident on its TPC, so a pair's gap only idles the pipe while
the other pair is in a gap too: for SMs that host the leaders of both pairs (one clock), the script also reports the time in which
both leaders have nothing queued, as a share of that SM's span.  Gaps behind the second part (B_ACT 1) and weight starvation are
not in that figure: it is a lower bound on the idle pipe.
"""
import ctypes as C
import os
import sys
from collections import defaultdict

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ataxxzero_b200 as az
from ataxxzero_b200 import _native, model, net

GAP, ACT0, ACT1, FULL, IN, UNIT_GAP = range(6)
MAX_REC = 1024
STRIDE = 4 + 3 * MAX_REC


def merge(iv):
    out = []
    for a, b in sorted(iv):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def overlap(x, y):
    i = j = 0
    tot = 0
    while i < len(x) and j < len(y):
        lo, hi = max(x[i][0], y[j][0]), min(x[i][1], y[j][1])
        if hi > lo:
            tot += hi - lo
        if x[i][1] < y[j][1]:
            i += 1
        else:
            j += 1
    return tot


def analyse(buf, nl):
    ctas = []
    for row in buf:
        n = int(row[3])
        if n <= 0:
            continue
        r = row[4:4 + 3 * n].reshape(n, 3)
        ctas.append((int(row[0]), int(row[1]), int(row[2]), r))
    span = sum(c[2] - c[1] for c in ctas)
    kinds = defaultdict(int)
    per_layer = defaultdict(lambda: defaultdict(int))
    for _, _, _, r in ctas:
        for code, t0, t1 in r:
            k, layer = int(code) & 255, int(code) >> 8
            kinds[k] += int(t1 - t0)
            per_layer[k][layer] += int(t1 - t0)
    print("  leader CTAs %d, mean issuer span %.0f clk" % (len(ctas), span / max(len(ctas), 1)))
    for k, name in ((FULL, "B_FULL (weights)"), (ACT0, "B_ACT 0 (+heads: both parts)"), (ACT1, "B_ACT 1"), (IN, "B_IN (input)"),
                    (GAP, "gap: acc done -> part 0 ready"), (UNIT_GAP, "gap: heads done -> input ready (incl. ramp)")):
        print("  %-44s %6.2f %% of issuer span" % (name, 100.0 * kinds[k] / span))
    print("  per layer, mean clk per CTA (layer 0 input conv, 1..%d tower, %d heads):" % (nl, nl + 1))
    for k, name in ((FULL, "full"), (ACT0, "act0"), (ACT1, "act1"), (GAP, "gap")):
        vals = [per_layer[k][layer] / len(ctas) for layer in range(nl + 2)]
        print("    %-5s %s" % (name, " ".join("%.0f" % v for v in vals)))
    # SMs with two leaders: time in which neither pair has an MMA queued
    by_sm = defaultdict(list)
    for c in ctas:
        by_sm[c[0]].append(c)
    both, tot, sms = 0, 0, 0
    for sm, cs in by_sm.items():
        if len(cs) != 2:
            continue
        lo, hi = min(c[1] for c in cs), max(c[2] for c in cs)
        idle = []
        for _, t_start, t_end, r in cs:
            iv = [[lo, t_start], [t_end, hi]]
            for code, t0, t1 in r:
                if (int(code) & 255) in (GAP, UNIT_GAP):
                    iv.append([int(t0), int(t1)])
            idle.append(merge(iv))
        both += overlap(idle[0], idle[1])
        tot += hi - lo
        sms += 1
    hist = defaultdict(int)
    for cs in by_sm.values():
        hist[len(cs)] += 1
    print("  SMs by leader count %s" % dict(sorted(hist.items())))
    if sms:
        print("  SMs with both leaders: %d; both pairs with nothing queued (layer and unit gaps, ramp, tail): %.2f %% of SM span"
              % (sms, 100.0 * both / tot))


def main():
    sizes = [int(a) for a in sys.argv[1:]] or [1776, 2048]
    ctx = az.Context(0)
    network = model.Network.random_init(seed=0)
    net.load_weights(ctx, network)
    nl = network.blocks * 2
    lib = _native.lib()
    prof = lib.az_net_pair_profile
    prof.restype, prof.argtypes = C.c_int, [C.c_void_p, C.c_void_p, C.c_int]
    dev = torch.device("cuda:0")
    stream = torch.cuda.ExternalStream(ctx.stream)
    for B in sizes:
        feats = (torch.rand(B, 196, device=dev, generator=torch.Generator(dev).manual_seed(B)) < 0.3).float()
        logits, values = torch.empty(B, 833, device=dev), torch.empty(B, device=dev)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        buf = torch.zeros(2 * sms * STRIDE, dtype=torch.int64, device=dev)      # one record block per CTA (two per SM)

        def run(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                _native.check(lib.az_net_forward_dev(ctx.handle, C.c_void_p(feats.data_ptr()), B, net.BF16,
                                                     C.c_void_p(logits.data_ptr()), C.c_void_p(values.data_ptr())))
            e1.record(stream)
            ctx.sync()
            return e0.elapsed_time(e1) / reps
        run(5)
        plain = run(20)
        _native.check(prof(ctx.handle, C.c_void_p(buf.data_ptr()), MAX_REC))
        run(5)
        profiled = run(20)
        _native.check(prof(ctx.handle, None, 0))
        print("B=%d  k_net_pair %.3f ms, profiling instantiation %.3f ms" % (B, plain, profiled))
        analyse(buf.view(-1, STRIDE).cpu().numpy(), nl)


if __name__ == "__main__":
    main()
