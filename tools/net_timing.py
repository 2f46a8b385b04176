"""Kernel time of the bf16 net passes, CUDA events over repeated launches after warm-up.

    python tools/net_timing.py [plain|sym8|cache] [batch sizes...]

plain: az_net_forward_dev over host feature planes (default sizes 256 .. 16384).  sym8: the symmetry ensemble over positions
(default 1, 16, 2S+1, 6S+5; S = SM count); the time includes its feature upload and output download.  cache: the speculative
search's pass through az_net_forward_pool_dev -- position input, values, softmax numerators and their sums through an output
map (default 1, 13, R+1, 2R+3 requests; R = 4S)."""
import sys, time, os, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import ataxxzero_b200 as az
from ataxxzero_b200 import model, net, rules, _native
kind = sys.argv[1] if len(sys.argv) > 1 and sys.argv[1] in ("plain", "sym8", "cache") else "plain"
sizes = [int(a) for a in sys.argv[1:] if a.isdigit()]
ctx = az.Context(0)
network = model.Network.random_init(seed=0)
t0 = time.perf_counter(); net.load_weights(ctx, network); print("load_weights %.1f ms" % ((time.perf_counter() - t0) * 1e3))
t0 = time.perf_counter(); net.load_weights(ctx, network); print("reload %.1f ms" % ((time.perf_counter() - t0) * 1e3))
lib = _native.lib()
dev = torch.device("cuda:0")
stream = torch.cuda.ExternalStream(ctx.stream)
S = torch.cuda.get_device_properties(0).multi_processor_count
if not sizes:
    sizes = {"plain": [256, 1024, 2048, 4096, 16384], "sym8": [1, 16, 2 * S + 1, 6 * S + 5], "cache": [1, 13, 4 * S + 1, 8 * S + 3]}[kind]
pool_fwd = lib.az_net_forward_pool_dev
pool_fwd.restype = C.c_int
pool_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5


def ptr(t):
    return C.c_void_p(t.data_ptr())


for B in sizes:
    if kind == "plain":
        feats = (torch.rand(B, 196, device=dev) < 0.3).float()
        logits = torch.empty(B, 833, device=dev); values = torch.empty(B, device=dev)
        call = lambda: _native.check(lib.az_net_forward_dev(ctx.handle, ptr(feats), B, net.BF16, ptr(logits), ptr(values)))
    elif kind == "sym8":
        planes = (np.random.default_rng(B).random((B, 7, 7, 4)) < 0.3).astype(np.float32)
        call = lambda: net.evaluate_symmetric(ctx, planes, net.BF16)
    else:
        pos = rules.positions_array([rules.set_board(rules.START_FEN)] * B)
        d_pos = torch.from_numpy(pos.view(np.uint8).copy()).to(dev)
        rows = 2 * B + 1
        d_map = torch.from_numpy(np.random.default_rng(B).permutation(2 * B)[:B].astype(np.int32)).to(dev)
        exps = torch.empty(rows, 833, dtype=torch.float64, device=dev)
        totals = torch.empty(rows, dtype=torch.float64, device=dev); values = torch.empty(rows, device=dev)
        call = lambda: _native.check(pool_fwd(ctx.handle, ptr(d_pos), B, None, net.BF16, 0, None, ptr(values), ptr(exps), ptr(totals), ptr(d_map)))
    torch.cuda.synchronize()
    for it in range(3):
        call()
    ctx.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record(stream)
    for it in range(reps):
        call()
    e1.record(stream); ctx.sync()
    dt = e0.elapsed_time(e1) / reps * 1e-3
    print("%s B=%d %.4f ms  %.1f kpos/s" % (kind, B, dt * 1e3, B / dt / 1e3), flush=True)
