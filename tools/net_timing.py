import sys, time, os, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import ataxxzero_b200 as az
from ataxxzero_b200 import model, net, _native
ctx = az.Context(0)
network = model.Network.random_init(seed=0)
t0 = time.perf_counter(); net.load_weights(ctx, network); print("load_weights %.1f ms" % ((time.perf_counter() - t0) * 1e3))
t0 = time.perf_counter(); net.load_weights(ctx, network); print("reload %.1f ms" % ((time.perf_counter() - t0) * 1e3))
lib = _native.lib()
dev = torch.device("cuda:0")
stream = torch.cuda.ExternalStream(ctx.stream)
for B in [int(a) for a in sys.argv[1:]] or (256, 1024, 2048, 4096, 16384):
    feats = (torch.rand(B, 196, device=dev) < 0.3).float()
    logits = torch.empty(B, 833, device=dev); values = torch.empty(B, device=dev)
    torch.cuda.synchronize()
    for mode in (net.BF16,):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for it in range(3):
            _native.check(lib.az_net_forward_dev(ctx.handle, C.c_void_p(feats.data_ptr()), B, mode, C.c_void_p(logits.data_ptr()), C.c_void_p(values.data_ptr())))
        e0.record(stream)
        reps = 10
        for it in range(reps):
            _native.check(lib.az_net_forward_dev(ctx.handle, C.c_void_p(feats.data_ptr()), B, mode, C.c_void_p(logits.data_ptr()), C.c_void_p(values.data_ptr())))
        e1.record(stream); ctx.sync()
        dt = e0.elapsed_time(e1) / reps * 1e-3
        print("tiles=%s B=%d mode=%d %.3f ms  %.1f kpos/s  %.1f TFLOP/s" % (os.environ.get("AZ_NET_TILES", "default"), B, mode, dt * 1e3, B / dt / 1e3, B * 347.49e6 / dt / 1e12), flush=True)
