"""Throughput of the network kernel alone (positions/s, tensor-roofline fraction) -- ch5 net, batch in HBM."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "reversi-alpha-zero_b200"))
FLOP_PER_POS = 2 * 755_343_616


def run(n=32768, iters=5, warmup=2, res_blocks=10):
    import torch
    from reversi_zero_b200.agent import model as M
    from reversi_zero_b200 import net as N, device as D
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    mc = M.ModelConfig(res_layer_num=res_blocks)
    flop = 2 * (64 * 256 * 18 + res_blocks * 2 * 64 * 256 * 2304 + 64 * 3 * 256 + 128 * 64 + 64 * 256 + 256)
    net = N.Net(mc)
    net.load_weights(M.build_random_weights(mc, 0))
    rng = np.random.default_rng(0)
    a = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64); r = rng.integers(0, 2 ** 64, size=n, dtype=np.uint64)
    d_own, d_en = D.to_device(a & r), D.to_device(a & ~r)
    d_pol, d_val = D.empty(n * 64, np.float32), D.empty(n, np.float32)
    s = torch.cuda.current_stream()
    for _ in range(warmup):
        net.predict_dev(d_own, d_en, d_pol, d_val, n, N.IMPL_TCGEN05, D.stream_ptr(s))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(iters):
        net.predict_dev(d_own, d_en, d_pol, d_val, n, N.IMPL_TCGEN05, D.stream_ptr(s))
    e1.record(s)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    tflops = n * flop / ms / 1e9
    return dict(n=n, res_blocks=res_blocks, flop_per_position=flop, ms=ms, pos_per_s=n / ms * 1e3, tflops=tflops, frac_of_burst_peak=tflops / peaks.get("bf16_tflops", 1590.0),
                frac_of_sustained_peak=tflops / peaks.get("bf16_tflops_sustained", 1400.0))


if __name__ == "__main__":
    # python tools/nn_bench.py [res_blocks] [iters]
    rb = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    for n in (296, 32768):
        r = run(n, iters=iters, res_blocks=rb)
        print(json.dumps(r))
