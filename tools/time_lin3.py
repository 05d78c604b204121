"""Times the small fp32 linear family (forward, data gradient, weight gradient) at the decoder's shapes.
  python tools/time_lin3.py"""
import sys

import torch

sys.path.insert(0, ".")
from helping_hand_for_egocentric_videos_b200 import ops  # noqa: E402


def gpu_us(fn, iters=30, warm=5):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def main():
    for R, N, K in [(832, 256, 256), (832, 512, 256), (832, 2048, 256), (832, 256, 2048), (19968, 256, 256), (4992, 256, 256),
                    (65, 256, 256), (19968, 4, 256)]:
        x = torch.randn(R, K, device="cuda")
        w = torch.randn(N, K, device="cuda") / K ** 0.5
        b = torch.randn(N, device="cuda")
        dy = torch.randn(R, N, device="cuda")
        y = torch.relu(torch.nn.functional.linear(x, w, b))
        f = gpu_us(lambda: ops.linear_f32(x, w, b, act=1))
        dg = gpu_us(lambda: ops.linear_f32_backward(dy, y, 1, w, x, need_dw=False))
        wg = gpu_us(lambda: ops.linear_f32_backward(dy, y, 1, w, x, need_dx=False))
        t = gpu_us(lambda: torch.nn.functional.linear(x, w, b))
        print("R=%5d N=%4d K=%4d  fwd %7.1f us  dgrad %7.1f us  wgrad %7.1f us   (torch fp32 linear fwd %7.1f us)" % (R, N, K, f, dg, wg, t))


if __name__ == "__main__":
    main()
