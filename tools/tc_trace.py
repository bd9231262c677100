"""Timeline of CTA 0 of a tcgen05 kernel (clock64 per warp role).

    python tools/tc_trace.py linear|ffn

Needs a variant build with the trace hooks compiled in:

    make -C fb-bev_b200/csrc OBJDIR=../../build/var_TRACE \\
         OUT=../../build/var_TRACE/libfbbev_b200.so EXTRA=-DTC_TRACE
    FBBEV_LIB=$PWD/build/var_TRACE/libfbbev_b200.so python tools/tc_trace.py ffn

Tags of linear_tf32_kernel (40000 x 80 -> 80 + residual + LayerNorm): 1 set-up
done; 100+w loads of round w issued; 200+i / 300+i stage of item i free /
filled; 400+i MMA sees item i; 500+t accumulator of tile t committed;
600..1000+t epilogue of tile t (wait, accumulator ready, pass 1 done,
normalised, stored); 2 kernel end.

Tags of ffn_tf32_kernel (40000 x 80 -> 320 -> 80 + residual + LayerNorm): 1
set-up done; 100/110/120+t loader of tile t (loads issued, X buffer free,
filled); 1000+i producer issues weight stage i; 200/210/220+t MMA warp (tile
start, X ready, all issued); 2000+i MMA sees weight stage i, 3000+i its hidden
K-block too; 4000/5000/6000+u convert of K-block u (chunk ready, lo stage free,
done); 300/310/320+t finish (slab free, Y ready, stored); 330 all stored.
"""
import ctypes
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from fbbev_b200 import _lib  # noqa: E402
from fbbev_b200.ops.linear import ffn_fused, linear_fused  # noqa: E402

KERNELS = {"linear": 0, "ffn": 1}
ROLES, CAP = 5, 200  # kTraceRoles, kTraceCap (tc5.cuh)
CLOCK_GHZ = 1.965    # B200 SM clock the timeline is converted with


def run(kernel):
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    m, e, h = 40000, 80, 320
    x = torch.randn(m, e, device=dev, generator=g)
    gm = torch.ones(e, device=dev)
    bt = torch.zeros(e, device=dev)
    with torch.no_grad():
        if kernel == "linear":
            w = torch.randn(e, e, device=dev, generator=g) / e ** .5
            b = torch.randn(e, device=dev, generator=g)
            r = torch.randn(m, e, device=dev, generator=g)
            for _ in range(4):
                linear_fused(x, w, b, residual=r, ln_weight=gm, ln_bias=bt)
        else:
            w1 = torch.randn(h, e, device=dev, generator=g) / e ** .5
            w2 = torch.randn(e, h, device=dev, generator=g) / h ** .5
            b1 = torch.randn(h, device=dev, generator=g)
            b2 = torch.randn(e, device=dev, generator=g)
            for _ in range(4):
                ffn_fused(x, w1, b1, w2, b2, residual=x, ln_weight=gm, ln_bias=bt)
        torch.cuda.synchronize()


def main():
    if len(sys.argv) != 2 or sys.argv[1] not in KERNELS:
        sys.exit("usage: tc_trace.py linear|ffn")
    kernel = sys.argv[1]
    run(kernel)
    buf = (ctypes.c_longlong * (ROLES * 2 * CAP))()
    cnt = (ctypes.c_int * ROLES)()
    fn = _lib.lib().fbbev_debug_tc_trace
    fn.restype = ctypes.c_int
    fn(KERNELS[kernel], buf, cnt)
    ev = sorted((buf[r * 2 * CAP + 2 * i + 1], buf[r * 2 * CAP + 2 * i])
                for r in range(ROLES) for i in range(min(cnt[r], CAP)))
    if not ev:
        sys.exit("no trace records: is the library a -DTC_TRACE build?")
    t0 = ev[0][0]
    for t, tag in ev:
        print(f"{(t - t0) / (CLOCK_GHZ * 1e3):8.2f} us  tag {tag}")


if __name__ == "__main__":
    main()
