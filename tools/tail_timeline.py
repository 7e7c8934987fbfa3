"""SM-clock timeline of one work item of the block-tail kernel in the form the forward runs (vitocm_block_tail_folded with stamps; layout: TailArgs::timeline in
csrc/block_tail_sm100.cuh) + its launch time.  Usage: python tools/tail_timeline.py [tiles] [precision]"""
import os
import sys
import ctypes as C

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import vitocm_b200 as vob  # noqa: E402
from gpu_util import make_engine, ptr, check, cur_stream  # noqa: E402

tiles = int(sys.argv[1]) if len(sys.argv) > 1 else 175
precision = int(sys.argv[2]) if len(sys.argv) > 2 else 2
M, D, Hd = tiles * 785, 384, 1536
dt = torch.float16 if precision == 2 else torch.bfloat16
lib = vob._lib.load_library()
eng = make_engine(embed_dim=D, heads=6, hidden=Hd, precision=precision)
g = torch.Generator(device="cuda").manual_seed(0)
rnd = lambda *s, sc=1.0: torch.randn(*s, device="cuda", generator=g) * sc
ctx = rnd(M, D).to(dt)
Wp, W1, W2 = rnd(D, D, sc=0.05).to(dt), rnd(Hd, D, sc=0.06).to(dt), rnd(D, Hd, sc=0.03).to(dt)
bp, b1, b2 = rnd(D, sc=0.1), rnd(Hd, sc=0.2), rnd(D, sc=0.1)
g2, be2, gn, ben = rnd(D, sc=0.1) + 1, rnd(D, sc=0.1), rnd(D, sc=0.1) + 1, rnd(D, sc=0.1)
x = rnd(M, D)
xn = torch.zeros(M, 2 * D, device="cuda", dtype=dt)
with_qkv = int(sys.argv[3]) if len(sys.argv) > 3 else 1   # 1: the kernel also computes the next block's QKV projection
Wq, bq = rnd(3 * D, D, sc=0.05).to(dt), rnd(3 * D, sc=0.1)
qkv = torch.zeros(M, 3 * D, device="cuda", dtype=dt)
wq_p, bq_p, qkv_p = (ptr(Wq), ptr(bq), ptr(qkv)) if with_qkv else (None, None, None)
stamps = torch.zeros(64, device="cuda", dtype=torch.int64)


def run(st):
    check(lib.vitocm_block_tail_folded(eng, ptr(ctx), ctx.stride(0), ptr(Wp), Wp.stride(0), ptr(bp), ptr(g2), ptr(be2), ptr(W1), W1.stride(0), ptr(W2),
                                W2.stride(0), M, D, Hd, ptr(b1), ptr(b2), ptr(x), ptr(gn), ptr(ben), ptr(xn), xn.stride(0), wq_p, Wq.stride(0), bq_p, qkv_p, qkv.stride(0), st, cur_stream()))


for _ in range(3):
    run(None)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 10
e0.record()
for _ in range(n):
    run(None)
e1.record()
torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 1e3 / n
flop = 2.0 * M * D * (D + 2 * Hd + (3 * D if with_qkv else 0))
print(f"block tail: tiles={tiles} M={M} precision={precision} with_qkv={with_qkv}: {us:.1f} us/launch, {flop / us / 1e6:.1f} TFLOP/s")
run(ptr(stamps))
torch.cuda.synchronize()
s = stamps.cpu().tolist()
t0 = s[60]
rel = lambda i: (s[i] - t0) & 0xFFFFFFFF if s[i] else -1
print("MMA thread : CTX landed=0  proj issued=%d  ep1 seen=%d" % (rel(56), rel(59)))
print("epilogue w0: proj complete=%d  ep1 pass1=%d  ep1 handed=%d" % (rel(57), rel(58), rel(55)))
print("epilogue w0: ep1 steps=%d %d %d  combined=%d" % (rel(15), rel(16), rel(17), rel(18)))
for c in range(0, 5, 2):
    print(" chunk %2d: fc1 complete=%d gelu done=%d handed=%d | mma: fc1 issued=%d gelu seen=%d" % (c, rel(3 * c), rel(3 * c + 1), rel(3 * c + 2), rel(36 + 2 * c), rel(36 + 2 * c + 1)))
print("epilogue w0: OUT complete=%d  ep2 stats=%d  steps stored=%d %d %d  stores read=%d  ep2 done=%d" % (rel(61), rel(54), rel(20), rel(21), rel(22), rel(24), rel(62)))
if with_qkv:
    print("next norm1 rows: epilogue w0 handed over=%d  MMA thread saw xn_ready=%d" % (rel(19), rel(63)))
    print("QKV chunks, epilogue w0 (its group's first two): " + " | ".join("complete=%d packed=%d staging free=%d stored=%d" % tuple(rel(25 + 4 * k + e) for e in range(4)) for k in range(2)))
    print("QKV chunks, MMA thread issued: " + " ".join(str(rel(46 + c)) for c in range(8)))
if int(os.environ.get("VITOCM_TAIL_DEBUG", "0")) & 16:
    names = ["accumulator complete", "in registers", "gelu done", "gelu buffer free", "stored+fenced", "handed"]
    print("chunk 4 (group 0, warp 0): " + " ".join("%s=%d" % (n, rel(25 + i)) for i, n in enumerate(names)))
    print("chunk 5 (group 1, warp 8): " + " ".join("%s=%d" % (n, rel(46 + i)) for i, n in enumerate(names)))
    print("MMA thread: gelu(4) seen=%d fc2(4) issued=%d | fc1(6): accumulator free=%d issued=%d | gelu(5) seen=%d fc2(5) issued=%d | fc1(7): accumulator free=%d issued=%d"
          % (rel(45), rel(33), rel(31), rel(32), rel(34), rel(53), rel(35), rel(52)))
