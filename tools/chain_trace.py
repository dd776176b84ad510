"""clock64 timeline of CTA 0 of the LAST chained GEMM launch of an encode (mlp1 -> mlp2 -> final_proj of
signature layer 6; 2 + 1 + 1 tiles) - MMA issue, accumulator ready, epilogue done, op-boundary waits."""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from linetr_b200 import LineBatch, LineTransformer, PairEngine, _native as N, synthetic as syn

lib = N.load()
dev = torch.device("cuda", 0)
sd = syn.make_state_dict(0, 1)
m = LineTransformer({"mode": "train"})
m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
m = m.eval().to(dev)
eng = PairEngine(m, dev)
b = LineBatch.from_images([syn.make_image_inputs(i, 128, 21) for i in range(128)]).to(dev)
for _ in range(3):
    eng.encode(b)
torch.cuda.synchronize()
sel = int(os.environ.get("LTR_TRACE_CHAIN", "7"))   # 0 = line chain, 1..6 = mlp1 -> mlp2 -> qkv of the next layer, 7 = ... -> final
lib.ltr_debug_trace_arm(100 + sel)
eng.encode(b)
torch.cuda.synchronize()
buf = (C.c_uint64 * 128)()
lib.ltr_debug_trace_read(buf)
lib.ltr_debug_trace_arm(0)
t0 = buf[110]
print(f"chain launch {sel}  t0 = after pdl_wait")
names = {0: ["fc+LN (K256)", "w1 nb0 (K256)", "w1 nb1 (K256)", "w2+LN (K512)", "qkv nb0 (K256)", "qkv nb1", "qkv nb2"],
         7: ["mlp1 nb0 (K512)", "mlp1 nb1 (K512)", "mlp2 (K512)", "final (K256, norm)"]}.get(
    sel, ["mlp1 nb0 (K512)", "mlp1 nb1 (K512)", "mlp2 (K512)", "qkv nb0 (K256)", "qkv nb1 (K256)", "qkv nb2 (K256)"])
for tl, nm in enumerate(names):
    a = [buf[40 + tl * 4 + i] for i in range(4)]
    af = buf[80 + tl]
    if not a[1]:
        continue
    print(f"{nm:20s} acc_empty ok +{a[0]-t0:7d} | first operands +{a[1]-t0:7d} | MMAs committed +{a[2]-t0:7d} | "
          f"epilogue sees acc +{af-t0:7d} | epilogue done +{a[3]-t0:7d}   (mma loop {a[2]-a[1]}, epilogue {a[3]-af})")
if buf[0]:
    print("first tile, warp 2, per k-block: [start -> accumulator chunk loaded -> bias/act/split done -> staging tile free]")
    for k in range(4):
        a = [buf[k * 4 + i] - t0 for i in range(4)]
        print(f"  k-block {k}: start +{a[0]}  tmem_ld {a[1] - a[0]}  math {a[2] - a[1]}  wait tile_free {a[3] - a[2]}")
print("store warp, hand-over processed (+cycles):", [int(buf[16 + i] - t0) for i in range(24) if buf[16 + i]])
print("third tile, per epilogue warp: accumulator seen", [int(buf[112 + i] - t0) for i in range(8)], " first k-block handed over", [int(buf[90 + i] - t0) for i in range(8)])
for d in (1, 2, 3):
    if buf[100 + d]:
        print(f"producer: op boundary {d} passed at +{buf[100 + d] - t0}")
print(f"kernel end (CTA 0 thread 0) +{buf[111] - t0}")
