"""The fused pyramid kernel alone: B VGA frames (4 levels) per launch from device memory (svob200_frame_bind), two alternating
input batches; and a digest of every level of a few images at three frame sizes, to compare library builds (SVOB200_LIB) bit for bit.
   python tools/pyr_probe.py [batch] [digest.npz]"""
import sys, os, ctypes as C, hashlib
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from android_svo_b200 import capi
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
ctx = capi.Context(0)
V = C.c_void_p
rng = np.random.default_rng(1)
if len(sys.argv) > 2:
    dig = {}
    for (w, h, nl, b, modes) in ((640, 480, 4, 96, None), (752, 480, 5, 80, None), (1920, 1080, 5, 64, None), (640, 480, 4, 70, [0, 0, 0]), (640, 480, 3, 65, [1, 0])):
        imgs = rng.integers(0, 256, (b, h, w), dtype=np.uint8)
        d = ctx.dev_alloc(b * w * h)
        ctx.dev_upload(d, imgs)
        ctx.frame_create(7, b, w, h, nl)
        ctx.frame_bind(7, d, w, round_modes=modes)
        ctx.sync()
        for im in (0, 1, b // 2, b - 1):
            for l in range(1, nl):
                dig["%dx%d_%d_%s_im%d_l%d" % (w, h, nl, "d" if modes is None else "".join(map(str, modes)), im, l)] = ctx.frame_download(7, im, l)
        ctx.frame_release(7)
        ctx.dev_free(d)
    np.savez(sys.argv[2], **dig)
    print("digest of %d level images written" % len(dig))
w, h, nl = 640, 480, 4
img = rng.integers(0, 256, (h, w), dtype=np.uint8)
d = [ctx.dev_alloc(B * w * h) for _ in range(2)]
host = np.ascontiguousarray(np.broadcast_to(img, (64, h, w)))
for p in d:
    for k in range(B // 64):
        ctx.dev_upload(p + k * 64 * w * h, host)
ctx.frame_create(1, B, w, h, nl)
def once(k):
    ctx._ck(ctx.L.svob200_frame_bind(ctx.h, 1, V(d[k & 1]), w, None))
for k in range(5):
    once(k)
ctx.sync()
best = []
for rep in range(5):
    ctx.timer_start()
    for k in range(20):
        once(k)
    best.append(ctx.timer_stop_ms() / 20)
alg = B * (w * h + sum((w >> l) * (h >> l) for l in range(1, nl)))
ms = float(np.median(best))
print("%s: pyramid alone %.4f ms per %d frames (min %.4f), %.0f GB/s algorithmic" % (os.environ.get("SVOB200_LIB", "base").split("/")[-1], ms, B, min(best), alg / ms / 1e6))
