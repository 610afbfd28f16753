"""BASELINE config 4a: 4096x4096 RGBA8 lossless Modular, decode stage times through LoadImage (CUDA events)."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, pkgload, oracle_py as O
P = pkgload.load()
n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
img = O.synthetic_image(n, n, seed=0, channels=4)
t = time.time(); data = O.encode(img, lossless=1, threads=os.cpu_count() or 1); print("oracle encode %.1f s, %.3f bpp" % (time.time() - t, len(data) * 8 / n / n))
for i in range(3):
    image = P.DecoderImage(); t = time.time(); P.JpegXLNative.LoadImage(data, image); dt = time.time() - t
    print("LoadImage wall %.1f ms" % (dt * 1e3), {k: round(v, 2) for k, v in P.last_stage_times().items()})
ld = image.layer_data
print("bit-exact:", bool(np.array_equal(ld.color, img[..., :3]) and np.array_equal(ld.transparency, img[..., 3])))
