import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from rebvo_b200 import capi, synth
cam = synth.EUROC
seq = synth.Sequence(w=cam["w"], h=cam["h"], seed=7, zf=cam["zfx"])
B = 64
ts, fr = seq.frames(B)
pl = capi.Pipeline(capi.default_params(cam), max_batch=B)
pl.push(fr, ts)
names = {4: "rgb2gray", 0: "rowscan_plain", 1: "rowscan_avg", 2: "colscan", 3: "blur_dog"}
for nimg in (4, 8, 16, 32, 64):
    out = []
    for pid in (4, 0, 1, 2, 3):
        ms, by = pl.bench_pass(pid, nimg, 20)
        out.append("%s %.1fus/img %.0fGB/s" % (names[pid], 1e3 * ms / nimg, by / ms / 1e6))
    print("nimg %2d: " % nimg + " | ".join(out))
