#!/usr/bin/env python
"""GPU tool for compute-sanitizer: a few clicks through the whole interactive path (resident image, announced click,
tensor-core conv1_1, 128-column split-K pairs) at 64x64 -- small enough for memcheck / racecheck to finish in
minutes.  Plan options given as opt:val pairs apply to the context.

    compute-sanitizer --tool memcheck python tools/sanitizer_click.py [size] [opt:val,...]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from interactive_deep_colorization_b200 import colorize_image as CI  # noqa: E402
from oracle import synth  # noqa: E402
from tests import util  # noqa: E402

X = int(sys.argv[1]) if len(sys.argv) > 1 else 64
EXTRA = {kv.split(":")[0]: int(kv.split(":")[1]) for kv in (sys.argv[2].split(",") if len(sys.argv) > 2 else []) if kv}
sd = synth.torch_state_dict(1234)
L, ab, m = synth.synthetic_batch(1, X, seed=0, max_hints=0)
ab, m = ab.copy(), m.copy()
ctx = util.make_ctx(sd, X, X, max_n=1, dist=True, options=EXTRA)
ctx.set_dist_resident(True)
buf = ctx.click_buffers(1)
buf["L_mc"][...] = L
ctx.set_image(buf["L_mc"])
rs = np.random.RandomState(0)
for i in range(3):
    loc = rs.randint(8, X - 8, 2)
    CI.put_point(ab[0], m[0], loc, 2, rs.uniform(-80, 80, 2))
    buf["ab"][...] = ab; buf["mask"][...] = m
    y4, x4 = int(loc[0]) // 4, int(loc[1]) // 4
    ctx.set_click(0, y4, x4, 5)
    ctx.forward_host(None, buf["ab"], buf["mask"], 0.5, want_rgb=True, want_abq=True, out_ab=buf["out_ab"],
                     out_rgb=buf["out_rgb"], out_abq=buf["out_abq"])
    pmf = ctx.fetch_dist(0, y4, x4)
    ctx.ab_reccs(0, y4, x4, K=5)
ctx.close()
print("sanitizer_click: %dx%d, 3 clicks done; pmf sum %.6f" % (X, X, float(pmf.sum())))
