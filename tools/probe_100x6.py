#!/usr/bin/env python
"""Why is 100 trees x depth 6 slower per tree than 30 x 6 and 100 x 10?  (tree-count / layout / pipe probes)"""
import json, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from quickchem_b200 import capi, synth  # noqa: E402

x = synth.quick_features(synth.raw_fields(180))
d = capi.DMatrix(x)
out = capi.DeviceArray(x.shape[0])


def t(b, lim=0, iters=5):
    for _ in range(2):
        b.predict_device(d, out, ntree_limit=lim)
    capi.synchronize(); capi.timer_start()
    for _ in range(iters):
        b.predict_device(d, out, ntree_limit=lim)
    return capi.timer_stop() / iters


for m in ("100x6", "100x10", "30x6"):
    b = capi.Booster(os.path.join(ROOT, "build", f"oh_booster_{m}.model"))
    for name, val in (("duo", -1), ("duo", 0)):
        capi.set_param(name, val)
        for lim in (10, 30, 60, 100):
            if lim > b.info().num_trees:
                continue
            print(json.dumps(dict(model=m, duo=val, ntree_limit=lim, ms=round(t(b, lim), 4), kernel=capi.last_predict_kernel())), flush=True)
    capi.set_param("duo", -1)
    b.free()
