import sys, os
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import toppra_b200 as ta
from problems import SHORTCUT_SETS
from oracle import oracle as orc
name = "scaled14"
g = np.load(os.path.join(ROOT, "tests", "golden", "shortcut_rows_%s.npz" % name))
gen, args = SHORTCUT_SETS[name]
rows, xb = gen(*args)
B, G, _, R = rows.shape
grid = np.linspace(0, 1, G)
dev = torch.device("cuda:0")
rec, W = ta.engine.alloc_records(B, G, R, dev)
host = np.zeros((B, G, W))
host[:, :, 0:R] = rows[:, :, 0]; host[:, :, R:2 * R] = rows[:, :, 1]; host[:, :, 2 * R:3 * R] = rows[:, :, 2]
host[:, :, 3 * R] = xb[:, :, 0]; host[:, :, 3 * R + 1] = xb[:, :, 1]
rec.copy_(torch.from_numpy(host))
z = torch.zeros(B, dtype=torch.float64, device=dev)
out = ta.engine.scan(rec, R, torch.from_numpy(grid).to(dev), z, z, z, counters=True)
K, sd, u, st, fs = (out[k].cpu().numpy() for k in ("K", "sd", "u", "status", "fail_stage"))
gK = g[name + "_K"]
bad = [i for i in range(B) if not np.array_equal(K[i], gK[i], equal_nan=True)]
print("mismatching paths:", len(bad), bad[:20])
for i in bad[:6]:
    d = np.nonzero(~((K[i] == gK[i]) | (np.isnan(K[i]) & np.isnan(gK[i]))))
    print("path", i, "status gpu/ref", st[i], g[name + "_status"][i], "fail_stage", fs[i], "xb_hi", xb[i, 0, 1])
    for s_, c_ in zip(*d):
        print("   stage", s_, "col", c_, "gpu", repr(K[i, s_, c_]), "ref", repr(gK[i, s_, c_]), "rel", (K[i, s_, c_] - gK[i, s_, c_]) / (abs(gK[i, s_, c_]) + 1e-300))
