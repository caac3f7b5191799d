import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from eirgrid_b200 import _abi, _lib, trainer as T
tr = T.BatchTrainer(65536, seed=99, device=0, asset_dir=os.path.join(ROOT, "tests", "golden", "ireland_map"))
for i in range(6):
    st = tr.step()
    res, traj = tr.fetch_results()
    print("train batch", i, "flagged", st.n_flagged, np.bincount(res["flags"], minlength=16)[:16].tolist()[:9], "max acts/yr", int((traj["n_deficit"].astype(int)+traj["n_additional"]).max()))
w = tr.weights
ctx = tr.ctx
for g in range(4):
    cfg = _abi.RunCfg(replay_best=1)
    res, traj, _, _ = ctx.rollout(w, 4096, seed=99, first_episode=10**7 + g * 4096, cfg=cfg)
    has, b, d = w.best()
    nb, nd = np.array([len(x) for x in b]), np.array([len(x) for x in d])
    st = w.update(res, traj, replay_best=True, rng_seed=99)
    print("replay gen", g, "flags hist", np.bincount(res["flags"], minlength=16)[:9].tolist(), "best list max", int(nb.max()), "deficit list max", int(nd.max()), "improved", st.n_improvements, "flagged", st.n_flagged)
