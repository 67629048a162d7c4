import os, sys, importlib.util
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]
import numpy as np
import oracle_py as O
from global_model import OracleCluster
from workloads import bench_requests, T0
spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py")); bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
W, n_keys, per_step, steps, pool_n = 2, 1000000, 16384, 2000, 32
hot = n_keys // 100
rng = [np.random.default_rng(100 + r) for r in range(W)]
pool = [[bench.gen_batch(rng[r], per_step, n_keys, T0 + 1 + k, 1.1, O.HREQ_DTYPE, global_hot=hot)[0] for k in range(pool_n)] for r in range(W)]
def run(consistent):
    cl = OracleCluster(W, T0)
    for b in range(10):
        cl.step([pool[r][b % pool_n] for r in range(W)], T0 + 1 + b)
    cl.tick(T0 + 1 + (10 % pool_n) if consistent else T0 + 1 + 10)
    for b in range(10, 10 + 150):   # (150 steps of the 2000 the bench runs: the buckets' own clock does not advance anyway)
        cl.step([pool[r][b % pool_n] for r in range(W)], T0 + 1 + b)
    end = 10 + steps
    tnow = T0 + 1 + (end % pool_n) if consistent else T0 + 1 + end
    cl.tick(tnow); cl.tick(tnow)
    q = bench_requests(np.arange(hot, dtype=np.int64), tnow)
    q["hits"] = 0; q["behavior"] = np.uint32(O.GLOBAL | O.REQ_IS_OWNER)
    outs = cl.step([q.copy() for _ in range(W)], T0 + 1 + end)
    tok = q["algorithm"] == 0
    d = np.abs(outs[0]["remaining"].astype(np.int64) - outs[1]["remaining"].astype(np.int64))
    print("consistent clocks" if consistent else "bench r02 (query / tick 2 s ahead of the requests' created_at)",
          "| token differing", int(((outs[0]["remaining"] != outs[1]["remaining"]) | (outs[0]["status"] != outs[1]["status"]))[tok].sum()),
          "| leaky max diff", int(d[~tok].max()), "differing", int((d[~tok] > 0).sum()), "of", int((~tok).sum()))
run(False); run(True)
