import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O
from workloads import bench_key_bytes, bench_key_hashes, bench_requests, zipf_ids

BENCH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")


def test_vectorised_bench_key_hashes_match_scalar():
    ids = np.array([0, 1, 9, 10, 42, 999_999_999, 123_456_789, 100_000_000 - 1] + list(np.random.default_rng(1).integers(0, 10**8, 200)))
    b = bench_key_bytes(ids)
    xx, fv = bench_key_hashes(ids)
    for j, i in enumerate(ids.tolist()):
        s = f"bench_k{i:09d}".encode()
        assert b[j].tobytes() == s
        assert int(xx[j]) == O.xxh64(s) and int(fv[j]) == O.fnv1_64(s)
    r = bench_requests(ids, 1_700_000_000_000)
    assert np.array_equal(r["algorithm"], ids & 1) and np.all(r["limit"] == 100)


def test_zipf_ids_shape():
    rng = np.random.default_rng(0)
    ids = zipf_ids(rng, 65536, 100_000_000, 1.1)
    assert ids.min() >= 0 and ids.max() < 100_000_000
    _, counts = np.unique(ids, return_counts=True)
    top = np.sort(counts)[::-1]
    # SURVEY.md §7: the top key draws about 11 % of a batch at K = 1e8, s = 1.1
    assert 0.07 < top[0] / 65536 < 0.15
    assert top[:100].sum() / 65536 > 0.35


def test_bench_parses_ncu_rows_of_templated_kernels(tmp_path):
    """bench.py's roofline.traffic leg: kernel names come out of ncu as `void k_rank<0>(BatchArgs)` / `gub::k_rank<1>(...)`; the parser
    keys them as k_rank etc.  Fed with the committed launch list of the final kernels, metric names swapped for the DRAM counters."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bench = _bench_module()
    src = open(os.path.join(root, "profiles", "r02_ncu_launches_final.csv")).read()
    both = src.replace("gpu__time_duration.sum", "dram__bytes_read.sum").replace('"ns"', '"byte"')
    extra = [ln.replace("dram__bytes_read.sum", "dram__bytes_write.sum") for ln in both.splitlines() if "dram__bytes_read.sum" in ln and "Metric Name" not in ln]
    p = tmp_path / "traffic.csv"
    p.write_text(both + "\n".join(extra) + "\n")
    out = bench.parse_traffic_csv(str(p))
    assert set(out) == {"k_group", "k_rank", "k_eval", "k_finish"}
    assert all(v["launches"] == 8 and v["dram_read_bytes_per_launch"] > 0 and v["dram_write_bytes_per_launch"] == v["dram_read_bytes_per_launch"] for v in out.values())


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def _run_bench_dump(out_dir, *args):
    """bench.py with --dump-outputs out_dir: (its JSON line, the dumped arrays by response field)."""
    res = subprocess.run([sys.executable, BENCH, *args, "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    return line, {f: np.load(os.path.join(out_dir, f + ".npy")) for f in O.HRESP_DTYPE.names}


def test_bench_reference_arm_dumps_its_last_step(tmp_path):
    """bench.py --impl reference times exactly --steps steps, and --dump-outputs writes the responses of the last one as float64
    arrays that are the same from run to run."""
    args = ("--impl", "reference", "--keys", "1000000", "--cpu-keys", "1000000", "--warmup", "1")
    line, a = _run_bench_dump(tmp_path / "a", *args, "--steps", "3")
    assert line["steps"] == 3
    _, b = _run_bench_dump(tmp_path / "b", *args, "--steps", "3")
    for f in O.HRESP_DTYPE.names:
        assert a[f].dtype == np.float64 and a[f].shape == (65536,), f
        assert np.array_equal(a[f], b[f]), f
    assert set(np.unique(a["status"])) <= {0.0, 1.0} and np.all(a["limit"] == 100)


@pytest.mark.gpu
def test_bench_dump_is_the_oracles_last_step(tmp_path):
    """bench.py --dump-outputs on the GPU arm at 1 M keys: the dumped responses are those the oracle gives for the last timed
    batch after the same fill, warm-up and timed batches in the same order."""
    keys, pool_n, warmup, steps = 1_000_000, 4, 2, 3
    line, got = _run_bench_dump(tmp_path, "--keys", str(keys), "--pool", str(pool_n), "--warmup", str(warmup), "--steps", str(steps),
                                "--no-cpu-baseline", "--no-traffic", "--no-e2e")
    assert line["steps"] == steps
    bench = _bench_module()
    rng = np.random.default_rng(0xB200 + 3)
    batches = [bench.gen_batch(rng, bench.BATCH, keys, bench.T0 + 1 + b, 1.1, O.HREQ_DTYPE)[0] for b in range(pool_n)]
    pool = O.Pool(workers=4, cache_size=10_000_000, now_ms=bench.T0)
    pool.submit_hashed(bench_requests(np.arange(keys, dtype=np.int64), bench.T0))
    for b in range(warmup + steps):
        pool.set_now(bench.T0 + 1 + b)
        want = pool.submit_hashed(batches[b % pool_n])
    for f in O.HRESP_DTYPE.names:
        assert np.array_equal(got[f], want[f].astype(np.float64)), f"{f}: {int((got[f] != want[f]).sum())} of {len(want)} differ"
