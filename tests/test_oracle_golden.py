"""Pins the CPU oracle (oracle/gub_oracle.c) against the reference's own golden vectors (SURVEY.md §8c).

CPU-only: runs in `pytest -m "not gpu"`.
"""
import calendar
import ctypes as C
import os

import numpy as np
import pytest

import oracle_py as O
from golden import reference_kat as K
from kat_player import play_missing_fields, play_scenario


def _ms(t):
    y, mo, d, h, mi, s, frac = t
    return calendar.timegm((y, mo, d, h, mi, s)) * 1000


# ---- hashes (third-party in the reference: OneOfOne/xxhash, segmentio/fasthash, crypto/md5) ----------------
def test_xxh64_vectors():
    for data, want in K.XXH64_VECTORS:
        assert O.xxh64(data) == want, data


def test_xxh64_against_python_xxhash():
    """python-xxhash's digests of these inputs are stored in tests/golden/xxh64_python_xxhash.npy (columns: seed 0, seed 12345),
    so the comparison runs without the package; where it is installed the stored digests are checked against it too."""
    try:
        import xxhash
    except ImportError:
        xxhash = None
    want = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "xxh64_python_xxhash.npy"))
    rng = np.random.default_rng(1)
    for j, n in enumerate(list(range(0, 70)) + [127, 128, 129, 1000]):
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert O.xxh64(b) == int(want[j, 0])
        assert O.xxh64(b, 12345) == int(want[j, 1])
        if xxhash is not None:
            assert int(want[j, 0]) == xxhash.xxh64(b, seed=0).intdigest()
            assert int(want[j, 1]) == xxhash.xxh64(b, seed=12345).intdigest()


def test_fnv_md5_vectors():
    import hashlib
    for data, want in K.FNV1_VECTORS:
        assert O.fnv1_64(data) == want
    for data, want in K.FNV1A_VECTORS:
        assert O.fnv1a_64(data) == want
    for data, want in K.MD5_VECTORS:
        assert O.md5_hex(data) == want
    rng = np.random.default_rng(2)
    for n in [0, 1, 55, 56, 57, 63, 64, 65, 119, 120, 121, 200]:
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert O.md5_hex(b) == hashlib.md5(b).hexdigest()


# ---- replicated_hash_test.go:56-101 ------------------------------------------------------------------------
@pytest.mark.parametrize("kind,name", [(0, "fnv1"), (1, "fnv1a")])
def test_ring_distribution(kind, name):
    ring = O.Ring(kind, 512)
    for h in K.RING_HOSTS:
        ring.add(h)
    dist = {h: 0 for h in K.RING_HOSTS}
    for i in range(10000):
        ip = f"192.168.{(i >> 8) & 255}.{i & 255}"
        dist[K.RING_HOSTS[ring.get(ip)]] += 1
    assert dist == K.RING_DISTRIBUTION[name]


def test_ring_empty_and_wrap():
    ring = O.Ring(0, 512)
    assert ring.get("x") == -1  # replicated_hash.go:105-107 "pool is empty"
    ring.add("a")
    hs, ps = ring.points()
    assert len(hs) == 512 and np.all(hs[:-1] <= hs[1:])
    assert ring.get_by_hash(int(hs[-1])) == 0
    if int(hs[-1]) < 2**64 - 1:
        assert ring.get_by_hash(int(hs[-1]) + 1) == int(ps[0])  # wraps to index 0, replicated_hash.go:114-116


# ---- workers_internal_test.go:46-55 ------------------------------------------------------------------------
def test_worker_index():
    p = O.Pool(workers=32)
    for h, idx in K.WORKER_INDEX:
        assert p.worker_index_for_hash63(h) == idx
    assert p.worker_index(b"Foobar") == (0x9DE0B9C33B6693DF >> 1) // ((1 << 63) // 32)


# ---- interval_test.go:47-136 -------------------------------------------------------------------------------
def test_gregorian_expiration():
    for now, d, want in K.GREGORIAN_EXPIRATION:
        got, err = O.gregorian_expiration(_ms(now), d)
        assert err == 0
        if isinstance(want, tuple):
            want = _ms(want) + want[6]
        assert got == want, (now, d)
    got, err = O.gregorian_expiration(_ms((2019, 1, 1, 0, 0, 0, 0)), 99)
    assert (got, err) == (0, 5)
    got, err = O.gregorian_expiration(_ms((2019, 1, 1, 0, 0, 0, 0)), K.GREG_WEEKS)
    assert (got, err) == (0, 4)


def test_gregorian_duration():
    now = _ms((2019, 11, 11, 22, 2, 23, 0))
    assert O.gregorian_duration(now, K.GREG_MINUTES) == (60000, 0)
    assert O.gregorian_duration(now, K.GREG_HOURS) == (3600000, 0)
    assert O.gregorian_duration(now, K.GREG_DAYS) == (86400000, 0)
    assert O.gregorian_duration(now, K.GREG_WEEKS)[1] == 4
    assert O.gregorian_duration(now, 6)[1] == 5
    # interval.go:99 precedence bug: end.UnixNano() - begin.UnixNano()/1000000
    begin_ns = _ms((2019, 11, 1, 0, 0, 0, 0)) * 1_000_000
    end_ns = _ms((2019, 12, 1, 0, 0, 0, 0)) * 1_000_000 - 1
    assert O.gregorian_duration(now, K.GREG_MONTHS) == (end_ns - begin_ns // 1_000_000, 0)
    begin_ns = _ms((2019, 1, 1, 0, 0, 0, 0)) * 1_000_000
    end_ns = _ms((2020, 1, 1, 0, 0, 0, 0)) * 1_000_000 - 1
    assert O.gregorian_duration(now, K.GREG_YEARS) == (end_ns - begin_ns // 1_000_000, 0)
    # December rolls the year
    dec = _ms((2019, 12, 15, 0, 0, 0, 0))
    assert O.gregorian_expiration(dec, K.GREG_MONTHS) == (_ms((2020, 1, 1, 0, 0, 0, 0)) - 1, 0)


# ---- functional_test.go known-answer tables ----------------------------------------------------------------
@pytest.mark.parametrize("sc", K.SCENARIOS, ids=[s["name"] for s in K.SCENARIOS])
@pytest.mark.parametrize("workers", [1, 8])
def test_functional_scenarios(sc, workers):
    pool = O.Pool(workers=workers, now_ms=K.T0)
    play_scenario(pool, sc)


def test_missing_fields():
    play_missing_fields(O.Pool(workers=4, now_ms=K.T0))


def test_batch_too_large():
    pool = O.Pool(now_ms=K.T0)
    reqs = [dict(name="n", unique_key=str(i), limit=1, duration=1000, hits=1) for i in range(1001)]
    with pytest.raises(ValueError, match="max size is '1000'"):  # gubernator.go:189-193
        pool.get_rate_limits(reqs)
    assert len(pool.get_rate_limits(reqs[:1000])) == 1000


def test_error_strings():
    pool = O.Pool(now_ms=K.T0)
    r = pool.get_rate_limits([dict(name="n", unique_key="k", algorithm=5, limit=1, duration=1, hits=1)])[0]
    assert r["error"] == "Error while apply rate limit for 'n_k': during workerPool.GetRateLimit: Invalid rate limit algorithm '5'"
    r = pool.get_rate_limits([dict(name="n", unique_key="k", behavior=K.GREGORIAN, duration=K.GREG_WEEKS, limit=1, hits=1)])[0]
    assert r["error"] == ("Error while apply rate limit for 'n_k': during workerPool.GetRateLimit: Error in tokenBucket: "
                          + K.GREGORIAN_WEEKS_MSG)
    r = pool.get_rate_limits([dict(name="n", unique_key="k", algorithm=1, behavior=K.GREGORIAN, duration=77, limit=1, hits=1)])[0]
    assert r["error"] == ("Error while apply rate limit for 'n_k': during workerPool.GetRateLimit: Error in leakyBucket: "
                          + K.GREGORIAN_INVALID_MSG)
    assert (r["status"], r["limit"], r["remaining"], r["reset_time"]) == (0, 0, 0, 0)


def test_same_key_index_order_within_one_call():
    # gubernator.go:203: the per-request loop applies same-key requests strictly in index order
    pool = O.Pool(workers=4, now_ms=K.T0)
    reqs = [dict(name="n", unique_key="k", limit=3, duration=1000, hits=1) for _ in range(5)]
    out = pool.get_rate_limits(reqs)
    assert [(o["status"], o["remaining"]) for o in out] == [(0, 2), (0, 1), (0, 0), (1, 0), (1, 0)]


# ---- store_test.go:76-125 (values a Loader sees at Save) ---------------------------------------------------
def test_loader_item_values():
    pool = O.Pool(now_ms=K.T0)
    pool.get_rate_limits([dict(name="test_over_limit", unique_key="account:1234", algorithm=0, duration=1000, limit=2, hits=1)])
    it = pool.get_item(b"test_over_limit_account:1234")
    assert it is not None and it.value_kind == 1
    assert (it.limit, it.remaining_i, it.status) == (2, 1, 0)  # store_test.go:120-124
    assert it.expire_at == K.T0 + 1000 and it.stamp == K.T0


# ---- lrucache_test.go:339-428 ------------------------------------------------------------------------------
def _mk_item(expire_at):
    it = O.Item()
    it.algorithm = 1; it.value_kind = 2; it.expire_at = expire_at
    return it


def test_lru_eviction_metrics():
    now = K.T0
    pool = O.Pool(workers=1, cache_size=10, now_ms=now)
    for i in range(10):
        pool.add_item(f"short-expiry-{i}".encode(), _mk_item(now + 5 * 60000))
    pool.advance(6 * 60000)
    pool.add_item(b"evict1", _mk_item(pool.now() + 3600000))
    assert pool.counters()["unexpired_evictions"] == 0 and pool.size() == 10
    assert pool.get_item(b"short-expiry-0") is None  # oldest was evicted

    pool = O.Pool(workers=1, cache_size=10, now_ms=now)
    for i in range(10):
        pool.add_item(f"long-expiry-{i}".encode(), _mk_item(now + 3600000))
    pool.add_item(b"evict2", _mk_item(now + 3600000))
    assert pool.counters()["unexpired_evictions"] == 1 and pool.size() == 10
    assert pool.get_item(b"long-expiry-0") is None and pool.get_item(b"long-expiry-1") is not None


def test_lru_happy_path_and_update():
    pool = O.Pool(workers=1, cache_size=0, now_ms=K.T0)  # NewLRUCache(0) -> 50 000
    for i in range(1000):
        pool.add_item(str(i).encode(), _mk_item(K.T0 + 3600000))
    assert pool.size() == 1000
    for i in range(1000):
        assert pool.get_item(str(i).encode()) is not None
    it = _mk_item(K.T0 + 3600000); it.limit = 7
    pool.add_item(b"5", it)
    assert pool.size() == 1000 and pool.get_item(b"5").limit == 7
    # strict expiry comparisons (cache.go:47,52): now == ExpireAt is still live
    pool.add_item(b"edge", _mk_item(K.T0 + 10))
    pool.set_now(K.T0 + 10)
    assert pool.get_item(b"edge") is not None
    pool.set_now(K.T0 + 11)
    assert pool.get_item(b"edge") is None
    c = pool.counters()
    assert c["cache_miss"] == 1


# ---- UpdatePeerGlobals (gubernator.go:425-459) -------------------------------------------------------------
def test_update_peer_global_items():
    pool = O.Pool(now_ms=K.T0)
    pool.update_peer_global(b"a_b", 0, 5000, 1, 10, 3, K.T0 + 5000)
    it = pool.get_item(b"a_b")
    assert (it.value_kind, it.status, it.limit, it.duration, it.remaining_i, it.stamp, it.expire_at) == (1, 1, 10, 5000, 3, K.T0, K.T0 + 5000)
    pool.update_peer_global(b"a_c", 1, 5000, 0, 10, 3, K.T0 + 5000)
    it = pool.get_item(b"a_c")
    assert (it.value_kind, it.limit, it.duration, it.remaining_f, it.stamp, it.burst, it.expire_at) == (2, 10, 5000, 3.0, K.T0, 10, K.T0 + 5000)


# ---- pre-hashed batch form agrees with the string form -----------------------------------------------------
def test_hashed_form_matches_string_form():
    rng = np.random.default_rng(7)
    p1 = O.Pool(workers=4, now_ms=K.T0)
    p2 = O.Pool(workers=4, now_ms=K.T0)
    n = 4000
    ids = rng.integers(0, 50, n)
    reqs, h = [], np.zeros(n, dtype=O.HREQ_DTYPE)
    for i in range(n):
        r = dict(name="bench", unique_key=f"k{ids[i]:09d}", hits=int(rng.integers(-1, 4)), limit=int(rng.choice([5, 10])),
                 duration=int(rng.choice([1000, 60000])), burst=int(rng.choice([0, 7])), algorithm=int(ids[i] & 1),
                 behavior=int(rng.choice([0, 0, 0, 8, 32])), created_at=K.T0 + int(rng.integers(0, 3)))
        reqs.append(r)
        key = f"bench_k{ids[i]:09d}".encode()
        h[i] = (O.xxh64(key), O.fnv1_64(key), r["hits"], r["limit"], r["duration"], r["burst"], r["created_at"],
                r["algorithm"], r["behavior"] | O.REQ_IS_OWNER)
    a = p1.get_rate_limits(reqs, unbounded=True)
    b = p2.submit_hashed(h)
    for i in range(n):
        assert (a[i]["status"], a[i]["limit"], a[i]["remaining"], a[i]["reset_time"]) == \
               (int(b[i]["status"]), int(b[i]["limit"]), int(b[i]["remaining"]), int(b[i]["reset_time"])), i
    assert p1.counters() == p2.counters()
    # and the multi-threaded worker-pool baseline gives the same answers as the sequential walk
    p3 = O.Pool(workers=4, now_ms=K.T0)
    c = p3.submit_hashed(h, threads=3)
    assert np.array_equal(b, c)


def test_go_float_to_int_conversion_edges():
    # leaky bucket with Limit == 0: rate = +Inf, int64(+Inf) = INT64_MIN on amd64 (parity unpinned by the reference)
    pool = O.Pool(now_ms=K.T0)
    r = pool.get_rate_limits([dict(name="n", unique_key="z", algorithm=1, limit=0, duration=1000, hits=1)])[0]
    assert r["status"] == 1 and r["remaining"] == 0
    # ResetTime = createdAt + (0 - 0) * INT64_MIN
    assert r["reset_time"] == K.T0


def test_hashed_item_api_routes_like_hashed_requests():
    # items installed through the pre-hashed API must be visible to pre-hashed requests whatever the worker count
    for workers in (1, 2, 7):
        pool = O.Pool(workers=workers, now_ms=K.T0)
        kx, kf = O.xxh64(b"glob_k1"), O.fnv1_64(b"glob_k1")
        pool.update_peer_global_hashed(kx, kf, 0, 60000, 0, 80, 24, K.T0 + 60000)
        assert pool.get_item_hashed(kx, kf).remaining_i == 24
        r = np.zeros(1, dtype=O.HREQ_DTYPE)
        r["key_xxh64"], r["key_fnv1"], r["hits"], r["limit"], r["duration"], r["created_at"] = kx, kf, 2, 80, 60000, K.T0
        assert int(pool.submit_hashed(r)[0]["remaining"]) == 22
