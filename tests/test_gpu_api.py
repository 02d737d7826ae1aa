"""The reference-facing Python surface end to end on the GPU: `connect().create_table().search()...`
with the reference's own doctest inputs (python/python/lancedb/table.py:3587-3603,
query.py:1555-1571) and an IVF_PQ table checked against the oracle through the same builder calls."""
import json

import numpy as np
import pytest

import lancedb_b200 as lancedb
import oracle

pytestmark = pytest.mark.gpu


def test_table_search_doctest_l2():
    db = lancedb.connect("memory://")
    data = [{"original_width": 100, "caption": "bar", "vector": [0.1, 2.3, 4.5]},
            {"original_width": 2000, "caption": "foo", "vector": [0.5, 3.4, 1.3]},
            {"original_width": 3000, "caption": "test", "vector": [0.3, 6.2, 2.6]}]
    table = db.create_table("my_table", data)
    out = table.search([0.4, 1.4, 2.4]).select(["caption", "original_width", "vector"]).limit(3).to_arrow()
    assert out.schema.names == ["caption", "original_width", "vector", "_distance"]
    assert str(out.schema.field("_distance").type) == "float"
    rows = out.to_pylist()
    assert [r["caption"] for r in rows] == ["foo", "bar", "test"]
    assert f"{rows[0]['_distance']:.6f}" == "5.220000" and f"{rows[2]['_distance']:.6f}" == "23.089996"


def test_table_search_doctest_cosine():
    db = lancedb.connect("memory://")
    data = [{"vector": [1.1, 1.2], "b": 2}, {"vector": [0.5, 1.3], "b": 4},
            {"vector": [0.4, 0.4], "b": 6}, {"vector": [0.4, 0.4], "b": 10}]
    table = db.create_table("my_table", data=data)
    df = table.search([0.4, 0.4]).distance_type("cosine").select(["b", "vector"]).limit(3).to_pandas()
    assert list(df["b"]) == [6, 10, 2]
    assert [f"{d:.6f}" for d in df["_distance"]] == ["0.000000", "0.000000", "0.000944"]


def test_exact_match_distance_zero_and_ordering():
    # python/python/tests/test_db.py:198-199, test_query.py:562-570
    db = lancedb.connect("memory://")
    t = db.create_table("t", [{"vector": [1.0, 2.0], "id": 1}, {"vector": [3.0, 4.0], "id": 2}])
    rows = t.search([1.0, 2.0]).to_list()
    assert rows[0]["id"] == 1 and rows[0]["_distance"] == 0.0
    assert [r["id"] for r in t.search([0.0, 0.0]).to_list()] == [1, 2]


@pytest.mark.parametrize("metric", ["l2", "cosine"])
def test_ivf_pq_table_vs_oracle(metric):
    rng = np.random.default_rng(0)
    x = rng.standard_normal((6000, 64)).astype(np.float32)
    db = lancedb.connect("memory://")
    t = db.create_table("v", {"vector": x, "id": np.arange(6000)})
    t.create_index(metric=metric, num_partitions=16, num_sub_vectors=8, max_iterations=4, accelerator="cuda")
    q = rng.standard_normal((5, 64)).astype(np.float32)
    orc = oracle.OracleIndex.from_data(t._index_data["vector"])
    oi, od, oc = orc.search(q, k=12, nprobes=4)          # top_k = limit + offset
    for i in range(5):
        out = t.search(q[i]).distance_type(metric).nprobes(4).limit(10).offset(2).with_row_id(True).to_arrow()
        assert out["_rowid"].to_pylist() == [int(v) for v in oi[i, 2:12]]
        assert np.array_equal(np.asarray(out["_distance"].to_pylist(), np.float32), od[i, 2:12])
        assert out["id"].to_pylist() == out["_rowid"].to_pylist()
    # refine_factor re-ranks with exact distances (rust/lancedb/src/query.rs:1302-1332)
    out = t.search(q[0]).distance_type(metric).nprobes(4).refine_factor(3).limit(5).to_arrow()
    ri, rd, rc = orc.search(q[:1], k=5, nprobes=4, refine_factor=3)
    assert np.array_equal(np.asarray(out["_distance"].to_pylist(), np.float32), rd[0])
    # bypass_vector_index -> exact flat search
    flat = t.search(q[0]).distance_type(metric).bypass_vector_index().limit(5).to_arrow()
    fi, fd, fc = oracle.flat_search(x, q[:1], k=5, metric=metric)
    assert flat["id"].to_pylist() == [int(v) for v in fi[0]]
    # multi-vector query: one result block per query vector, tagged with query_index
    multi = t.search(q[:3]).distance_type(metric).nprobes(4).limit(4).to_arrow()
    assert multi["query_index"].to_pylist() == [0] * 4 + [1] * 4 + [2] * 4
    with pytest.raises(ValueError, match="minimum_nprobes must be greater than 0"):
        t.search(q[0]).nprobes(0).to_arrow()


_GRAPH_SCRIPT = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
from tests.util import random_index, queries
from lancedb_b200._native import GpuIvfPq, GpuFlat
rng = np.random.default_rng(5)
ix = random_index(rng, dim=64, nlist=24, m=8, n=6000, with_vectors=True)
g = GpuIvfPq(ix)
f = GpuFlat(ix.vectors, ix.row_ids)
out = []
for rep in range(4):                       # call 1 eager, call 2 captured, calls 3-4 replayed
    q = queries(np.random.default_rng(100 + rep), 33, 64)
    ids, dist, cnt = g.search(q, k=7, nprobes=5)
    fi, fd, fc = f.search(q, k=7, metric="l2")
    out.append((ids.copy(), dist.copy(), cnt.copy(), fi.copy(), fd.copy()))
ids, dist, cnt = g.search(queries(np.random.default_rng(9), 17, 64), k=3, nprobes=24)   # new key
np.savez({dst!r}, **{{f"a{{i}}_{{j}}": a for i, t in enumerate(out) for j, a in enumerate(t)}}, last_ids=ids, last_dist=dist)
"""


def test_graph_replay_matches_eager(tmp_path):
    """Graph replay (the default: capture on the 2nd call of a shape, replay afterwards; LGPU_NO_GRAPH=1
    disables it) returns exactly what the eager launch sequence returns, for fresh query contents on every
    replay."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for mode in ("0", "1"):
        dst = str(tmp_path / f"g{mode}.npz")
        env = dict(os.environ, LGPU_NO_GRAPH="1" if mode == "0" else "0")
        subprocess.run([sys.executable, "-c", _GRAPH_SCRIPT.format(root=root, dst=dst)], check=True, env=env,
                       timeout=300)
        res[mode] = np.load(dst)
    assert set(res["0"].files) == set(res["1"].files)
    for name in res["0"].files:
        assert np.array_equal(res["0"][name], res["1"][name]), name


def test_query_builder_with_prefilter_and_postfilter():
    """python/python/tests/test_query.py:911-986: where() prefilters by default, prefilter=False filters
    the vector search's results (possibly to nothing), repeated where() calls AND."""
    db = lancedb.connect("memory://")
    t = db.create_table("t", [{"vector": [1.0, 2.0], "id": 1, "b": 5}, {"vector": [3.0, 4.0], "id": 2, "b": 20},
                              {"vector": [5.0, 6.0], "id": 3, "b": 7}, {"vector": [0.5, 0.1], "id": 4, "b": 9}])
    rs = t.search([0, 0]).where("id = 2").to_list()
    assert len(rs) == 1 and rs[0]["id"] == 2 and rs[0]["vector"] == [3.0, 4.0]
    df = t.search([0, 0]).where("id = 2", prefilter=True).limit(1).to_pandas()
    assert df["id"].values[0] == 2
    df = t.search([0, 0]).where("id = 2", prefilter=False).limit(1).to_pandas()
    assert len(df) == 0                                   # the nearest row is id 4; the filter drops it
    assert len(t.search([0, 0]).where("id = 2").postfilter().limit(1).to_list()) == 0
    rs = t.search([0, 0]).where("id >= 1").where("b < 10").limit(10).to_list()
    assert [r["id"] for r in rs] == [4, 1, 3]
    assert t.search([0, 0]).where("id < 0").to_list() == []
    with pytest.raises(ValueError):
        t.search([0, 0]).where("nosuchcolumn = 1").to_list()


def test_ivf_pq_table_prefilter_vs_oracle():
    rng = np.random.default_rng(17)
    n, dim = 4000, 32
    vec = rng.standard_normal((n, dim)).astype(np.float32)
    db = lancedb.connect("memory://")
    t = db.create_table("t", {"vector": list(vec), "id": np.arange(n), "grp": np.arange(n) % 7})
    t.create_index(metric="l2", num_partitions=16, num_sub_vectors=8, accelerator="cuda")
    q = rng.standard_normal(dim).astype(np.float32)
    out = t.search(q).where("grp = 3 AND id >= 100").nprobes(8).limit(10).with_row_id(True).to_arrow()
    data = t._index_data["vector"]
    mask = (np.arange(n) % 7 == 3) & (np.arange(n) >= 100)
    oi, od, oc = oracle.OracleIndex.from_data(data).search(q, k=10, nprobes=8, allow=oracle.allow_bitmap(
        np.nonzero(mask)[0], n), allow_bits=n)
    assert out["_rowid"].to_pylist() == oi[0, :oc[0]].tolist()
    assert np.array_equal(np.asarray(out["_distance"]).view(np.uint32), od[0, :oc[0]].view(np.uint32))
    assert all(g == 3 for g in out["grp"].to_pylist())


# ---------------------------------------------------------------- boundary robustness (round 2)
def test_nan_and_zero_queries_return_nothing_and_do_not_poison_the_context():
    """A NaN / Inf query (any metric) or an all-zero cosine query has no finite centroid distance: fewer than
    nprobes probes come back from the coarse step and the unused slots must behave as empty partitions --
    count 0, no illegal address (ADVICE r01: group.cu read part_n[0xffffffff])."""
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(31)
    for metric in ("l2", "cosine", "dot"):
        ix = random_index(rng, dim=64, nlist=12, m=8, metric=metric, n=3000)
        gpu = _native.GpuIvfPq(ix)
        q = queries(rng, 6, 64)
        q[1, 3] = np.nan
        q[4, :] = np.inf
        if metric == "cosine":
            q[2, :] = 0.0
        gi, gd, gc = gpu.search(q, k=5, nprobes=4)
        oi, od, oc = oracle.OracleIndex.from_data(ix).search(q, k=5, nprobes=4)
        # (an Inf query is not "no distance": for l2 every distance is +inf, which IS NOT NULL; only the
        # survival of the context is asserted for it)
        assert gc[1] == 0 and (metric != "cosine" or gc[2] == 0)
        good = [0, 3, 5]
        assert np.array_equal(gi[good], oi[good]) and np.array_equal(gc[good], oc[good])
        assert np.array_equal(gd[good].view(np.uint32), od[good].view(np.uint32))
        gi2, _, gc2 = gpu.search(q[:1], k=5, nprobes=4)          # the context is still healthy
        assert np.array_equal(gi2[0], oi[0])
        gpu.close()


def test_closed_handle_is_rejected_not_dereferenced():
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(32)
    ix = random_index(rng, dim=32, nlist=4, m=4, n=500)
    gpu = _native.GpuIvfPq(ix)
    h = gpu._h
    gpu.search(queries(rng, 2, 32), k=3, nprobes=2)
    gpu.close()
    gpu._h = h                                   # a stale handle value, as a buggy host might keep
    with pytest.raises(ValueError, match="closed"):
        gpu.search(queries(rng, 2, 32), k=3, nprobes=2)
    gpu._h = None


def test_close_waits_for_searches_in_flight():
    """lgpu_index_close while other threads are inside lgpu_search must not free the index under them."""
    import threading
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(33)
    ix = random_index(rng, dim=64, nlist=16, m=8, n=20000)
    gpu = _native.GpuIvfPq(ix)
    q = queries(rng, 64, 64)
    want = gpu.search(q, k=10, nprobes=8)
    errs, oks = [], []

    def worker():
        for _ in range(30):
            try:
                got = gpu.search(q, k=10, nprobes=8)
                oks.append(np.array_equal(got[0], want[0]))
            except ValueError as e:              # the handle was closed between two calls: the documented outcome
                errs.append(str(e))
                return
    ths = [threading.Thread(target=worker) for _ in range(4)]
    for t in ths:
        t.start()
    h = gpu._h
    _native.load().lgpu_index_close(h)
    for t in ths:
        t.join()
    gpu._h = None
    assert all(oks) and all("closed" in e for e in errs)


def test_timeout_status_and_builder_argument():
    """QueryExecutionOptions.timeout (python/python/tests/test_query.py:1846,1957): an impossible deadline
    maps to LGPU_TIMEOUT -> TimeoutError and leaves the outputs untouched; a generous one changes nothing."""
    import datetime
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(34)
    ix = random_index(rng, dim=128, nlist=64, m=16, n=400000)
    gpu = _native.GpuIvfPq(ix)
    q = queries(rng, 512, 128)
    want = gpu.search(q, k=10, nprobes=32)
    got = gpu.search(q, k=10, nprobes=32, timeout_ms=60000)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    ids = np.full((512, 10), 7, np.uint64); dist = np.full((512, 10), -1.0, np.float32); cnt = np.full(512, 9, np.uint32)
    p = _native.make_params(k=10, nprobes=32, timeout_ms=1)
    big = np.ascontiguousarray(np.tile(q, (8, 1)))
    ids8 = np.full((4096, 10), 7, np.uint64); dist8 = np.full((4096, 10), -1.0, np.float32); cnt8 = np.full(4096, 9, np.uint32)
    with pytest.raises(TimeoutError, match="timeout"):
        gpu.search_into(big, p, ids8, dist8, cnt8)          # 4096 x 32 probes cannot finish within 1 ms
    assert (ids8 == 7).all() and (dist8 == -1.0).all() and (cnt8 == 9).all()
    gpu.close()
    db = lancedb.connect("memory://")
    t = db.create_table("t", [{"vector": [1.0, 2.0], "id": 1}, {"vector": [3.0, 4.0], "id": 2}])
    rows = t.search([1.0, 2.0]).to_list(timeout=datetime.timedelta(seconds=30))
    assert rows[0]["id"] == 1
    with pytest.raises(ValueError):
        t.search([1.0, 2.0]).to_arrow(timeout=datetime.timedelta(seconds=-1))


def test_async_tickets_pipeline_and_match_sync():
    import torch
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(35)
    ix = random_index(rng, dim=64, nlist=32, m=8, n=30000)
    gpu = _native.GpuIvfPq(ix)
    p = _native.make_params(k=10, nprobes=6)
    qs = [torch.from_numpy(queries(rng, 128, 64)).pin_memory().numpy() for _ in range(5)]
    bufs = [(torch.empty(128, 10, dtype=torch.int64).pin_memory().numpy().view(np.uint64),
             torch.empty(128, 10, dtype=torch.float32).pin_memory().numpy(),
             torch.empty(128, dtype=torch.int32).pin_memory().numpy().view(np.uint32)) for _ in range(5)]
    n0 = _native.kernel_launch_count()
    tickets = [gpu.search_async(qs[i], p, *bufs[i]) for i in range(5)]     # five calls in flight
    for t in tickets:
        _native.ticket_wait(t)
    assert _native.kernel_launch_count() > n0
    for i in range(5):
        want = gpu.search(qs[i], k=10, nprobes=6)
        assert np.array_equal(bufs[i][0], want[0]) and np.array_equal(bufs[i][2], want[2])
        assert np.array_equal(bufs[i][1].view(np.uint32), want[1].view(np.uint32))
    gpu.close()


def test_flat_search_device_matches_host_call():
    """ADVICE r01: GpuFlat.search_device had fallen out of the class."""
    import torch
    from lancedb_b200 import _native
    from tests.util import queries
    rng = np.random.default_rng(36)
    v = queries(rng, 9000, 64)
    q = queries(rng, 16, 64)
    fl = _native.GpuFlat(v)
    want = fl.search(q, k=7, metric="l2")
    dq = torch.from_numpy(q).cuda()
    oi = torch.empty(16, 7, dtype=torch.int64, device="cuda"); od = torch.empty(16, 7, device="cuda")
    oc = torch.empty(16, dtype=torch.int32, device="cuda")
    fl.search_device("l2", dq.data_ptr(), 16, _native.make_params(k=7, nprobes=0), oi.data_ptr(), od.data_ptr(),
                     oc.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(oi.cpu().numpy().view(np.uint64), want[0])
    assert np.array_equal(od.cpu().numpy().view(np.uint32), want[1].view(np.uint32))
    fl.close()


def test_coalesced_single_vector_calls_share_batches(monkeypatch):
    """lgpu_search_coalesced: 48 threads each with one query vector get exactly the rows of a solitary search, and
    the batcher turns them into far fewer kernel launches than 48 separate searches would take."""
    import threading
    monkeypatch.setenv("LGPU_COALESCE_US", "3000")      # (read once, at the first coalesced call of the process)
    from lancedb_b200 import _native
    from tests.util import queries, random_index
    rng = np.random.default_rng(37)
    ix = random_index(rng, dim=64, nlist=32, m=8, n=30000)
    gpu = _native.GpuIvfPq(ix)
    q = queries(rng, 48, 64)
    want = gpu.search(q, k=10, nprobes=6)
    n0 = _native.kernel_launch_count()
    gpu.search(q[:1], k=10, nprobes=6)
    per_call = _native.kernel_launch_count() - n0
    got = [None] * 48
    barrier = threading.Barrier(48)

    def worker(i):
        barrier.wait()
        got[i] = gpu.search_one(q[i], k=10, nprobes=6)
    n1 = _native.kernel_launch_count()
    ths = [threading.Thread(target=worker, args=(i,)) for i in range(48)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    used = _native.kernel_launch_count() - n1
    for i in range(48):
        assert np.array_equal(got[i][0], want[0][i]) and got[i][2] == want[2][i]
        assert np.array_equal(got[i][1].view(np.uint32), want[1][i].view(np.uint32))
    assert used < 48 * per_call / 2, (used, per_call)          # at least half of the calls rode someone else's batch
    gpu.close()


def test_remote_wire_format_query_node():
    """SURVEY.md 8f-4: a `/v1/table/{name}/query/` JSON body (as the reference's remote client builds it,
    rust/lancedb/src/remote/table.rs:724-929) served by the GPU path, Arrow IPC file back."""
    from lancedb_b200 import remote
    rng = np.random.default_rng(38)
    x = rng.standard_normal((5000, 32)).astype(np.float32)
    t = lancedb.connect("memory://").create_table("v", {"vector": x, "id": np.arange(5000), "grp": np.arange(5000) % 5})
    t.create_index(metric="l2", num_partitions=8, num_sub_vectors=4, max_iterations=4, accelerator="cuda")
    q = rng.standard_normal(32).astype(np.float32)
    body = remote.build_query_body(q, k=7, minimum_nprobes=4, maximum_nprobes=4, filter="grp = 2", columns=["id", "grp"],
                                   with_row_id=True)
    out = remote.read_ipc_file(remote.handle_query(t, json.dumps(body)))
    want = t.search(q).nprobes(4).limit(7).where("grp = 2").select(["id", "grp"]).with_row_id(True).to_arrow()
    assert out.equals(want) and out.schema.names == ["id", "grp", "_distance", "_rowid"]
    assert all(g == 2 for g in out["grp"].to_pylist())
    multi = remote.build_query_body(np.stack([q, -q]), k=3, minimum_nprobes=4, maximum_nprobes=4, bypass_vector_index=True)
    out = remote.read_ipc_file(remote.handle_query(t, multi))
    assert out.num_rows == 6 and out["query_index"].to_pylist() == [0, 0, 0, 1, 1, 1]
    with pytest.raises(NotImplementedError):
        remote.handle_query(t, remote.build_query_body([], k=3))


def test_index_loaded_from_lance_files_searches_like_the_in_memory_one(tmp_path):
    """SURVEY.md 8f-3: an IVF_PQ index read back from `_indices/<uuid>/{index.idx,auxiliary.idx}` (layout recalled,
    lancedb_b200/lance_index.py) gives the same ids and distance bits as the index it was written from, plain and with
    refine_factor (raw vectors re-gathered from the table by row id)."""
    rng = np.random.default_rng(8)
    x = rng.standard_normal((5000, 32)).astype(np.float32)
    db = lancedb.connect("memory://")
    t = db.create_table("v", {"vector": x, "id": np.arange(5000)})
    t.create_index(metric="l2", num_partitions=12, num_sub_vectors=4, max_iterations=4, accelerator="cuda")
    d = str(tmp_path / "v.lance" / "_indices" / "11111111-2222")
    t.save_lance_index(d)
    t2 = db.create_table("w", {"vector": x, "id": np.arange(5000)})
    t2.load_lance_index(d)
    assert t2.list_indices()[0]["index_type"] == "IVF_PQ"
    q = rng.standard_normal((40, 32)).astype(np.float32)
    for kw in ({}, {"refine": 3}):
        a = t.search(q).nprobes(5).limit(7)
        b = t2.search(q).nprobes(5).limit(7)
        if kw:
            a, b = a.refine_factor(3), b.refine_factor(3)
        a, b = a.with_row_id(True).to_arrow(), b.with_row_id(True).to_arrow()
        assert a["_rowid"].to_pylist() == b["_rowid"].to_pylist()
        assert np.array_equal(np.asarray(a["_distance"].to_pylist(), np.float32).view(np.uint32),
                              np.asarray(b["_distance"].to_pylist(), np.float32).view(np.uint32))


_BENCH_LAST_STEP_SCRIPT = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
import bench, oracle
cfg = bench.WORKLOADS["tiny"]
ix = bench.get_index(cfg, "tiny", "cuda:0")[0]          # the index the run trained (read back from its cache)
q = bench.synth_vectors(cfg, 8 * cfg["batch"], 43, "cuda:0").reshape(8, cfg["batch"], cfg["dim"])[{step} % 8]
ids, dist, cnt = oracle.OracleIndex.from_data(ix).search(q.cpu().numpy(), k=cfg["k"], nprobes=cfg["nprobes"])
np.savez({dst!r}, ids=ids, distances=dist, counts=cnt)
"""


def test_bench_dump_outputs_reproducible_and_equal_to_the_oracle(tmp_path):
    """bench.py --dump-outputs on the timed device-resident path: two runs that each train their index on the GPU dump
    the same bytes, and the dump is the oracle's answer for the last timed step's batch (queries 8 batches deep, step
    i searches batch i % 8).  The bench inherits the suite's LGPU_SMALL_SLOTS=0, so its tiny batches take the batched
    kernels that the flagship workload times."""
    import os, subprocess, sys
    from tests.util import bench_dumps
    steps = 5
    (a, da), (b, _) = bench_dumps(tmp_path, "--workload", "tiny", "--steps", str(steps), "--warmup", "3",
                                  "--no-cpu-baseline")
    assert da["steps"] == steps and da["gate"]["gpu_equals_oracle_plain"]
    for name in ("ids", "distances", "counts"):
        assert np.array_equal(a[name], b[name]), name
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dst = str(tmp_path / "want.npz")
    subprocess.run([sys.executable, "-c", _BENCH_LAST_STEP_SCRIPT.format(root=root, step=steps - 1, dst=dst)],
                   check=True, timeout=300, cwd=root, env=dict(os.environ, TMPDIR=str(tmp_path / "tmp0")))
    want = np.load(dst)
    assert np.array_equal(a["ids"], want["ids"].astype(np.float64))
    assert np.array_equal(a["distances"].view(np.uint32), want["distances"].view(np.uint32))
    assert np.array_equal(a["counts"], want["counts"].astype(np.float64))
