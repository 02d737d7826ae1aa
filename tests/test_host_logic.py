"""Host-side logic that needs no GPU: builder defaults / validation mirroring the reference,
index parameter defaults, partition sharding, and the world_size-2 all-gather + merge pattern
over gloo (the oracle stands in for the per-rank GPU search)."""
import json
import os
import socket
import sys

import numpy as np
import pytest

import lancedb_b200
from lancedb_b200.index import assign_partitions, suggested_num_partitions, suggested_num_sub_vectors
from lancedb_b200.query import LanceVectorQueryBuilder
from tests.util import queries, random_index


class _FakeTable:
    def __init__(self, dim=4):
        self.dim = dim
        self.calls = []

    def _dim(self, column):
        return self.dim

    def count_rows(self):
        return 100

    def _vector_search(self, q, **kw):
        self.calls.append(kw)
        B, k = q.shape[0], kw["k"]
        ids = np.tile(np.arange(k, dtype=np.uint64), (B, 1))
        return ids, np.tile(np.arange(k, dtype=np.float32), (B, 1)), np.full(B, k, np.uint32)

    def _take(self, row_ids, columns):
        import pyarrow as pa
        return pa.table({"id": pa.array(np.asarray(row_ids, np.int64))})


def test_request_defaults_match_reference():
    # rust/lancedb/src/query.rs:36, 1097-1113: k=10, nprobes min=max=20, no refine
    t = _FakeTable()
    out = LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").to_arrow()
    kw = t.calls[0]
    assert kw["k"] == 10 and kw["nprobes"] == 20 and kw["refine_factor"] is None
    assert kw["distance_type"] is None and kw["lower"] is None and kw["upper"] is None and kw["use_index"]
    assert out.schema.names == ["id", "_distance"] and str(out.schema.field("_distance").type) == "float"


def test_limit_offset_and_multivector():
    t = _FakeTable()
    out = (LanceVectorQueryBuilder(t, [[1, 2, 3, 4], [4, 3, 2, 1]], "vector").limit(3).offset(2)
           .with_row_id(True).to_arrow())
    assert t.calls[0]["k"] == 5                       # top_k = limit + offset (table/query.rs:231)
    assert out.num_rows == 6 and out["query_index"].to_pylist() == [0, 0, 0, 1, 1, 1]
    assert out["_rowid"].to_pylist()[:3] == [2, 3, 4]


def test_builder_validation_errors():
    t = _FakeTable()
    with pytest.raises(ValueError, match="minimum_nprobes must be greater than 0"):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").nprobes(0).to_arrow()
    with pytest.raises(ValueError, match="No vector column found to match with the query vector dimension: 3"):
        LanceVectorQueryBuilder(t, [1, 2, 3], "vector").to_arrow()
    with pytest.raises(ValueError):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").limit(0)
    with pytest.raises(ValueError, match="maximum_nprobes"):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").minimum_nprobes(10).maximum_nprobes(5).to_arrow()
    # one setter alone is validated against the OTHER one's default of 20 (table.py:5777-5787 lowering onto
    # query.rs:1232-1275; python/python/tests/test_query.py:936-961); the final state counts, not the call order
    with pytest.raises(ValueError, match="minimum_nprobes must be less than or equal to maximum_nprobes"):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").minimum_nprobes(100).to_arrow()
    with pytest.raises(ValueError, match="maximum_nprobes must be greater than or equal to minimum_nprobes"):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").maximum_nprobes(5).to_arrow()
    B = lambda: LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector")
    assert B().minimum_nprobes(5)._resolve()[2:] == (5, 20)                     # maximum stays at its default
    assert B().maximum_nprobes(50)._resolve()[2:] == (20, 50)
    assert B().minimum_nprobes(2).maximum_nprobes(4)._resolve()[2:] == (2, 4)
    assert B().nprobes(30).maximum_nprobes(20).minimum_nprobes(20)._resolve()[2:] == (20, 20)
    assert B().minimum_nprobes(300).maximum_nprobes(0)._resolve()[2:] == (300, 1 << 30)   # 0 = no limit
    for empty in ([], [[]]):                                            # test_query.py:2007-2016
        with pytest.raises(ValueError, match="non-empty"):
            LanceVectorQueryBuilder(t, empty, "vector")
    b = LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").where("a > 1").where("a < 5", prefilter=False)
    assert b._where == "(a > 1) AND (a < 5)" and b._postfilter        # test_query.py:600-604
    with pytest.raises(NotImplementedError):
        LanceVectorQueryBuilder(t, [1, 2, 3, 4], "vector").where(object())


def test_index_parameter_defaults():
    # rust/lancedb/src/index/vector.rs:306-319; create_index.rs:734-795
    assert suggested_num_sub_vectors(768) == 48 and suggested_num_sub_vectors(24) == 3
    assert suggested_num_sub_vectors(7) == 1
    assert suggested_num_partitions(16384) == 2


def test_table_surface_and_column_inference():
    db = lancedb_b200.connect("memory://")
    t = db.create_table("t", [{"vector": [1.0, 2.0], "id": 1}, {"vector": [3.0, 4.0], "id": 2}])
    assert db.table_names() == ["t"] and t.count_rows() == 2
    assert t.search([0.0, 0.0])._vector_column == "vector"
    with pytest.raises(ValueError, match="dimension: 3"):
        t.search([0.0, 0.0, 0.0])
    with pytest.raises(ValueError, match="already exists"):
        db.create_table("t", [{"vector": [1.0, 2.0]}])


def test_shard_partitions_cover_index_exactly():
    rng = np.random.default_rng(0)
    ix = random_index(rng, dim=16, nlist=13, m=2, n=900)
    sizes = np.diff(ix.part_offsets.astype(np.int64))
    owner = assign_partitions(sizes, 4)
    loads = [int(sizes[owner == r].sum()) for r in range(4)]
    assert max(loads) - min(loads) <= sizes.max()
    seen = []
    for r in range(4):
        sh = ix.shard(r, 4)
        sh.validate()
        assert np.array_equal(sh.centroids, ix.centroids) and np.array_equal(sh.codebook, ix.codebook)
        for p in range(ix.nlist):
            if owner[p] == r:
                assert np.array_equal(sh.partition_codes(p), ix.partition_codes(p))
            else:
                assert sh.part_offsets[p + 1] == sh.part_offsets[p]
        seen.append(sh.row_ids)
    assert np.array_equal(np.sort(np.concatenate(seen)), np.sort(ix.row_ids))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _rank_main(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import oracle
    from lancedb_b200 import _native
    from lancedb_b200.distributed import gather_shape, merge_records, pack_records
    dist.init_process_group("gloo", rank=rank, world_size=world, init_method=f"tcp://127.0.0.1:{port}")
    rng = np.random.default_rng(7)
    ix = random_index(rng, dim=32, nlist=9, m=4, n=1500)
    q = queries(rng, 11, 32)
    k, nprobes = 10, 5
    ids, dst, cnt = oracle.OracleIndex.from_data(ix.shard(rank, world)).search(q, k=k, nprobes=nprobes)
    # the library's exchange step, restated on the host: ONE all-gather of [B][k] 16-byte records
    # (lgpu_search_sharded packs (id u64, dist f32, pad u32) and gathers them as bytes), then the merge
    assert _native.TOPK_RECORD.itemsize == 16
    send = pack_records(ids, dst)
    recv = torch.empty(world * send.nbytes, dtype=torch.uint8)
    dist.all_gather_into_tensor(recv, torch.from_numpy(send.view(np.uint8).reshape(-1)))
    gathered = recv.numpy().view(_native.TOPK_RECORD).reshape(gather_shape(world, 11, k))
    m_ids, m_dst, m_cnt = merge_records(gathered, k)
    full_ids, full_dst, full_cnt = oracle.OracleIndex.from_data(ix).search(q, k=k, nprobes=nprobes)
    assert np.array_equal(m_cnt, full_cnt) and np.array_equal(m_ids, full_ids)
    assert np.array_equal(m_dst.view(np.uint32), full_dst.view(np.uint32))
    dist.barrier()
    dist.destroy_process_group()
    open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")


def test_sharded_search_pattern_world2_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = _free_port()
    mp.spawn(_rank_main, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


# ---------------------------------------------------------------- where() filters (host side)
def test_filter_evaluator_matches_reference_test_predicates():
    """The predicate forms the reference's tests pass to .where() (python/python/tests/test_query.py:
    284-308, 600-604, 911-986, 1024) evaluated on the host; NULL predicates exclude the row."""
    import pyarrow as pa
    from lancedb_b200 import filter as F
    t = pa.table({"id": [1, 2, 3, 4, None], "b": [5.0, 15.0, 2.5, None, 9.0], "name": ["aa", "ab", "ca", None, "zz"]})
    cases = {
        "id = 2": [0, 1, 0, 0, 0], "id >= 2": [0, 1, 1, 1, 0], "b < 10": [1, 0, 1, 0, 1],
        "(id >= 1) AND (id < 2)": [1, 0, 0, 0, 0], "id < 0": [0, 0, 0, 0, 0],
        "id IN (1, 3) OR name LIKE 'z%'": [1, 0, 1, 0, 1], "NOT id = 2": [1, 0, 1, 1, 0],
        "b IS NULL": [0, 0, 0, 1, 0], "id IS NOT NULL and b BETWEEN 2 AND 9": [1, 0, 1, 0, 0],
        "name = 'ab'": [0, 1, 0, 0, 0], "id NOT IN (1, 2)": [0, 0, 1, 1, 0],
    }
    for w, want in cases.items():
        assert F.evaluate(t, w).astype(int).tolist() == want, w
    assert F.combine(None, "id >= 1") == "id >= 1"
    assert F.combine("id >= 1", "id < 2") == "(id >= 1) AND (id < 2)"       # test_query.py:600-604
    for bad in ("id ==== 2", "nosuchcolumn = 1", "id = ", ""):
        with pytest.raises(ValueError):
            F.evaluate(t, bad)


def test_allow_bitmaps_agree():
    from lancedb_b200 import _native
    import oracle
    rng = np.random.default_rng(5)
    for n in (1, 31, 32, 33, 1000):
        mask = rng.random(n) < 0.3
        a = _native.mask_bitmap(mask)
        b = _native.allow_bitmap(np.nonzero(mask)[0], n)
        c = oracle.allow_bitmap(np.nonzero(mask)[0], n)
        assert a.dtype == np.uint32 and a.size == (n + 31) // 32
        assert np.array_equal(a, b) and np.array_equal(a, c)


def test_oracle_prefilter_semantics():
    """Prefilter = rows dropped before the top-k: the filtered result equals the unfiltered search over
    only the allowed rows (flat), and every returned id is allowed (IVF_PQ)."""
    import oracle
    from tests.util import queries, random_index
    rng = np.random.default_rng(6)
    v = rng.standard_normal((300, 16)).astype(np.float32)
    q = rng.standard_normal((5, 16)).astype(np.float32)
    allowed = np.sort(rng.choice(300, 40, replace=False)).astype(np.uint64)
    bm = oracle.allow_bitmap(allowed, 300)
    fi, fd, fc = oracle.flat_search(v, q, k=7, allow=bm, allow_bits=300)
    si, sd, sc = oracle.flat_search(v[allowed], q, k=7, row_ids=allowed)
    assert np.array_equal(fi, si) and np.array_equal(fd, sd) and np.array_equal(fc, sc)
    ix = random_index(rng, dim=32, nlist=8, m=4, n=2000)
    orc = oracle.OracleIndex.from_data(ix)
    allowed = rng.choice(2000, 150, replace=False).astype(np.uint64)
    bm = oracle.allow_bitmap(allowed, 2000)
    ids, dist, cnt = orc.search(queries(rng, 9, 32), k=10, nprobes=8, allow=bm, allow_bits=2000)
    ok = set(allowed.tolist())
    for i in range(9):
        assert cnt[i] == 10 and all(int(x) in ok for x in ids[i, :cnt[i]])
    # ids beyond allow_bits are excluded
    ids2, _, cnt2 = orc.search(queries(rng, 3, 32), k=10, nprobes=8, allow=oracle.allow_bitmap(np.arange(64), 64), allow_bits=64)
    assert all(int(x) < 64 for i in range(3) for x in ids2[i, :cnt2[i]])


def test_bench_reference_arm_prints_one_json_line(tmp_path):
    """bench.py --impl reference (the CPU arm the driver times next to ours) on the tiny workload: exactly one
    line on stdout, the contract's keys, `impl: reference`, and a cpu_baseline that describes this run."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, NCCL_DEBUG="VERSION")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 2 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in d["config"]


def test_bench_dump_outputs_reproducible(tmp_path):
    """bench.py --dump-outputs writes the last timed step's results (ids / distances / counts of the whole batch), and
    two runs that each train their own index write the same bytes."""
    from tests.util import bench_dumps
    (a, da), (b, _) = bench_dumps(tmp_path, "--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1")
    assert da["steps"] == 2
    assert sorted(a) == ["counts", "distances", "ids"]
    assert a["ids"].shape == a["distances"].shape == (64, 10) and a["counts"].shape == (64,)
    assert a["ids"].dtype == a["counts"].dtype == np.float64 and a["distances"].dtype == np.float32
    assert np.all(a["counts"] == 10) and np.all(np.diff(a["distances"], axis=1) >= 0)
    for name in a:
        assert np.array_equal(a[name], b[name]), name


def test_bench_index_cache_only_in_a_private_directory_of_this_user(tmp_path, monkeypatch):
    """bench.py caches trained indexes in <tmp>/lancedb_b200_bench_<uid>, created 0700; a directory of that name that
    is not this user's private directory (other mode, a link) is not used and nothing is cached."""
    import importlib, stat, tempfile
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", os.environ.get("CUBLAS_WORKSPACE_CONFIG", ":4096:8"))
    bench = importlib.import_module("bench")
    monkeypatch.setattr(tempfile, "tempdir", str(tmp_path))
    cfg = bench.WORKLOADS["tiny"]
    d = str(tmp_path / f"lancedb_b200_bench_{os.getuid()}")
    path = bench.index_cache_path(cfg, "tiny", "cpu")
    assert os.path.dirname(path) == d and stat.S_IMODE(os.lstat(d).st_mode) == 0o700
    assert bench.index_cache_path(cfg, "tiny", "cpu") == path
    os.chmod(d, 0o755)
    assert bench.index_cache_path(cfg, "tiny", "cpu") is None
    os.rmdir(d)
    os.symlink(str(tmp_path), d)
    assert bench.index_cache_path(cfg, "tiny", "cpu") is None


def test_oracle_pq_encode_is_argmin_of_the_distance_table():
    """orc_pq_encode picks, per sub-vector, the first minimum of the very table row orc_build_lut produces for
    the row's residual; orc_ivf_assign is find_partitions with nprobes 1."""
    import oracle
    from tests.util import queries, random_index
    rng = np.random.default_rng(8)
    for metric, dim, m in (("l2", 32, 4), ("cosine", 48, 3), ("dot", 16, 16)):
        ix = random_index(rng, dim=dim, nlist=7, m=m, metric=metric, n=100)
        orc = oracle.OracleIndex.from_data(ix)
        v = queries(rng, 20, dim)
        parts = orc.ivf_assign(v)
        codes = orc.pq_encode(v, parts)
        for r in range(20):
            qn = oracle.normalize(v[r]) if metric == "cosine" else v[r]
            assert parts[r] == orc.find_partitions(qn, 1)[0][0]
            resid = qn if metric == "dot" else (qn - ix.centroids[parts[r]]).astype(np.float32)
            lut = orc.build_lut(resid)
            assert np.array_equal(codes[r], lut.argmin(axis=1).astype(np.uint8))


def test_full_size_property_checker_on_the_oracle():
    """tests/test_gpu_zz_fullsize.py's property checker, run here with the oracle standing in for the CUDA
    path on a reduced shape (it must hold for any correct implementation; on the GPU box it runs at the
    BASELINE configs[1] size)."""
    import oracle
    from tests.test_gpu_zz_fullsize import check_properties
    from tests.util import queries, random_index
    rng = np.random.default_rng(78)
    ix = random_index(rng, dim=64, nlist=64, m=8, n=40000, shuffle_ids=False)
    q = queries(rng, 256, 64)
    cache = {}

    def search(data, qq):
        if id(data) not in cache:                    # keep `data` referenced (id() of a freed shard could be reused)
            cache[id(data)] = (data, oracle.OracleIndex.from_data(data))
        return cache[id(data)][1].search(qq, k=10, nprobes=20, nthreads=4)

    check_properties(search, ix, q, 10, 20)


# ---------------------------------------------------------------- remote wire format (SURVEY.md 8f-4)
def test_remote_query_bodies_match_the_reference_mock_server_pins():
    """The request bodies pinned by the reference's own tests: test_query_vector_default_values
    (rust/lancedb/src/remote/table.rs:4650-4671) and test_query_vector_all_params (:4809-4840)."""
    from lancedb_b200 import remote
    v = np.asarray([0.1, 0.2, 0.3], np.float32)
    assert remote.build_query_body(v) == {
        "prefilter": True, "nprobes": 20, "minimum_nprobes": 20, "maximum_nprobes": 20, "lower_bound": None,
        "upper_bound": None, "k": 10, "ef": None, "refine_factor": None, "version": None,
        "vector": [float(x) for x in v]}
    got = remote.build_query_body(v, k=42, offset=10, prefilter=False, columns=["a", "b"], distance_type="Cosine",
                                  minimum_nprobes=12, maximum_nprobes=12, refine_factor=2, vector_column="my_vector",
                                  bypass_vector_index=True)
    want = {"vector_column": "my_vector", "prefilter": False, "k": 42, "offset": 10, "distance_type": "cosine",
            "bypass_vector_index": True, "columns": ["a", "b"], "nprobes": 12, "minimum_nprobes": 12,
            "maximum_nprobes": 12, "lower_bound": None, "upper_bound": None, "ef": None, "refine_factor": 2,
            "version": None, "vector": [float(x) for x in v]}
    assert got == want                                                   # (order_by is not a vector-query parameter here)
    assert remote.build_query_body(v, maximum_nprobes=None)["maximum_nprobes"] == 0      # None -> 0 = unbounded
    assert remote.build_query_body(np.zeros((2, 3), np.float32))["vector"] == [[0.0] * 3] * 2
    assert remote.build_query_body([])["vector"] == []
    assert remote.QUERY_PATH.format(name="my_table") == "/v1/table/my_table/query/"
    # the f32 -> f64 widening serde does: 0.1f32 is not 0.1f64
    assert json.loads(json.dumps(remote.build_query_body(v)))["vector"][0] == float(np.float32(0.1)) != 0.1


def test_remote_ipc_file_round_trip():
    import pyarrow as pa
    from lancedb_b200 import remote
    t = pa.table({"a": pa.array([1, 2, 3], pa.int32()), "_distance": pa.array([0.0, 0.5, 2.0], pa.float32())})
    data = remote._ipc_file(t)
    assert data[:6] == b"ARROW1"                                          # the IPC *file* framing the client expects
    assert remote.read_ipc_file(data).equals(t)


# ---------------------------------------------------------------------------------------------- Lance index files
def test_lance_index_file_round_trip_and_rejections(tmp_path):
    """SURVEY.md 8f-3: `_indices/<uuid>/{index.idx,auxiliary.idx}` -> the arrays of lgpu_index_desc.  The layout is
    recalled (no Lance file or writer exists in the reference tree), so what is pinned here is self-consistency:
    writer -> reader reproduces every array for both code layouts and paged columns, the footer / offset tables are
    range-checked, and pieces outside the handled subset fail loudly."""
    import struct
    from lancedb_b200 import lance_index as L
    from tests.util import random_index
    rng = np.random.default_rng(12)
    ix = random_index(rng, dim=32, nlist=9, m=4, metric="cosine", n=700)
    for transposed in (True, False):
        for page_rows in (0, 100):
            d = str(tmp_path / f"i{int(transposed)}{page_rows}")
            L.write_ivf_pq_index(d, ix, transposed=transposed, page_rows=page_rows)
            got = L.read_ivf_pq_index(d)
            got.validate()
            assert got.metric == "cosine" and (got.dim, got.nlist, got.m) == (32, 9, 4)
            for name in ("centroids", "codebook", "part_offsets", "codes_t", "row_ids"):
                assert np.array_equal(getattr(got, name), getattr(ix, name)), name
    # protobuf helpers: packed and unpacked repeated ints, nested messages
    msg = L.pb_int(1, 300) + L.pb_packed(2, [1, 128, 1 << 40]) + L.pb_int(2, 7) + L.pb_bytes(3, L.pb_int(1, 5))
    f = L.pb_fields(msg)
    assert f[1] == [300] and L.pb_repeated_ints(f[2]) == [1, 128, 1 << 40, 7] and L.pb_fields(f[3][0])[1] == [5]
    # rejections
    base = str(tmp_path / "i10")
    raw = open(base + "/auxiliary.idx", "rb").read()
    bad = tmp_path / "bad"; bad.mkdir()
    (bad / "index.idx").write_bytes(open(base + "/index.idx", "rb").read())
    (bad / "auxiliary.idx").write_bytes(raw[:-4] + b"XXXX")
    with pytest.raises(L.LanceFormatError, match="magic"):
        L.read_ivf_pq_index(str(bad))
    foot = bytearray(raw)
    struct.pack_into("<H", foot, len(foot) - 6, 1)                       # minor version 1: format 2.1 page layouts
    (bad / "auxiliary.idx").write_bytes(bytes(foot))
    with pytest.raises(L.LanceFormatError, match="2.1"):
        L.read_ivf_pq_index(str(bad))
    foot = bytearray(raw)
    struct.pack_into("<Q", foot, len(foot) - 40 + 8, len(raw))           # column-metadata offset table past the end
    (bad / "auxiliary.idx").write_bytes(bytes(foot))
    with pytest.raises(L.LanceFormatError, match="out of range"):
        L.read_ivf_pq_index(str(bad))
    assert L.find_index_dirs(str(tmp_path)) == []
    tbl = tmp_path / "t.lance" / "_indices" / "0000-uuid"
    tbl.mkdir(parents=True)
    L.write_ivf_pq_index(str(tbl), ix)
    assert L.find_index_dirs(str(tmp_path / "t.lance")) == [str(tbl)]


def test_lance_index_golden_fixture(tmp_path):
    """The committed Lance index files (tests/golden/lance_ivfpq_small, written by the fixture writer from the cosine
    index of ivfpq_small.npz; layout recalled -- see lance_index.py) read back to exactly those arrays, and the
    writer still produces the same bytes: a change of either side of the recalled layout shows up here."""
    from lancedb_b200 import lance_index as L
    from lancedb_b200.index import IvfPqIndexData
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    z = np.load(os.path.join(gold, "ivfpq_small.npz"))
    got = L.read_ivf_pq_index(os.path.join(gold, "lance_ivfpq_small"))
    got.validate()
    assert got.metric == "cosine" and (got.dim, got.nlist, got.m) == (32, 8, 4)
    for name in ("centroids", "codebook", "part_offsets", "codes_t", "row_ids"):
        assert np.array_equal(getattr(got, name), z[f"cosine_{name}"]), name
    ix = IvfPqIndexData(32, 8, 4, "cosine", z["cosine_centroids"], z["cosine_codebook"], z["cosine_part_offsets"],
                        z["cosine_codes_t"], z["cosine_row_ids"], None)
    L.write_ivf_pq_index(str(tmp_path / "again"), ix, transposed=True, page_rows=256)
    for f in ("index.idx", "auxiliary.idx"):
        assert open(tmp_path / "again" / f, "rb").read() == open(os.path.join(gold, "lance_ivfpq_small", f), "rb").read(), f


# ---------------------------------------------------------------------------------------------- async surface
def _stub_vector_search(monkeypatch):
    """Route Table._vector_search to the CPU oracle's flat search so the async plumbing is testable without a GPU
    (the GPU tests cover the same surface against the library)."""
    import oracle
    from lancedb_b200.table import Table

    def fake(self, queries, *, column, k, nprobes, refine_factor, distance_type, lower, upper, use_index,
             allow_mask=None, max_nprobes=0, timeout_ms=0):
        assert nprobes > 0 and k > 0
        x = self._vectors(column)
        kw = {}
        if allow_mask is not None:
            kw = dict(allow=oracle.allow_bitmap(np.nonzero(allow_mask)[0].astype(np.uint64), len(allow_mask)),
                      allow_bits=len(allow_mask))
        return oracle.flat_search(x, queries, k=k, metric=distance_type or "l2", lower=lower, upper=upper, **kw)
    monkeypatch.setattr(Table, "_vector_search", fake)


def test_async_query_surface_matches_the_sync_builder(monkeypatch):
    """python/python/lancedb/query.py:3307-3405, 3551-3723, 2867-2960: AsyncTable.query().nearest_to(...) with the
    reference's setter names and defaults, multi-vector queries tagged with query_index, concurrent coroutines."""
    import asyncio
    from lancedb_b200 import aio
    _stub_vector_search(monkeypatch)
    rng = np.random.default_rng(77)
    x = rng.standard_normal((300, 8)).astype(np.float32)
    q = rng.standard_normal((6, 8)).astype(np.float32)

    async def main():
        db = await aio.connect_async("memory://")
        t = await db.create_table("v", {"vector": x, "id": np.arange(300), "b": np.arange(300) % 7})
        assert await t.count_rows() == 300 and await t.count_rows("b = 3") == len([i for i in range(300) if i % 7 == 3])
        sync = t._table
        one = await t.query().nearest_to(q[0]).to_arrow()
        ref = sync.search(q[0]).to_arrow()
        assert one.num_rows == 10 and one.equals(ref)                                  # default limit 10
        assert "query_index" not in one.column_names
        # every setter, against the sync builder with the same request
        got = await (t.query().where("b < 5").nearest_to(q[1]).column("vector").distance_type("cosine").nprobes(7)
                     .refine_factor(2).distance_range(0.0, 1.5).limit(4).offset(1).select(["id"]).with_row_id()
                     .to_arrow())
        want = (sync.search(q[1], vector_column_name="vector").where("b < 5").distance_type("cosine").nprobes(7)
                .refine_factor(2).distance_range(0.0, 1.5).limit(4).offset(1).select(["id"]).with_row_id(True).to_arrow())
        assert got.equals(want) and got.column_names == ["id", "_distance", "_rowid"]
        post = await t.query().where("b = 2").postfilter().nearest_to(q[2]).limit(20).to_list()
        assert all(r["b"] == 2 for r in post) and len(post) < 20                      # filters the 20 results
        # several vectors: list form and add_query_vector give the same union, tagged with query_index
        multi = await t.query().nearest_to([q[0], q[1], q[2]]).limit(3).to_arrow()
        added = await t.vector_search(q[0]).add_query_vector(q[1]).add_query_vector(q[2]).limit(3).to_arrow()
        assert multi.equals(added) and multi["query_index"].to_pylist() == [0] * 3 + [1] * 3 + [2] * 3
        # concurrent coroutines (tokio workers in the reference, worker threads here)
        outs = await asyncio.gather(*[t.vector_search(v).limit(5).to_arrow() for v in q])
        for v, o in zip(q, outs):
            assert o.equals(sync.search(v).limit(5).to_arrow())
        reader = await t.vector_search(q[3]).limit(9).to_batches(max_batch_length=4)
        sizes = [b.num_rows async for b in reader]
        assert sizes == [4, 4, 1] and (await reader.read_all()).num_rows == 0
        # plain scan (host side), and the builder's validation errors surface unchanged
        scan = await t.query().where("b = 6").select(["id"]).limit(3).offset(1).to_list()
        assert [r["id"] for r in scan] == [13, 20, 27]
        with pytest.raises(ValueError, match="query_vector can not be None"):
            t.query().nearest_to(None)
        with pytest.raises(ValueError, match="minimum_nprobes must be greater than 0"):
            await t.vector_search(q[0]).minimum_nprobes(0).to_list()
        # python/python/tests/test_query.py:948-961: validated against the request's defaults (20 / 20), eagerly
        with pytest.raises(ValueError, match="maximum_nprobes must be greater than or equal to minimum_nprobes"):
            await t.vector_search(q[0]).maximum_nprobes(5).to_list()
        with pytest.raises(ValueError, match="minimum_nprobes must be less than or equal to maximum_nprobes"):
            await t.vector_search(q[0]).minimum_nprobes(100).to_list()
        with pytest.raises(ValueError, match="minimum_nprobes must be less than or equal to maximum_nprobes"):
            t.vector_search(q[0]).minimum_nprobes(30).maximum_nprobes(40)          # order matters, as in Rust
        await t.vector_search(q[0]).maximum_nprobes(40).minimum_nprobes(30).to_list()
        await t.vector_search(q[0]).maximum_nprobes(0).minimum_nprobes(300).to_list()  # 0 = no limit
        with pytest.raises(ValueError, match="No vector column found to match"):
            await t.vector_search(np.zeros(5, np.float32)).to_arrow()
        assert list(await db.table_names()) == ["v"]
    asyncio.run(main())


def test_search_on_an_empty_table_returns_no_rows():
    """python/python/tests/test_query.py:1990-2004 (issue 303): no crash, no GPU call, the result schema intact."""
    import pyarrow as pa
    import lancedb_b200 as lancedb
    db = lancedb.connect("memory://")
    schema = pa.schema([pa.field("vector", pa.list_(pa.float32(), 2)), pa.field("id", pa.int64())])
    t = db.create_table("test_empty_search", schema=schema)
    assert t.search([1.0, 2.0]).limit(5).to_list() == []
    out = t.search([[1.0, 2.0], [0.0, 1.0]]).with_row_id(True).to_arrow()
    assert out.num_rows == 0 and out.column_names == ["vector", "id", "_distance", "_rowid", "query_index"]
    with pytest.raises(ValueError, match="Either data or schema"):
        db.create_table("nothing")
