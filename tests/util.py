"""Test helpers: synthetic IVF_PQ indexes with arbitrary (untrained) contents.  Parity does
not depend on index quality -- the CUDA path and the oracle consume the identical arrays --
so random centroids / codebooks / codes exercise the arithmetic just as well and let the
tests shape edge cases (empty, tiny and multi-tile partitions)."""
import numpy as np

from lancedb_b200.index import IvfPqIndexData


def random_index(rng, *, dim, nlist, m, metric="l2", sizes=None, n=None, with_vectors=False, scale=1.0,
                 shuffle_ids=True):
    dsub = dim // m
    if sizes is None:
        w = rng.random(nlist) + 0.2
        sizes = np.floor(w / w.sum() * n).astype(np.int64)
        sizes[0] += n - sizes.sum()
    sizes = np.asarray(sizes, np.int64)
    n = int(sizes.sum())
    cent = (rng.standard_normal((nlist, dim)) * scale).astype(np.float32)
    if metric == "cosine":
        cent /= np.linalg.norm(cent, axis=1, keepdims=True)
    cb = (rng.standard_normal((m, 256, dsub)) * 0.5 * scale).astype(np.float32)
    off = np.zeros(nlist + 1, np.uint64)
    off[1:] = np.cumsum(sizes)
    codes_t = rng.integers(0, 256, size=n * m, dtype=np.uint8)
    # ascending row ids inside each partition (lance scan order), interleaved across partitions
    ids = np.empty(n, np.uint64)
    perm = rng.permutation(n).astype(np.uint64) if shuffle_ids else np.arange(n, dtype=np.uint64)
    for p in range(nlist):
        a, b = int(off[p]), int(off[p + 1])
        ids[a:b] = np.sort(perm[a:b])
    vec = None
    if with_vectors:
        vec = (rng.standard_normal((n, dim)) * scale).astype(np.float32)
    ix = IvfPqIndexData(dim, nlist, m, metric, cent, cb, off, codes_t, ids, vec)
    ix.validate()
    return ix


def queries(rng, B, dim, scale=1.0):
    return (rng.standard_normal((B, dim)) * scale).astype(np.float32)


GOLDEN_CASES = {"plain": dict(k=7, nprobes=3), "range": dict(k=7, nprobes=3, lower=2.0, upper=30.0),
                "refine": dict(k=5, nprobes=3, refine_factor=3), "prefilter": dict(k=7, nprobes=4)}


def load_golden(metric):
    """tests/golden/ivfpq_small.npz (made by tests/golden/make_golden.py): index, queries, and per case the
    search kwargs + the committed (ids, dist, cnt)."""
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ivfpq_small.npz"))
    g = lambda name: z[f"{metric}_{name}"]
    ix = IvfPqIndexData(32, 8, 4, metric, g("centroids"), g("codebook"), g("part_offsets"), g("codes_t"), g("row_ids"),
                        g("vectors"))
    ix.validate()
    cases = {}
    for name, kw in GOLDEN_CASES.items():
        kw = dict(kw)
        if name == "prefilter":
            kw.update(allow=g("allow"), allow_bits=600)
        cases[name] = (kw, (g(f"{name}_ids"), g(f"{name}_dist"), g(f"{name}_cnt")))
    flat = (g("flat_ids"), g("flat_dist"), g("flat_cnt"))
    return ix, g("queries"), cases, flat


def bench_dumps(tmp_path, *args, runs=2):
    """Runs `bench.py --dump-outputs` `runs` times, each with a temporary directory of its own (so every run trains
    its index afresh) and returns the dumped arrays of each run as {name: array} plus its JSON line."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = []
    for r in range(runs):
        tmp, dump = tmp_path / f"tmp{r}", tmp_path / f"dump{r}"
        tmp.mkdir()
        proc = subprocess.run([sys.executable, os.path.join(root, "bench.py"), *args, "--dump-outputs", str(dump)],
                              capture_output=True, text=True, timeout=900, cwd=root, env=dict(os.environ, TMPDIR=str(tmp)))
        assert proc.returncode == 0, proc.stderr[-2000:]
        out.append(({f[:-4]: np.load(dump / f) for f in sorted(os.listdir(dump))}, json.loads(proc.stdout)))
    return out


def same_result(got, want):
    gi, gd, gc = got
    wi, wd, wc = want
    return (np.array_equal(gc, wc) and np.array_equal(gi, wi)
            and np.array_equal(np.asarray(gd, np.float32).view(np.uint32), np.asarray(wd, np.float32).view(np.uint32)))
