"""CPU: pin the C restatement against the COMPILED REFERENCE on fresh seeded data.  What the reference returned
for these inputs is kept as digests in tests/golden/oracle_vs_ref.json; `python tests/test_oracle_vs_ref.py`
recomputes them where oracle/_ref is built (oracle/build_ref.py).  The graph each case searches is built by the
product's host builder, which reproduces the reference's single-threaded graph byte for byte (checked against the
digest of the reference's graph, before and after deletions).  Also checks the documented equivalence used to work
around the reference's knn_query segfault (SURVEY.md section 0.4)."""
import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repository root on sys.path when run as a script)
import oracle as O
from annlite_b200.engine import Engine
from helpers import digest, graph_digest, knn_digest, load_golden_json, save_golden_json

GOLDEN_FILE = 'oracle_vs_ref.json'
CASES = [
    (3000, 32, 4, 256, 'euclidean', 21, False),
    (3000, 48, 8, 256, 'cosine', 22, False),
    (2000, 16, 4, 12, 'euclidean', 23, True),
    (2000, 24, 4, 400, 'inner_product', 24, False),
]
SEARCHES = [(10, 48), (1, 10), (30, 20)]     # (k, ef)


def case_key(N, D, M, Ks, metric, seed, ties):
    return f'{N}-{D}-{M}-{Ks}-{metric}-{seed}-{ties}'


def case_inputs(N, D, M, Ks, metric, seed, ties):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D)).astype(np.float32)
    Q = rng.standard_normal((80, D)).astype(np.float32)
    if ties:
        X, Q = np.round(X), np.round(Q)
    ds = D // M
    cb = np.stack([X[rng.choice(N, Ks, replace=False), m * ds:(m + 1) * ds] for m in range(M)]).astype(np.float32)
    labels = rng.permutation(N).astype(np.uint64) * 3 + 1
    allow = np.sort(labels[rng.random(N) < 0.4])
    return X, Q, cb, labels, allow


def pre(x, metric):
    """HnswIndex.pre_process (hnsw/index.py:28-29)."""
    return O.l2_normalize(x).astype(np.float32) if metric == 'cosine' else x


def reference_digests(N, D, M, Ks, metric, seed, ties):
    """What the compiled reference returns for case_inputs (needs oracle/_ref)."""
    from oracle import ref_driver as R
    X, Q, cb, labels, allow = case_inputs(N, D, M, Ks, metric, seed, ties)
    codec = R.RefCodec(cb, metric)
    idx = R.RefHnswIndex(codec, metric, capacity=N, ef_search=48)
    idx.add_with_ids(X, labels, num_threads=1)
    Qp = idx._pre(Q)
    T = codec.get_dist_mat(Qp)
    out = {'tables': digest(np.asarray(T, dtype=np.float32)), 'graph': graph_digest(idx.state())}
    for k, ef in SEARCHES:
        idx.ef_search = ef
        out[f'knn_{k}_{ef}'] = knn_digest(*idx.knn_query(Q, k, num_threads=1, tables=T))
        # multi-threaded and "filter = all ids" routes (SURVEY 0.3 / 0.4)
        out[f'knn_{k}_{ef}_8_threads'] = knn_digest(*idx.knn_query(Q, k, num_threads=8, tables=T))
        out[f'knn_{k}_{ef}_filter_all'] = knn_digest(*idx.knn_query(Q, k, indices=labels, tables=T))
    idx.ef_search = 48
    rl, rd = idx.knn_query(Q, 10, indices=allow, tables=T)
    # None: a binary-fuse false positive leaked into the reference result, which the oracle does not model
    out['filtered'] = knn_digest(rl, rd) if np.isin(rl, allow).all() else None
    for l in labels[::11]:
        idx._index.mark_deleted(int(l))
    out['graph_deleted'] = graph_digest(idx.state())
    out['knn_deleted'] = knn_digest(*idx.knn_query(Q, 10, num_threads=1, tables=T))
    codes = O.Graph.from_state(idx.state(), M, Ks).codes()
    out['scan_q3'] = digest(np.asarray(R.pq_bind().dist_pqcodes_to_codebooks(T[3], codes), dtype=np.float32))
    out['single_table_q5'] = digest(np.asarray(codec.precompute_adc(Qp[5]), dtype=np.float32))
    return out


def reference_linear_scan_digests():
    from oracle import ref_driver as R
    X, cb, Qs = linear_scan_inputs()
    codec = R.RefCodec(cb, 'euclidean')
    codes = codec.encode(X)
    out = []
    for q in Qs:
        d, i = R.ref_pq_linear_scan(codec, codes, q, 10)
        out.append({'dists': digest(np.asarray(d, dtype=np.float32)), 'sorted_ids': digest(np.sort(np.asarray(i, dtype=np.int64)))})
    return out


@pytest.mark.parametrize('N,D,M,Ks,metric,seed,ties', CASES)
def test_oracle_equals_compiled_reference(N, D, M, Ks, metric, seed, ties):
    ref = load_golden_json(GOLDEN_FILE)[case_key(N, D, M, Ks, metric, seed, ties)]
    X, Q, cb, labels, allow = case_inputs(N, D, M, Ks, metric, seed, ties)
    Xp, Qp = pre(X, metric), pre(Q, metric)
    To = O.adc_table(Qp, cb, metric)
    assert digest(To) == ref['tables']
    # the graph the reference built (RefHnswIndex defaults: M=16, ef_construction=200), rebuilt by the host builder
    e = Engine(D, M, Ks, metric, device=-1)
    e.init_graph(N, M=16, ef_construction=200)
    e.add_items_with_tables(O.encode(Xp, cb), O.adc_table(Xp, cb, metric), labels, num_threads=1)
    assert graph_digest(e.get_graph()) == ref['graph']
    g = O.Graph.from_state(e.get_graph(), M, Ks)
    for k, ef in SEARCHES:
        ol, od, found = O.hnsw_search(g, To, k, ef)
        got = knn_digest(ol, od)
        assert got == ref[f'knn_{k}_{ef}']
        assert got == ref[f'knn_{k}_{ef}_8_threads'] and got == ref[f'knn_{k}_{ef}_filter_all']
    if ref['filtered'] is not None:
        ol, od, _ = O.hnsw_search(g, To, 10, 48, filter_labels=allow)
        assert knn_digest(ol, od) == ref['filtered']
    for l in labels[::11]:
        e.mark_deleted(int(l))
    assert graph_digest(e.get_graph()) == ref['graph_deleted']
    g = O.Graph.from_state(e.get_graph(), M, Ks)
    ol, od, _ = O.hnsw_search(g, To, 10, 48)
    assert knn_digest(ol, od) == ref['knn_deleted']
    # exhaustive scan + single-query table
    assert digest(O.scan(To[3], g.codes())) == ref['scan_q3']
    assert digest(O.adc_table(Qp[5:6], cb, 'euclidean')[0]) == ref['single_table_q5']


def linear_scan_inputs():
    rng = np.random.default_rng(9)
    N, D, M, Ks = 4000, 32, 8, 256
    X = rng.standard_normal((N, D)).astype(np.float32)
    cb = np.stack([X[rng.choice(N, Ks, replace=False), m * 4:(m + 1) * 4] for m in range(M)]).astype(np.float32)
    return X, cb, rng.standard_normal((5, D)).astype(np.float32)


def test_ref_linear_scan_equals_oracle_topk():
    ref = load_golden_json(GOLDEN_FILE)['linear_scan']
    X, cb, Qs = linear_scan_inputs()
    codes = O.encode(X, cb)
    for q, r in zip(Qs, ref, strict=True):
        oi, od = O.scan_topk(O.adc_table(q[None], cb), codes, 10)
        assert digest(od[0]) == r['dists']
        assert digest(np.sort(oi[0].astype(np.int64))) == r['sorted_ids'] or len(set(od[0].tolist())) < 10


if __name__ == '__main__':
    save_golden_json(GOLDEN_FILE, {**{case_key(*c): reference_digests(*c) for c in CASES},
                                   'linear_scan': reference_linear_scan_digests()})
