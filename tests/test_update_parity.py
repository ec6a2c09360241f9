"""CPU: re-adding existing labels (hnswalg.h:958-1096 updatePoint / repairConnectionsForUpdate -- what
AnnLite.update does through add_with_ids, annlite/container.py:343-347) reproduces the compiled reference's
graph byte for byte (single-threaded), including the un-delete of a re-added deleted label.  The reference's
graphs and search results for these inputs are kept as digests in tests/golden/update_parity.json;
`python tests/test_update_parity.py` recomputes them where oracle/_ref is built (oracle/build_ref.py)."""
import numpy as np
import pytest

import conftest  # noqa: F401  (puts the repository root on sys.path when run as a script)
import oracle as O
from annlite_b200.engine import Engine
from helpers import digest, graph_digest, knn_digest, load_golden_json, save_golden_json

GOLDEN_FILE = 'update_parity.json'
METRICS = [('euclidean', 1), ('cosine', 2), ('inner_product', 3)]
N, D, M, Ks = 1500, 32, 4, 64


def pre(x, metric):
    """HnswIndex.pre_process (hnsw/index.py:28-29)."""
    return O.l2_normalize(x).astype(np.float32) if metric == 'cosine' else x


def update_inputs(metric, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, D)).astype(np.float32)
    Xn = pre(X, metric)
    ds = D // M
    cb = np.stack([Xn[rng.choice(N, Ks, replace=False), m * ds:(m + 1) * ds] for m in range(M)]).astype(np.float32)
    labels = rng.permutation(N).astype(np.uint64) + 3
    # 40 stored points get new vectors, mixed with 5 brand-new labels in the same call
    upd = rng.choice(N, 40, replace=False)
    new_lab = np.concatenate([labels[upd], np.arange(10 ** 6, 10 ** 6 + 5, dtype=np.uint64)])
    Y = rng.standard_normal((45, D)).astype(np.float32)
    order = rng.permutation(45)
    new_lab, Y = new_lab[order], Y[order]
    # then 6 of them are deleted and two of those re-added
    deleted = labels[upd[:6]]
    Z = rng.standard_normal((2, D)).astype(np.float32)
    back = labels[upd[:2]]
    Q = rng.standard_normal((30, D)).astype(np.float32)
    return dict(X=X, cb=cb, labels=labels, new_lab=new_lab, Y=Y, deleted=deleted, Z=Z, back=back, Q=Q)


def reference_digests(metric, seed):
    """The compiled reference's graph after each step and its search over the last one (needs oracle/_ref)."""
    from oracle import ref_driver as R
    a = update_inputs(metric, seed)
    codec = R.RefCodec(a['cb'], metric)
    ref = R.RefHnswIndex(codec, metric, capacity=N + 10, ef_construction=60, ef_search=32, max_connection=8)
    ref.add_with_ids(a['X'], a['labels'], num_threads=1)
    out = {'build': graph_digest(ref.state())}
    ref.add_with_ids(a['Y'], a['new_lab'], num_threads=1)
    out['update'] = graph_digest(ref.state())
    for l in a['deleted']:
        ref._index.mark_deleted(int(l))
    ref.add_with_ids(a['Z'], a['back'], num_threads=1)
    out['readd'] = graph_digest(ref.state())
    T = codec.get_dist_mat(ref._pre(a['Q']))
    out['tables'] = digest(np.asarray(T, dtype=np.float32))
    out['knn'] = knn_digest(*ref.knn_query(a['Q'], 5, num_threads=1, tables=T))
    return out


def reference_entry_point_digest():
    from oracle import ref_driver as R
    cb, x = entry_point_inputs()
    codec = R.RefCodec(cb, 'euclidean')
    ref = R.RefHnswIndex(codec, 'euclidean', capacity=8, ef_construction=10, max_connection=4)
    ref.add_with_ids(x, np.array([7], dtype=np.uint64), num_threads=1)
    ref.add_with_ids(x * 2, np.array([7], dtype=np.uint64), num_threads=1)     # single element: early return (:965)
    return graph_digest(ref.state())


def add(e, x, labels, cb, metric):
    """HnswIndex.add_with_ids (hnsw/index.py:125-137) with the oracle's encode and tables."""
    xp = pre(x, metric)
    e.add_items_with_tables(O.encode(xp, cb), O.adc_table(xp, cb, metric), labels, num_threads=1)


@pytest.mark.parametrize('metric,seed', METRICS)
def test_update_existing_labels_matches_reference(metric, seed):
    ref = load_golden_json(GOLDEN_FILE)[f'{metric}-{seed}']
    a = update_inputs(metric, seed)
    cb = a['cb']
    e = Engine(D, M, Ks, metric, device=-1)
    e.init_graph(N + 10, M=8, ef_construction=60)
    add(e, a['X'], a['labels'], cb, metric)
    assert graph_digest(e.get_graph()) == ref['build']

    # 1) update 40 stored points with new vectors, mixed with 5 brand-new labels in the same call
    add(e, a['Y'], a['new_lab'], cb, metric)
    assert e.get_graph()['cur_element_count'] == N + 5
    assert graph_digest(e.get_graph()) == ref['update']

    # 2) delete a few labels, then re-add two of them: the mark is cleared and the point re-linked
    for l in a['deleted']:
        e.mark_deleted(int(l))
    add(e, a['Z'], a['back'], cb, metric)
    assert graph_digest(e.get_graph()) == ref['readd']
    g = O.Graph.from_state(e.get_graph(), M, Ks)
    assert g.links0()[2].sum() == 4

    # 3) searches over the updated graph agree (oracle on our graph == reference on its own)
    T = O.adc_table(pre(a['Q'], metric), cb, metric)
    assert digest(T) == ref['tables']
    ol, od, _ = O.hnsw_search(g, T, 5, 32)
    assert knn_digest(ol, od) == ref['knn']


def entry_point_inputs():
    cb = np.random.default_rng(0).standard_normal((2, 8, 4)).astype(np.float32)
    x = np.random.default_rng(1).standard_normal((1, 8)).astype(np.float32)
    return cb, x


def test_update_only_entry_point_graph():
    cb, x = entry_point_inputs()
    e = Engine(8, 2, 8, 'euclidean', device=-1)
    e.init_graph(8, M=4, ef_construction=10)
    for v in (x, x * 2):
        add(e, v, np.array([7], dtype=np.uint64), cb, 'euclidean')
    assert graph_digest(e.get_graph()) == load_golden_json(GOLDEN_FILE)['entry_point_only']
    assert e.element_count == 1


if __name__ == '__main__':
    save_golden_json(GOLDEN_FILE, {**{f'{m}-{s}': reference_digests(m, s) for m, s in METRICS},
                                   'entry_point_only': reference_entry_point_digest()})
