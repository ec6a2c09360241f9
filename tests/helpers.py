import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def tie_aware_rows(labels, dists, ref_labels, ref_dists):
    """Per-row verdict comparing a result against the oracle/reference.

    'exact'  : labels and fp32 distances identical
    'tie'    : distances bit-identical, labels differ only where equal distances make the order
               (or the choice at the k-th boundary) ambiguous -- the only freedom the GPU walk takes
    'diff'   : anything else
    """
    out = []
    k = labels.shape[1]
    for r in range(labels.shape[0]):
        if np.array_equal(labels[r], ref_labels[r]) and np.array_equal(bits(dists[r]), bits(ref_dists[r])):
            out.append('exact')
            continue
        if not np.array_equal(bits(dists[r]), bits(ref_dists[r])):
            out.append('diff')
            continue
        ok = True
        for p in np.nonzero(labels[r] != ref_labels[r])[0]:
            d = dists[r, p]
            tied = (p > 0 and dists[r, p - 1] == d) or (p + 1 < k and dists[r, p + 1] == d) or p == k - 1
            ok &= bool(tied)
        out.append('tie' if ok else 'diff')
    return out


def recall(pred, truth):
    """annlite/utils.py:52-71: |pred ∩ truth| / |truth| averaged over queries."""
    return float(np.mean([len(set(p.tolist()) & set(t.tolist())) / len(t) for p, t in zip(pred, truth)]))


def digest(*arrays):
    """SHA-256 over the dtype, shape and bytes of each array: how a test compares with outputs of the compiled
    reference that are kept in tests/golden as digests rather than as arrays."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f'{a.dtype.str}{a.shape}'.encode())
        h.update(a.tobytes())
    return h.hexdigest()


def knn_digest(labels, dists):
    return digest(np.asarray(labels, dtype=np.uint64), np.asarray(dists, dtype=np.float32))


def graph_digest(st):
    """Digest of an exported graph (Index.__getstate__()[0] or Engine.get_graph()): records, upper-level lists,
    levels, size, top level and entry point."""
    return digest(np.asarray(st['data_level0']).view(np.uint8), np.asarray(st['link_lists']).view(np.uint8),
                  np.asarray(st['element_levels'], dtype=np.int32)[:int(st['cur_element_count'])],
                  np.array([st['cur_element_count'], st['max_level'], st['enterpoint_node']], dtype=np.int64))


def load_golden_json(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def save_golden_json(name, obj):
    with open(os.path.join(GOLDEN, name), 'w') as f:
        json.dump(obj, f, indent=1, sort_keys=True)
        f.write('\n')
