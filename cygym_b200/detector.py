"""Host side of the trained detector (defender actions 10 / 5; volt_typhoon_env.py:945-962, :1020-1069,
CDSimulator.py:681-723).

The reference's Detector is scikit-learn's IsolationForest(n_estimators=2, max_samples=256) fitted on the (from, to)
pairs of the last <= 2000 hop-log records.  Here the FIT is scikit-learn's, drawing from numpy's global random stream;
with a seed per env the same fit also runs on the device (VectorCyberDefenseEnv.fit_detectors, csrc/cyg_iforest.cuh),
into the same slot format, word for word.  What the step kernels need is PREDICT, and that is two tree walks plus a
threshold on a function of the two leaves reached.  `pack_detector` ships exactly that: the trees, and the forest's verdict for every
PAIR of leaves, computed here with the same numpy expressions scikit-learn evaluates (_compute_score_samples,
decision_function, predict of sklearn/ensemble/_iforest.py, 1.9) -- so the device never evaluates 2 ** x.
"""
import numpy as np

from ._capi import DET_TABLE, DET_TREE0, DET_TREE_STRIDE, DET_WORDS

MAX_NODES = 512


def fit_detector(records, seed=None):
    """records: int array [n, 2] of (from_device, to_device), in log order (what Detector.train builds, CDSimulator.py:
    691-692).  seed: numpy's GLOBAL stream is seeded with it first -- the reference's IsolationForest has
    random_state=None, i.e. it draws from that stream; parity runs seed it identically on both sides."""
    from sklearn.ensemble import IsolationForest
    if seed is not None:
        np.random.seed(int(seed))
    model = IsolationForest(n_estimators=2, max_samples=256, n_jobs=1)
    model.fit([[int(a), int(b)] for a, b in np.asarray(records).reshape(-1, 2)])
    return model


def pack_detector(model):
    """A fitted IsolationForest -> one detector slot (uint32[CYG_DET_WORDS])."""
    from sklearn.ensemble._iforest import _average_path_length
    slot = np.zeros(DET_WORDS, np.uint32)
    assert len(model.estimators_) == 2
    leaf_vals = []
    for t, (est, feats) in enumerate(zip(model.estimators_, model.estimators_features_)):
        tr = est.tree_
        n = tr.node_count
        if n > MAX_NODES:
            raise ValueError(f"tree of {n} nodes (max_samples > 256?)")
        is_leaf = tr.children_left == -1
        leaf_nodes = np.nonzero(is_leaf)[0]
        leaf_idx = np.full(n, 0, np.int64)
        leaf_idx[leaf_nodes] = np.arange(len(leaf_nodes))
        base = DET_TREE0 + t * DET_TREE_STRIDE
        thr = np.ascontiguousarray(tr.threshold, np.float64).view(np.uint32).reshape(n, 2)
        for i in range(n):
            slot[base + 4 * i + 0], slot[base + 4 * i + 1] = thr[i, 0], thr[i, 1]
            if is_leaf[i]:
                slot[base + 4 * i + 2] = 0
                slot[base + 4 * i + 3] = 2 | (int(leaf_idx[i]) << 16)
            else:
                slot[base + 4 * i + 2] = int(tr.children_left[i]) | (int(tr.children_right[i]) << 16)
                slot[base + 4 * i + 3] = int(feats[int(tr.feature[i])])
        # what _parallel_compute_tree_depths adds for a sample that lands in this leaf
        leaf_vals.append(model._decision_path_lengths[t][leaf_nodes] + model._average_path_length_per_tree[t][leaf_nodes] - 1.0)
    L0, L1 = len(leaf_vals[0]), len(leaf_vals[1])
    depths = np.zeros((L0, L1), order="f")
    depths += leaf_vals[0][:, None]
    depths += leaf_vals[1][None, :]
    denominator = len(model.estimators_) * _average_path_length([model._max_samples])
    scores = 2 ** (-np.divide(depths, denominator, out=np.ones_like(depths), where=denominator != 0))
    anomaly = ((-scores) - model.offset_) < 0  # decision_function < 0 -> predict == -1 -> "A" (CDSimulator.py:722-723)
    slot[0] = L1
    bits = np.zeros((L0 * L1 + 31) // 32, np.uint32)
    flat = np.nonzero(anomaly.reshape(-1))[0]
    np.bitwise_or.at(bits, flat >> 5, (np.uint32(1) << (flat & 31).astype(np.uint32)))
    slot[DET_TABLE: DET_TABLE + len(bits)] = bits
    return slot


def predict_packed(slot, from_dev, to_dev):
    """The kernels' predict, on the host (tests): True = "A"."""
    leaves = []
    for t in range(2):
        base, node = DET_TREE0 + t * DET_TREE_STRIDE, 0
        while True:
            w = slot[base + 4 * node: base + 4 * node + 4]
            feat = int(w[3]) & 0xFFFF
            if feat >= 2:
                leaves.append(int(w[3]) >> 16)
                break
            thr = np.array([w[0], w[1]], np.uint32).view(np.float64)[0]
            x = float(from_dev if feat == 0 else to_dev)
            node = (int(w[2]) & 0xFFFF) if x <= thr else (int(w[2]) >> 16)
    idx = leaves[0] * int(slot[0]) + leaves[1]
    return bool((int(slot[DET_TABLE + (idx >> 5)]) >> (idx & 31)) & 1)
