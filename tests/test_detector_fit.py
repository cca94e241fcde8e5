"""The device restatement of the detector fit (cygym_b200/csrc/cyg_iforest.cuh) against scikit-learn / numpy, through
the host build of the device source (tests/emu/cyg_emu_iforest.cpp).  Runs on the CPU."""
import os
import re
import warnings

import numpy as np
import pytest

pytest.importorskip("sklearn")

from cygym_b200 import _capi as K  # noqa: E402
from cygym_b200 import detector as DET  # noqa: E402
from tests.emu import iforest as emu  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEEDS = [0, 1, 12345, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1]


def _ring(recs, log_cap=2048):
    """Records [n, 2] (the whole log, in order) -> a ring of log_cap words holding them at i % log_cap."""
    ring = np.zeros(log_cap, np.uint32)
    n = len(recs)
    ring[np.arange(n) % log_cap] = (recs[:, 0] | (recs[:, 1] << 16)).astype(np.uint32)
    return ring


def _host_slot(recs, seed):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # max_samples > n_samples
        return DET.pack_detector(DET.fit_detector(recs[-K.DET_WINDOW:], seed))


def _check(recs, seed, log_cap=2048):
    want = _host_slot(recs, seed)
    got = emu.fit_detector(_ring(recs, log_cap), len(recs), seed)
    bad = np.nonzero(want != got)[0]
    assert bad.size == 0, f"n={len(recs)} seed={seed}: {bad.size} words differ, first at {bad[:8]}"


# ---- numpy's legacy stream -------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", SEEDS + [987654321, 4000000000])
def test_uniform_and_seed_draws(seed):
    rs = np.random.RandomState(seed)
    want = list(rs.uniform(size=700)) + list(rs.randint(2 ** 31 - 1, size=3))
    got = emu.np_stream(seed, [("uniform", None)] * 700 + [("bounded", 2 ** 31 - 2)] * 3)
    assert np.array_equal(np.array(want, np.float64), got)


@pytest.mark.parametrize("seed", SEEDS)
def test_randint_rejection(seed):
    """randint(0, k) for k at and just above powers of two, where the masked rejection discards up to half the draws."""
    ks = [k for p in range(1, 31) for k in (2 ** p, 2 ** p + 1)] + [3, 257, 258, 1999, 2000]
    rs = np.random.RandomState(seed)
    want = [rs.randint(0, k) for k in ks]
    got = emu.np_stream(seed, [("bounded", k - 1) for k in ks])
    assert np.array_equal(np.array(want, np.float64), got)


@pytest.mark.parametrize("seed", SEEDS)
def test_permutation(seed):
    rs = np.random.RandomState(seed)
    want = np.concatenate([rs.permutation(n) for n in (1, 2, 259, 2000)])
    got = emu.np_stream(seed, [("permutation", n) for n in (1, 2, 259, 2000)])
    assert np.array_equal(want.astype(np.float64), got)


# ---- whole slots -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 17, 255, 256, 257, 258, 259, 300, 1999, 2000])
@pytest.mark.parametrize("M", [20, 100, 128])
def test_slot_uniform_records(n, M):
    rng = np.random.default_rng(1000 * n + M)
    recs = rng.integers(0, M, size=(n, 2))
    for seed in (0, int(rng.integers(0, 2 ** 32))):
        _check(recs, seed)


def test_slot_reads_only_the_tail_of_a_long_log():
    rng = np.random.default_rng(5)
    recs = rng.integers(0, 100, size=(5000, 2))  # wraps a 2048-record ring twice; the fit reads the last 2000
    for seed in (3, 2 ** 32 - 1):
        _check(recs, seed)
    _check(recs[:2001], 11, log_cap=2000)


@pytest.mark.parametrize("case", ["few_senders", "identical", "constant_from", "constant_to", "duplicates"])
def test_slot_degenerate_logs(case):
    rng = np.random.default_rng(sum(map(ord, case)))
    for n in (2, 40, 256, 600, 2000):
        recs = rng.integers(0, 100, size=(n, 2))
        if case == "few_senders":
            recs[:, 0] = rng.choice([3, 71], size=n)
        elif case == "identical":  # both features constant: the root is a leaf
            recs[:] = (7, 42)
        elif case == "constant_from":
            recs[:, 0] = 9
        elif case == "constant_to":
            recs[:, 1] = 0
        else:
            recs = rng.choice(rng.integers(0, 100, size=(4, 2)), size=n, axis=0)
        for seed in (0, 77, 2 ** 32 - 1):
            _check(recs, seed)


def test_epsilon_leaf_search():
    """The builder's leaf tests `impurity <= EPSILON` (a node of >= 2 samples whose targets are equal to ~1e-8) and
    `improvement + EPSILON < 0`.  The targets are numpy uniforms, so a node of >= 2 samples with impurity <= 2.2e-16
    needs two uniforms within ~3e-8 of each other in one small node.  This search fits 2-record logs (the root's
    impurity is ((y0 - y1) / 2) ** 2) and 40-record logs for 300 seeds each and found no such node, nor a negative
    improvement: no fixed case exercises these branches, and every trial is still compared word for word."""
    found = 0
    rng = np.random.default_rng(17)
    for n in (2, 40):
        for seed in range(300):
            recs = rng.integers(0, 30, size=(n, 2))
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                model = DET.fit_detector(recs, seed)
            for est in model.estimators_:
                tr = est.tree_
                leaf = tr.children_left == -1
                found += int(np.any(leaf & (tr.n_node_samples >= 2) & (tr.impurity <= np.finfo(float).eps)))
            got = emu.fit_detector(_ring(recs), n, seed)
            assert np.array_equal(DET.pack_detector(model), got), (n, seed)
    assert found == 0, "a case was found: commit it as a fixed parameter"


# ---- the verdict rule and the c(k) table -----------------------------------------------------------------------
def test_verdict_rule_boundary():
    """The device sets a verdict bit when q <= 1 - 2**-52 instead of evaluating 2 ** -q > 0.5."""
    q_in, q_out = 1.0 - 2.0 ** -52, 1.0 - 2.0 ** -53
    assert np.power(2.0, -np.array([q_in]))[0] > 0.5
    assert np.power(2.0, -np.array([q_out]))[0] == 0.5
    assert np.power(2.0, -np.array([1.0]))[0] == 0.5
    assert np.nextafter(q_in, 1.0) == q_out  # nothing in between


def test_average_path_length_table():
    from sklearn.ensemble._iforest import _average_path_length
    src = open(os.path.join(ROOT, "cygym_b200", "csrc", "cyg_iforest.cuh")).read()
    body = re.search(r"#define CYG_APL_TABLE \{(.*?)\n\}", src, re.S).group(1)
    words = np.array([int(x, 16) for x in re.findall(r"0x([0-9a-f]{16})ull", body)], np.uint64)
    assert words.size == 257
    assert np.array_equal(words, _average_path_length(np.arange(257)).view(np.uint64))


def test_window_refusal():
    with pytest.raises(ValueError):
        emu.fit_detector(np.zeros(30, np.uint32), 31, 0)
