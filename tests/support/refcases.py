"""What the parity tests compare with the reference, as functions of the library that runs them.

Every function drives one library (`impl`: "b200" or "reference") through the public C API and returns
a dict of arrays.  tools/make_golden.py runs them on the unmodified reference (oracle/_ref) and stores
the results in tests/golden/reference_cases.npz; the tests run them on this library and compare, so
they need no reference binary.  Large state vectors are kept as a fixed, seeded sample of nodes
(`idx`); orderings of large graphs as a SHA-256 digest.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np

from aprilsam_b200 import datasets
from aprilsam_b200 import harness as H

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden", "reference_cases.npz")
SAMPLE = 128  # nodes kept per state vector of a large graph


def sample(n: int, k: int = SAMPLE, seed: int = 0) -> np.ndarray:
    """A fixed subset of node ids of an n-node graph (all of them when n <= k); always holds node n - 1."""
    if n <= k:
        return np.arange(n, dtype=np.int32)
    rng = np.random.default_rng(seed)
    return np.union1d(rng.choice(n - 1, size=k - 1, replace=False), [n - 1]).astype(np.int32)


def digest(a) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a, dtype="<i4").tobytes()).digest(), dtype=np.uint8)


def load(prefix: str) -> dict:
    """The stored reference result of one case."""
    z = np.load(GOLDEN)
    return {k[len(prefix) + 1:]: z[k] for k in z.files if k.startswith(prefix + "/")}


def _stack(rows: list) -> tuple[np.ndarray, np.ndarray]:
    """Ragged list of (n_i, 3) arrays -> rows concatenated + offsets."""
    off = np.cumsum([0] + [len(r) for r in rows]).astype(np.int64)
    return np.concatenate(rows).reshape(-1, 3), off


# ---------------------------------------------------------------------------------------------
# batch solves
# ---------------------------------------------------------------------------------------------
def batch_once(impl: str, d) -> dict:
    """One april_graph_cholesky call from the initial estimate: ordering, elimination tree, states, chi2."""
    with H.Harness(impl) as h:
        h.load_full(d)
        h.batch()
        return {"order": h.ordering(), "parents": h.tree_parents(), "states": h.states(), "chi2": np.array(h.chi2())}


def batch_iters(impl: str, d, iters: int) -> dict:
    """`iters` consecutive batch calls; sampled states and chi2 after each, the ordering of the first."""
    idx = sample(d.n_nodes)
    states, chi2 = [], []
    with H.Harness(impl) as h:
        h.load_full(d)
        chi2_0 = h.chi2()
        for it in range(iters):
            h.batch()
            if it == 0:
                order = digest(h.ordering())
            states.append(h.states()[idx])
            chi2.append(h.chi2())
    return {"idx": idx, "states": np.array(states), "chi2_0": np.array(chi2_0), "chi2": np.array(chi2), "order": order}


# ---------------------------------------------------------------------------------------------
# replays
# ---------------------------------------------------------------------------------------------
def replay_lockstep(impl: str, d, checkpoints, per_cp: int) -> dict:
    """Demo-protocol replay stopped at every checkpoint: naffected / start_over / chi2 of every step,
    `per_cp` sampled node states at every checkpoint (seeded by the checkpoint)."""
    chi2, info, idx, rows = [], [], [], []
    with H.Harness(impl) as h:
        h.replay_begin(d)
        for k in checkpoints:
            c, _, i = h.replay_to(int(k))
            chi2.append(c)
            info.append(i)
            s = sample(h.n_nodes, per_cp, seed=int(k))
            idx.append(s)
            rows.append(h.states()[s])
    info = np.concatenate(info)
    states, off = _stack(rows)
    return {"chi2": np.concatenate(chi2), "naffected": info[:, 0].copy(), "start_over": info[:, 1].copy(),
            "idx": np.concatenate(idx), "states": states, "off": off, "checkpoints": np.asarray(checkpoints)}


def sparse_bulk_then_incremental(impl: str, poses: int = 30000, s0: int = 29700, step: int = 25, n_inc: int = 200) -> dict:
    """The first s0 poses of a sparse synthetic graph loaded at once at ground truth and batch-solved twice,
    then the next n_inc poses appended one by one (states sampled every `step` poses)."""
    d = datasets.manhattan_sparse(poses, seed=1)
    sub = d.head(s0)
    naff, so, rows = [], [], []
    with H.Harness(impl) as h:
        h.replay_begin(d)
        h.load_full(sub)
        h.set_states(sub.truth)
        h.batch()
        h.batch()
        bulk_idx = sample(s0)
        bulk = h.states()[bulk_idx]
        cps = list(range(s0 + step, s0 + n_inc + 1, step))
        for k in cps:
            _, _, i = h.replay_to(k, want_chi2=False)
            naff.append(i[:, 0])
            so.append(i[:, 1])
            rows.append(h.states()[sample(k, 32, seed=k)])
        chi2 = h.chi2()
    states, off = _stack(rows)
    return {"bulk_idx": bulk_idx, "bulk_states": bulk, "checkpoints": np.array(cps), "naffected": np.concatenate(naff),
            "start_over": np.concatenate(so), "states": states, "off": off, "chi2": np.array(chi2)}


# ---------------------------------------------------------------------------------------------
# caller-side protocols
# ---------------------------------------------------------------------------------------------
def edge_cases(impl: str) -> dict:
    """Full information matrices, reversed and duplicate edges, priors on two poses, a non-default Tikhonov
    term; three batch calls, then incremental appends.  The inputs are drawn from a fixed seed in the same
    order on every call, so both libraries see the same numbers."""
    rng = np.random.default_rng(5)
    n0, n1 = 30, 38
    truth = np.cumsum(np.c_[np.ones(n1), 0.3 * rng.standard_normal(n1), 0.2 * rng.standard_normal(n1)], axis=0)

    def rel(a, b):
        c, s = np.cos(truth[a, 2]), np.sin(truth[a, 2])
        d = truth[b] - truth[a]
        return np.array([c * d[0] + s * d[1], -s * d[0] + c * d[1], d[2]]) + 0.01 * rng.standard_normal(3)

    def full_W():
        M = rng.standard_normal((3, 3))
        # symmetric: with a non-symmetric W the reference's "upper triangle of each block" rule
        # (aprilsam.c:171-172) assembles an indefinite matrix more often than not and cs_chol's NULL is
        # dereferenced (tools/edge_diag.py) -- there is no oracle to compare with; this library aborts
        # with "not positive definite" in that case
        return 30.0 * (M @ M.T + 0.5 * np.eye(3))

    edges = [(i, i + 1) for i in range(n1 - 1)]
    extra = [(3, 11), (11, 3), (3, 11), (20, 7), (25, 2), (14, 13), (29, 0), (28, 9)]  # duplicates and reversed pairs
    recs = {e: (rel(*e), full_W()) for e in sorted(set(edges + extra))}
    init = truth + 0.05 * rng.standard_normal(truth.shape)
    W_prior2 = full_W()

    rows, chi2, naff = [], [], []
    with H.Harness(impl, nthreshold=10**9) as h:
        h.set_tikhanov(3e-3)
        for k in range(n0):
            h.add_node(init[k])
        h.add_xytpos(0, truth[0], np.diag([1e4, 1e4, 1e3]))
        h.add_xytpos(17, truth[17] + 0.01, W_prior2)
        for (a, b) in edges + extra:
            if max(a, b) < n0:
                h.add_xyt(a, b, *recs[(a, b)])
        for it in range(3):
            h.batch()
            rows.append(h.states())
            chi2.append(h.chi2())
            naff.append(0)
        for k in range(n0, n1):
            h.add_node(init[k])
            for (a, b) in edges + [(k, k - 9), (k - 4, k)]:
                if max(a, b) == k:
                    z, W = recs.get((a, b), (None, None))
                    if z is None:
                        z, W = rel(a, b), full_W()
                        recs[(a, b)] = (z, W)
                    h.add_xyt(a, b, z, W)
            h.inc()
            rows.append(h.states())
            chi2.append(h.chi2())
            naff.append(h.info()["naffected"])
    states, off = _stack(rows)
    return {"states": states, "off": off, "chi2": np.array(chi2), "naffected": np.array(naff)}


def multi_pose_append(impl: str, m3500) -> dict:
    """Several M3500 poses appended between two incremental calls."""
    db, estart = m3500.bucketed()
    rows, chi2, naff = [], [], []
    n = 0
    with H.Harness(impl) as h:
        for upto in (1, 4, 9, 10, 30, 33, 80, 150):
            for k in range(n, upto):
                h.add_node(m3500.init[k])
                if k == 0:
                    h.add_xytpos(0, [0, 0, 0], [1e4, 0, 0, 0, 1e4, 0, 0, 0, 1e3])
                for e in range(estart[k], estart[k + 1]):
                    h.add_xyt(int(db.ea[e]), int(db.eb[e]), db.ez[e], db.eW[e])
            if n == 0:
                h.batch()
            else:
                h.inc()
            n = upto
            rows.append(h.states())
            chi2.append(h.chi2())
            naff.append(h.info()["naffected"])
    states, off = _stack(rows)
    return {"states": states, "off": off, "chi2": np.array(chi2), "naffected": np.array(naff)}


def factor_values_edited(impl: str, m3500, n: int = 600) -> dict:
    """Batch solve, then z / W of 40 seeded factors edited in place, states reset, batch solve again."""
    sub = m3500.head(n)
    rng = np.random.default_rng(3)
    with H.Harness(impl) as h:
        h.load_full(sub)
        h.batch()
        before = h.states()
        idx = rng.choice(h.n_factors - 1, size=40, replace=False) + 1  # factor 0 is the prior
        z2s, W2s = [], []
        for i in idx:
            _, _, _, z, W = h.factor(int(i))
            z2s.append(z + rng.normal(0, 0.05, 3))
            W2s.append(W * rng.uniform(0.2, 3.0))
        for i, z2, W2 in zip(idx, z2s, W2s):
            h.set_factor(int(i), z2, W2)
        h.set_states(sub.init)
        h.batch()
        return {"before": before, "edit_idx": idx, "edit_z": np.array(z2s), "edit_W": np.array(W2s),
                "states": h.states(), "chi2": np.array(h.chi2())}


REPLACED_W = np.diag([30.0, 30.0, 50.0]).reshape(9)


def factor_replaced(impl: str, m3500, n: int = 400) -> dict:
    """Batch solve, then the last factor replaced by one between other poses (same N and F), batch again."""
    sub = m3500.head(n)
    with H.Harness(impl) as h:
        h.load_full(sub)
        h.batch()
        h.replace_xyt(h.n_factors - 1, 17, 311, [0.3, -0.2, 0.1], REPLACED_W)
        h.set_states(sub.init)
        h.batch()
        return {"states": h.states(), "order": h.ordering(), "chi2": np.array(h.chi2())}


def inc_solver(impl: str, m3500) -> dict:
    """april_graph_cholesky_inc_solver after 150 replay steps, then 50 more steps."""
    with H.Harness(impl) as h:
        h.replay_begin(m3500)
        h.replay_to(150)
        h.inc_solver()
        s150, info = h.states(), h.info()
        h.replay_to(200)
        return {"states_150": s150, "start_over": np.array(info["start_over"]),
                "nlinearized": np.array(info["nlinearized"]), "states_200": h.states()}


# ---------------------------------------------------------------------------------------------
# ".graph" files
# ---------------------------------------------------------------------------------------------
def build_small(h, m3500, n: int = 40):
    """The first n M3500 poses with graph, node and factor attributes (what the file tests save)."""
    sub = m3500.head(n)
    h.load_full(sub)
    h.attr_put(h.GRAPH, 0, "name", "M3500 head")
    h.attr_put(h.GRAPH, 0, "poses", n)
    h.attr_put(h.NODE, 3, "tag", "third")
    for f in range(1, h.n_factors):
        t, a, b, _, _ = h.factor(f)
        h.attr_put(h.FACTOR, f, "type", "odom" if abs(a - b) == 1 else "scan")
    return sub
