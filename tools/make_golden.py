#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref, deterministic clock).

Needs oracle/_ref built from the reference sources (oracle/Makefile).  The fixtures let the
parity tests run where the reference binary is absent.
  m3500_batch.npz          config 1/2: 6 consecutive april_graph_cholesky calls on the full graph
  m3500_replay.npz         config 3: demo-protocol pose-by-pose replay, chi2 / naffected / start_over
                           after every step, full state vectors at checkpoints
  tutorial.npz             the 6-pose dog-leg of examples/aprilsam_tutorial.c (incremental + batch)
  reference_cases.npz      what every other parity test compares with (tests/support/refcases.py)
  m3500_head40.graph       a ".graph" file written by the reference (attributes included)

    python tools/make_golden.py [m3500_batch m3500_replay tutorial reference_cases]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from aprilsam_b200 import datasets  # noqa: E402
from aprilsam_b200.harness import Harness, PoseGraphData  # noqa: E402
from support import refcases as R  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")


def m3500_batch(d):
    h = Harness("reference")
    h.load_full(d)
    chi2 = [h.chi2()]
    states = []
    for _ in range(6):
        h.batch()
        chi2.append(h.chi2())
        states.append(h.states())
    order = h.ordering()
    parents = h.tree_parents()
    h.close()
    np.savez_compressed(os.path.join(G, "m3500_batch.npz"), chi2=np.array(chi2), states=np.array(states),
                        ordering=order, tree_parents=parents)
    print("m3500_batch chi2", chi2)


def m3500_replay(d):
    h = Harness("reference")
    h.replay_begin(d)
    checkpoints = [1, 2, 10, 100, 500, 1000, 2000, 3000, 3500]
    chi2, info, states = [], [], {}
    for cp in checkpoints:
        c, _, i = h.replay_to(cp)
        chi2.append(c)
        info.append(i)
        states[f"states_{cp}"] = h.states()
    chi2 = np.concatenate(chi2)
    info = np.concatenate(info)
    h.close()
    np.savez_compressed(os.path.join(G, "m3500_replay.npz"), chi2=chi2, naffected=info[:, 0].astype(np.int32),
                        start_over=info[:, 1].astype(np.int32), checkpoints=np.array(checkpoints), **states)
    print("m3500_replay final chi2", chi2[-1], "batch escalations", int((np.diff(info[:, 1]) < 0).sum()))


def tutorial():
    # examples/aprilsam_tutorial.c: 6 poses, unit odometry with small lateral noise, one closure
    init = np.array([[0, 0, 0], [1.0, 0.1, 0.0], [2.1, 0.3, 0.02], [3.0, 0.55, 0.03], [4.1, 0.6, 0.0], [5.0, 0.9, 0.05]])
    W = np.diag([100.0, 100.0, 1000.0]).reshape(-1)
    ea = np.array([0, 1, 2, 3, 4, 0], dtype=np.int32)
    eb = np.array([1, 2, 3, 4, 5, 5], dtype=np.int32)
    ez = np.array([[1, 0.15, 0.01], [1, 0.17, 0.0], [1, 0.2, 0.0], [1.02, 0.15, 0.0], [1, 0.2, -0.01], [5.0, 0.85, 0.012]])
    d = PoseGraphData(init, ea, eb, ez, np.tile(W, (6, 1)))
    out = {}
    for mode, batch_only in (("inc", False), ("batch", True)):
        h = Harness("reference")
        h.replay_begin(d)
        chi2, _, info = h.replay_to(6, batch_only=batch_only)
        out[f"{mode}_chi2"] = chi2
        out[f"{mode}_states"] = h.states()
        h.close()
    np.savez_compressed(os.path.join(G, "tutorial.npz"), init=init, ea=ea, eb=eb, ez=ez, eW=np.tile(W, (6, 1)), **out)
    print("tutorial", out["inc_chi2"], out["batch_chi2"])


def reference_cases(d):
    out = {}

    def put(prefix, res, keys=None):
        for k, v in res.items():
            if keys is None or k in keys:
                out[f"{prefix}/{k}"] = v

    # CPU tests: orderings / elimination trees of M3500 sub-graphs, single batch steps
    for n in (1, 2, 3, 4, 7, 11, 13, 64, 150, 257, 900):
        keys = (("order", "parents") if n in (1, 2, 3, 4, 7, 13, 64, 257, 900) else ()) + \
               (("states", "chi2") if n in (1, 2, 3, 11, 150) else ())
        put(f"head{n}", R.batch_once("reference", d.head(n)), keys)
    put("synth1500", R.batch_once("reference", datasets.manhattan_dense(1500, seed=3)), ("order",))
    put("synth600", R.batch_once("reference", datasets.manhattan_dense(600, seed=2)), ("states",))
    # GPU tests
    for n in (1, 2, 3, 7, 50):
        put(f"small{n}", R.batch_iters("reference", d.head(n), 3))
    for n, iters in ((2000, 2), (30000, 2), (100000, 3)):
        put(f"manhattan{n}", R.batch_iters("reference", datasets.manhattan_dense(n, seed=1), iters))
    put("m3500_replay400", R.replay_lockstep("reference", d, range(1, 401), 2))
    put("sparse_replay2500", R.replay_lockstep("reference", datasets.manhattan_sparse(2500, seed=1), range(50, 2501, 50), 8))
    put("sparse_bulk_inc", R.sparse_bulk_then_incremental("reference"))
    put("edge_cases", R.edge_cases("reference"))
    put("multi_pose_append", R.multi_pose_append("reference", d))
    put("factor_values_edited", R.factor_values_edited("reference", d), ("states", "chi2"))
    put("factor_replaced", R.factor_replaced("reference", d))
    put("inc_solver", R.inc_solver("reference", d))
    np.savez_compressed(R.GOLDEN, **out)
    with Harness("reference") as h:
        R.build_small(h, d)
        h.save(os.path.join(G, "m3500_head40.graph"))
    print("reference_cases", len(out), "arrays", os.path.getsize(R.GOLDEN), "bytes")


if __name__ == "__main__":
    d = PoseGraphData.load(os.path.join(G, "m3500.npz"))
    which = sys.argv[1:] or ["m3500_batch", "m3500_replay", "tutorial", "reference_cases"]
    for name in which:
        fn = globals()[name]
        fn() if name == "tutorial" else fn(d)
