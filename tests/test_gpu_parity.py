"""GPU parity tests: the drop-in library (CUDA path) against the reference, through the public
C API (harness/harness.c).  What the reference computes is stored under tests/golden/
(tools/make_golden.py runs tests/support/refcases.py on it); the tests run the same protocols
on this library and compare.

Tolerance: 1e-6 relative on node states and chi2 (BASELINE.json north_star); observed
differences are ~1e-9 (different elimination arithmetic order, GPU sin/cos).
"""
import numpy as np
import pytest

from aprilsam_b200 import harness as H
from conftest import golden
from support import refcases

pytestmark = pytest.mark.gpu

RTOL = 1e-6


def rel_state_err(a, b):
    """max |a-b| / max(1, |b|) with theta compared modulo 2 pi."""
    d = a - b
    d[:, 2] = (d[:, 2] + np.pi) % (2 * np.pi) - np.pi
    return float(np.max(np.abs(d) / np.maximum(1.0, np.abs(b))))


def assert_matches_reference(got, want, what):
    """Every array a refcases function returned against the stored reference result: integers (counters,
    orderings, sample ids) exactly, chi2 and node states to RTOL."""
    assert set(want) <= set(got), (what, sorted(set(want) - set(got)))
    for k, w in want.items():
        g = np.asarray(got[k])
        assert g.shape == w.shape, (what, k, g.shape, w.shape)
        if "states" in k:
            err = rel_state_err(g.reshape(-1, 3), w.reshape(-1, 3))
            assert err < RTOL, (what, k, err)
        elif "chi2" in k:
            bad = np.flatnonzero(np.abs(g - w) > RTOL * np.maximum(1.0, np.abs(w)))
            assert bad.size == 0, (what, k, "first differing entry", int(bad[0]), g.flat[bad[0]], w.flat[bad[0]])
        else:
            bad = np.flatnonzero(g.reshape(-1) != w.reshape(-1))
            assert bad.size == 0, (what, k, "first differing entry", int(bad[0]))


def test_chi2_kernel(m3500):
    g = golden("m3500_batch.npz")
    with H.Harness("b200") as h:
        h.load_full(m3500)
        c0 = h.chi2()
    assert abs(c0 - g["chi2"][0]) <= RTOL * g["chi2"][0]


def test_m3500_batch_six_iterations(m3500):
    g = golden("m3500_batch.npz")
    with H.Harness("b200") as h:
        h.load_full(m3500)
        for it in range(6):
            h.batch()
            assert np.array_equal(h.ordering(), g["ordering"]) or it > 0
            c = h.chi2()
            assert abs(c - g["chi2"][it + 1]) <= RTOL * g["chi2"][it + 1], (it, c, g["chi2"][it + 1])
            err = rel_state_err(h.states(), g["states"][it])
            assert err < RTOL, (it, err)
        assert np.array_equal(h.tree_parents(), g["tree_parents"])


def test_small_graphs_batch(m3500):
    """Ragged / tiny inputs: 1, 2, 3, 7, 50 poses, three batch calls each."""
    for n in (1, 2, 3, 7, 50):
        assert_matches_reference(refcases.batch_iters("b200", m3500.head(n), 3), refcases.load(f"small{n}"), n)


def test_tutorial_graph():
    g = golden("tutorial.npz")
    d = H.PoseGraphData(g["init"], g["ea"], g["eb"], g["ez"], g["eW"])
    for mode, batch_only in (("inc", False), ("batch", True)):
        with H.Harness("b200") as h:
            h.replay_begin(d)
            chi2, _, _ = h.replay_to(6, batch_only=batch_only)
            assert rel_state_err(h.states(), g[f"{mode}_states"]) < RTOL
            assert abs(chi2[-1] - g[f"{mode}_chi2"][-1]) <= RTOL * max(1.0, g[f"{mode}_chi2"][-1])


@pytest.mark.parametrize("nsteps", [400])
def test_m3500_replay_lockstep(m3500, nsteps):
    """Every step: chi2, naffected and start_over must match; node states (the newest pose and a seeded
    sample of the others) after every step."""
    got = refcases.replay_lockstep("b200", m3500, range(1, nsteps + 1), 2)
    assert_matches_reference(got, refcases.load(f"m3500_replay{nsteps}"), "m3500 replay")


def test_m3500_replay_full_golden(m3500):
    """Whole 3500-step replay against the committed per-step chi2 / counters and checkpoints."""
    g = golden("m3500_replay.npz")
    with H.Harness("b200") as h:
        h.replay_begin(m3500)
        done = 0
        for cp in g["checkpoints"]:
            chi2, _, info = h.replay_to(int(cp))
            n = len(chi2)
            assert np.array_equal(info[:, 0], g["naffected"][done:done + n]), f"naffected differs before step {cp}"
            assert np.array_equal(info[:, 1], g["start_over"][done:done + n]), f"start_over differs before step {cp}"
            ref = g["chi2"][done:done + n]
            assert np.all(np.abs(chi2 - ref) <= RTOL * np.maximum(1.0, ref)), f"chi2 differs before step {cp}"
            err = rel_state_err(h.states(), g[f"states_{int(cp)}"])
            assert err < RTOL, (int(cp), err)
            done += n
        assert abs(chi2[-1] - 68.965607796) < 1e-6


# ---------------------------------------------------------------------------------------------
# synthetic graphs: big fronts (multi-CTA team path), full sizes, incremental on sparse graphs
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [2000, 30000])
def test_manhattan_batch_vs_reference(n):
    """Dense synthetic Manhattan world: fronts up to m ~ 700 exercise the team path of k_factor."""
    from aprilsam_b200 import datasets
    d = datasets.manhattan_dense(n, seed=1)
    assert_matches_reference(refcases.batch_iters("b200", d, 2), refcases.load(f"manhattan{n}"), n)


def test_manhattan_100k_batch_vs_reference():
    """BASELINE.json configs[3] at full size: 100 000 poses / ~400 k factors, three Gauss-Newton iterations,
    each relinearised at the previous result; the ordering of the first is compared as a digest."""
    from aprilsam_b200 import datasets
    d = datasets.manhattan_dense(100000, seed=1)
    got = refcases.batch_iters("b200", d, 3)
    assert got["chi2"][0] < got["chi2_0"]
    assert_matches_reference(got, refcases.load("manhattan100000"), "100k")


def test_manhattan_100k_properties_without_reference():
    """Size-independent properties at full size (no oracle needed): the Gauss-Newton step lowers
    chi2, a second call from the same states reproduces the first up to the summation order of the
    assembly atomics (factor / solve kernels are deterministic), and further steps stay finite."""
    from aprilsam_b200 import datasets
    d = datasets.manhattan_dense(100000, seed=1)
    with H.Harness("b200") as a:
        a.load_full(d)
        c0 = a.chi2()
        a.batch()
        s1, c1 = a.states(), a.chi2()
        assert np.isfinite(s1).all() and c1 < c0
        a.set_states(d.init)
        a.batch()
        assert rel_state_err(a.states(), s1) < 1e-9, "same input must give the same output"
        for _ in range(3):
            a.batch()
        assert np.isfinite(a.states()).all() and a.chi2() < c0


def test_sparse_replay_lockstep():
    """Config-5 style graph (odometry + 5 % closures), pose-by-pose: chi2 / naffected / start_over of every
    step, sampled node states every 50 poses."""
    from aprilsam_b200 import datasets
    d = datasets.manhattan_sparse(2500, seed=1)
    got = refcases.replay_lockstep("b200", d, range(50, d.n_nodes + 1, 50), 8)
    assert_matches_reference(got, refcases.load("sparse_replay2500"), "sparse replay")


def test_sparse_bulk_then_incremental_lockstep():
    """Incremental steps on a LARGE sparse graph (fronts of the multi-CTA team path are re-factored
    by incremental steps): the first 29 700 poses are loaded at once at the generator's ground truth and
    batch-solved twice, then 200 poses are appended one by one (sampled states every 25 poses)."""
    assert_matches_reference(refcases.sparse_bulk_then_incremental("b200"), refcases.load("sparse_bulk_inc"), "bulk + inc")


def test_edge_cases_full_W_duplicates_reversed_edges_several_priors():
    """What the M3500 file never exercises: full information matrices (off-diagonal terms), edges given as (higher id, lower id), several factors on the same pose pair, priors on more than one
    pose, a non-default Tikhonov term; then incremental appends on top."""
    assert_matches_reference(refcases.edge_cases("b200"), refcases.load("edge_cases"), "edge cases")


def test_empty_and_trivial_graphs():
    """april_graph_cholesky on a graph without factors returns silently (aprilsam.c:90-91); a single
    anchored pose solves to its prior."""
    with H.Harness("b200") as h:
        h.batch()
        h.add_node([1.0, 2.0, 0.3])
        h.batch()
        assert np.allclose(h.states(), [[1.0, 2.0, 0.3]])
        h.add_xytpos(0, [0.5, -0.5, 0.1], np.diag([1e4, 1e4, 1e3]))
        h.batch()
        assert np.allclose(h.states(), [[0.5, -0.5, 0.1]], atol=1e-6)
        assert h.chi2() < 1e-6


def test_multi_pose_append_per_call(m3500):
    """Several poses appended between two incremental calls (aprilsam.c:887-904 path)."""
    assert_matches_reference(refcases.multi_pose_append("b200", m3500), refcases.load("multi_pose_append"), "multi-pose append")


def test_factor_between_old_poses_is_exact(m3500):
    """A factor between two already-solved poses takes the general path (full symbolic rebuild,
    no relinearisation).  The reference corrupts its tree here, so the check is against the exact
    solution of the linear system (numpy emulation of the assembled Hessian)."""
    import scipy.sparse.linalg as spl
    from support import emul
    from support.hostplan import HostPlan
    n = 120
    sub = m3500.head(n)
    with H.Harness("b200", nthreshold=10**9) as h:  # no batch escalation: the step stays linear
        h.load_full(sub)
        h.batch()
        lp = h.l_points()
        sa, sb = h.states()[17], h.states()[95]
        ca, sn_ = np.cos(sa[2]), np.sin(sa[2])
        dx, dy = sb[0] - sa[0], sb[1] - sa[1]
        z = np.array([ca * dx + sn_ * dy + 0.05, -sn_ * dx + ca * dy - 0.03, sb[2] - sa[2] + 0.02])
        W = np.diag([50.0, 50.0, 80.0])
        h.add_xyt(17, 95, z, W)
        h.inc()
        st = h.states()
        assert np.array_equal(h.l_points(), lp), "no relinearisation on this path"
    ftype = np.r_[2, np.ones(sub.n_edges + 1, dtype=np.int32)].astype(np.int32)
    fa = np.r_[0, sub.ea, 17].astype(np.int32)
    fb = np.r_[-1, sub.eb, 95].astype(np.int32)
    fz = np.vstack([[0, 0, 0], sub.ez, z])
    fW = np.vstack([[1e4, 0, 0, 0, 1e4, 0, 0, 0, 1e3], sub.eW, W.reshape(1, 9)])
    p = HostPlan().build(n, ftype, fa, fb)
    Hs = emul.Hessian(n, p.info()["n_slots"])
    Hs.reset(n, 1e-4)
    Hs.linearize(range(len(ftype)), ftype, fa, fb, fz, fW, lp, lp, p.array("node2q"), p.array("fslot"))
    fslot = p.array("fslot")
    pairs = {}
    for f in range(len(ftype)):
        if ftype[f] == 1:
            pairs[fslot[f]] = (min(fa[f], fb[f]), max(fa[f], fb[f]))
    A = Hs.dense([pairs[s] for s in range(p.info()["n_slots"])])
    x = spl.spsolve(A.tocsc(), Hs.B.reshape(-1)).reshape(n, 3)
    want = lp + x
    want[:, 2] = emul.mod2pi(want[:, 2])
    assert rel_state_err(st, want) < RTOL


def test_replay_cli_text_and_graph_files(m3500, tmp_path):
    """examples/asam_replay (SURVEY.md section 8f item 1): a Manhattan text file and the ".graph" file the CLI
    saves from it replay to the same final chi2 as the harness-driven replay of the same poses."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "examples", "_build", "asam_replay")
    assert os.path.exists(cli), "run __graft_entry__.build()"
    sub = m3500.head(150)
    txt, gfile = str(tmp_path / "m150.txt"), str(tmp_path / "m150.graph")
    with open(txt, "w") as f:
        for i, p in enumerate(sub.init):
            f.write("VERTEX2 %d %r %r %r\n" % (i, float(p[0]), float(p[1]), float(p[2])))
        for a, b, z, W in zip(sub.ea, sub.eb, sub.ez, sub.eW):
            f.write("EDGE2 %d %d " % (a, b) + " ".join(repr(float(v)) for v in (*z, W[0], W[1], W[4], W[8], W[2], W[5])) + "\n")
    with H.Harness("b200") as h:
        h.replay_begin(sub)
        chi2, _, _ = h.replay_to(sub.n_nodes)
    want = chi2[-1]
    for args in (["--datapath", txt, "--save", gfile, "--quiet"], ["--datapath", gfile, "--quiet"]):
        out = subprocess.run([cli] + args, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr
        got = float(re.search(r"final chi2 ([0-9.eE+-]+)", out.stdout).group(1))
        assert abs(got - want) <= RTOL * max(1.0, want), (args, got, want)


def test_reference_example_programs_unchanged_on_this_library(m3500, tmp_path):
    """The reference's own aprilsam_tutorial.c / aprilsam_demo.c, compiled WITHOUT a source change against
    include/ + libaprilsam_b200 (oracle/Makefile, binaries only): the tutorial prints what it prints
    with the reference library (tests/golden/tutorial_stdout_*.txt, generated with oracle/_ref), the demo
    replays a Manhattan text file to the chi2 of the harness-driven replay."""
    import os
    import re
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tut = os.path.join(root, "oracle", "_ref", "ref_aprilsam_tutorial")
    demo = os.path.join(root, "oracle", "_ref", "ref_aprilsam_demo")
    if not (os.path.exists(tut) and os.path.exists(demo)):
        pytest.skip("the reference's example programs were not built (no reference sources at build time)")

    def norm(text):
        return [l.rstrip().replace("-0.00", "0.00") for l in text.splitlines()
                if l.strip() and "running time" not in l and "APRILSAM" not in l and set(l.strip()) - set("=|")]

    for args, gold in (([], "tutorial_stdout_inc.txt"), (["--batch_update_only"], "tutorial_stdout_batch.txt")):
        out = subprocess.run([tut] + args, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-1000:]
        want = norm(open(os.path.join(root, "tests", "golden", gold)).read())
        got = norm(out.stdout)
        assert got == want, "\n".join(f"{a!r} | {b!r}" for a, b in zip(got, want) if a != b)[:2000]

    sub = m3500.head(200)
    txt = str(tmp_path / "m200.txt")
    with open(txt, "w") as f:
        for i, p in enumerate(sub.init):
            f.write("VERTEX2 %d %r %r %r\n" % (i, float(p[0]), float(p[1]), float(p[2])))
        for a, b, z, W in zip(sub.ea, sub.eb, sub.ez, sub.eW):
            f.write("EDGE2 %d %d " % (a, b) + " ".join(repr(float(v)) for v in (*z, W[0], W[1], W[4], W[8], W[2], W[5])) + "\n")
    with H.Harness("b200") as h:
        h.replay_begin(sub)
        chi2, _, _ = h.replay_to(sub.n_nodes)
    out = subprocess.run([demo, "--datapath", txt], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-1000:]
    vals = [float(v) for v in re.findall(r"[Cc]hi[^0-9-]*([0-9.eE+-]+)", out.stdout)]
    assert vals, out.stdout[-500:]
    assert abs(vals[-1] - chi2[-1]) <= 1e-5 * max(1.0, chi2[-1]), (vals[-1], chi2[-1])


# ---------------------------------------------------------------------------------------------
# round 2: caller-side edits, policy hook, show_timing, several GPUs
# ---------------------------------------------------------------------------------------------
def test_factor_values_edited_in_place_between_batch_calls(m3500):
    """The reference reads every factor on every batch call (aprilsam.c:154-195): re-weighting W or moving z
    between two calls must show in the next solve although ordering + symbolic plan are cached."""
    sub = m3500.head(600)
    got = refcases.factor_values_edited("b200", m3500, 600)
    edits = list(zip(got["edit_idx"], got["edit_z"], got["edit_W"]))
    # same graph built from scratch with the edited values
    with H.Harness("b200") as fresh:
        fresh.load_full(sub)
        for i, z2, W2 in edits:
            fresh.set_factor(int(i), z2, W2)
        fresh.batch()
        assert rel_state_err(got["states"], fresh.states()) < 1e-9
        want = fresh.states()
    with H.Harness("b200") as stale:  # what ignoring the edit would have produced
        stale.load_full(sub)
        stale.batch()
        assert rel_state_err(stale.states(), want) > 1e-4, "the edit must matter for this test to mean anything"
    assert rel_state_err(got["before"], want) > 1e-4
    assert_matches_reference(got, refcases.load("factor_values_edited"), "edited factors")


def test_factor_replaced_with_same_count_rebuilds_the_plan(m3500):
    """zarray_set of another factor keeps N and F but changes the structure: the cached plan must not be reused."""
    sub = m3500.head(400)
    got = refcases.factor_replaced("b200", m3500, 400)
    with H.Harness("b200") as fresh:
        fresh.load_full(sub)
        fresh.replace_xyt(fresh.n_factors - 1, 17, 311, [0.3, -0.2, 0.1], refcases.REPLACED_W)
        fresh.batch()
        assert rel_state_err(got["states"], fresh.states()) < 1e-9
        assert np.array_equal(got["order"], fresh.ordering())
    assert_matches_reference(got, refcases.load("factor_replaced"), "replaced factor")


def test_invalidate_plan_gives_the_same_solution(m3500):
    with H.Harness("b200") as a:
        a.load_full(m3500)
        a.batch()
        s1 = a.states()
        a.set_states(m3500.init)
        a.invalidate_plan()
        a.batch()
        assert rel_state_err(a.states(), s1) < 1e-9


def test_inc_solver_entry_point_matches_reference(m3500):
    """april_graph_cholesky_inc_solver (aprilsam.h:276) re-runs the back-substitution + bookkeeping of the last
    step; the reference ignores idxs (aprilsam.c:578-597)."""
    assert_matches_reference(refcases.inc_solver("b200", m3500), refcases.load("inc_solver"), "inc_solver")


def test_escalation_policy_hook_is_deterministic(m3500):
    """aprilsam_b200_set_escalation_policy: a policy that always fires turns every incremental step into
    "incremental update, then batch solve" (fresh tree after every step), identically on every run; a policy that
    never fires changes nothing against the default; the built-in 1/3 work-ratio rule escalates on some steps only."""
    n = 120
    with H.Harness("b200") as pol, H.Harness("b200") as pol2, H.Harness("b200") as dflt, H.Harness("b200") as big:
        pol.set_policy_ratio(1e-12)
        pol2.set_policy_ratio(1e-12)
        big.set_policy_ratio(1e12)
        for h in (pol, pol2, dflt, big):
            h.replay_begin(m3500)
        cp, _, ip = pol.replay_to(n)
        cp2, _, ip2 = pol2.replay_to(n)
        _, _, idf = dflt.replay_to(n)
        _, _, ib = big.replay_to(n)
        assert (ip[1:, 0] == 0).all(), "every incremental step ended in a batch solve (fresh tree, naffected 0)"
        assert (idf[1:, 0] > 0).all(), "no escalation in the first 120 default steps"
        assert np.array_equal(ip, ip2) and rel_state_err(pol.states(), pol2.states()) < 1e-12
        assert np.allclose(cp, cp2, rtol=1e-12, atol=0)
        assert np.array_equal(idf, ib) and rel_state_err(dflt.states(), big.states()) == 0.0
        # an escalated replay is the better-converged estimate of the same problem (the default one leaves the
        # poses that back-substitution pruned stale until the next batch)
        assert pol.chi2() <= dflt.chi2() * (1 + 1e-9)
    with H.Harness("b200") as third, H.Harness("b200") as dflt:
        third.set_policy_ratio(1.0 / 3.0)
        for h in (third, dflt):
            h.replay_begin(m3500)
        c, _, it = third.replay_to(400)
        _, _, idf = dflt.replay_to(400)
        assert np.isfinite(c).all()
        n_pol, n_dflt = int((it[1:, 0] == 0).sum()), int((idf[1:, 0] == 0).sum())
        assert n_dflt <= n_pol < 399, (n_pol, n_dflt)


def test_show_timing_prints_the_reference_table_format(m3500, tmp_path, capfd):
    """param->show_timing (aprilsam.c:317-318, :553-555): rows "%2d %32s %15f ms %15f ms" like
    aprilsam/common/timeprofile.h:89-106, first row 'begin' at 0 ms, cumulative column non-decreasing."""
    import re
    with H.Harness("b200") as a:
        a.set_show_timing(True)
        a.replay_begin(m3500)
        a.replay_to(3)
    out = capfd.readouterr().out
    rows = [l for l in out.splitlines() if re.match(r"^\s*\d+ .{32} +[0-9.]+ ms +[0-9.]+ ms$", l)]
    assert len(rows) >= 6, out
    assert rows[0].split()[1] == "begin" and float(rows[0].split()[-4]) == 0.0
    tables, cur = [], []
    for l in rows:
        if l.split()[0] == "0" and cur:
            tables.append(cur)
            cur = []
        cur.append(l)
    tables.append(cur)
    assert len(tables) == 3  # one batch call + two incremental steps
    for t in tables:
        cum = [float(l.split()[-2]) for l in t]
        assert all(b >= a_ for a_, b in zip(cum, cum[1:]))
        assert [int(l.split()[0]) for l in t] == list(range(len(t)))
    assert "device: k_factor" in out and "device: k_linearize" in out


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize("poses", [30000])
def test_sharded_two_gpu_solve_matches_single_gpu(poses):
    """SURVEY.md section 8e on hardware: two processes, one GPU each, elimination-tree shards + NCCL exchange;
    the sharded batch solve must reproduce the single-GPU solve (tools/shard_check.py exits non-zero above 1e-6)."""
    import os
    import subprocess
    import sys
    from aprilsam_b200 import capi
    if capi.lib().asam_device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(root, "tools", "shard_check.py"), "--poses", str(poses), "--iters", "3"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert "RESULT world 2" in r.stdout
