"""CPU-only tests (-m "not gpu"): ABI surface, host symbolic layer, oracle vs golden vectors.

The numeric checks replay the plan that would be uploaded to HBM with tests/support/emul.py (a
numpy emulation of the kernels' index arithmetic) -- that validates ordering, elimination tree,
supernode row lists, relative indices, gather lists and task order without a device.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse.linalg as spl

from aprilsam_b200 import datasets
from aprilsam_b200 import harness as H
from conftest import ROOT, golden
from support import emul
from support import refcases
from support.hostplan import HostPlan


def factor_arrays(d, n_edges=None):
    E = d.n_edges if n_edges is None else n_edges
    ftype = np.r_[2, np.ones(E, dtype=np.int32)].astype(np.int32)
    fa = np.r_[0, d.ea[:E]].astype(np.int32)
    fb = np.r_[-1, d.eb[:E]].astype(np.int32)
    fz = np.vstack([[0, 0, 0], d.ez[:E]])
    fW = np.vstack([[1e4, 0, 0, 0, 1e4, 0, 0, 0, 1e3], d.eW[:E]])
    return ftype, fa, fb, fz, fW


# ---------------------------------------------------------------------------------------------
# ABI
# ---------------------------------------------------------------------------------------------
def declared_functions(header):
    src = open(header).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"^\s*#.*$", "", src, flags=re.M)
    src = re.sub(r"static inline[^{;]*\{", "{", src)
    names = set()
    skip = {"defined", "_Static_assert", "sizeof", "offsetof", "void", "int", "double", "char", "float"}
    for m in re.finditer(r"\b([A-Za-z_][A-Za-z0-9_]*)\s*\([^;{}]*\)\s*;", src):
        n = m.group(1)
        if n not in skip and not n.startswith("__"):
            names.add(n)
    return names


def test_library_exports_every_declared_symbol(built):
    lib = C.CDLL(built)
    missing = []
    for hdr in ("include/asam_cuda.h", "include/aprilsam/aprilsam.h", "include/aprilsam/common/matd.h"):
        for name in sorted(declared_functions(os.path.join(ROOT, hdr))):
            if "(*" in name:
                continue
            try:
                getattr(lib, name)
            except AttributeError:
                missing.append(f"{hdr}:{name}")
    assert not missing, missing


def test_struct_abi_matches_reference_layout(built, tmp_path):
    """Offsets from SURVEY.md section 8b (measured against the reference headers)."""
    src = tmp_path / "abi.c"
    src.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "aprilsam.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(zarray_t), sizeof(april_graph_t), sizeof(april_graph_node_t),
         sizeof(april_graph_factor_t), sizeof(search_tree_node_t), sizeof(search_tree_t), sizeof(april_graph_cholesky_param_t));
  printf("%zu %zu %zu %zu %zu %zu %zu\n", offsetof(april_graph_node_t, state), offsetof(april_graph_node_t, l_point),
         offsetof(april_graph_node_t, delta_X), offsetof(april_graph_factor_t, u.common.z), offsetof(april_graph_factor_t, u.common.W),
         offsetof(april_graph_cholesky_param_t, tr), offsetof(april_graph_cholesky_param_t, delta_theta));
  return 0; }''')
    exe = tmp_path / "abi"
    subprocess.check_call(["gcc", "-std=gnu99", "-I" + os.path.join(ROOT, "include", "aprilsam"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    assert [int(x) for x in out] == [24, 32, 112, 104, 40, 80, 128, 16, 40, 48, 64, 80, 72, 120]


def test_solver_fails_loudly_without_gpu(built):
    """No CPU fallback: on a box without a CUDA device the solver entry points abort."""
    from aprilsam_b200 import capi
    if capi.lib().asam_device_count() > 0:
        pytest.skip("a CUDA device is present")
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from aprilsam_b200 import harness as H\n"
            "h = H.Harness('b200'); h.add_node([0,0,0]); h.add_xytpos(0,[0,0,0],[1,0,0,0,1,0,0,0,1]); h.batch()\n"
            "print('SOLVED')\n") % ROOT
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert p.returncode != 0 and "SOLVED" not in p.stdout
    assert "no usable CUDA device" in p.stderr


# ---------------------------------------------------------------------------------------------
# ordering + elimination tree == reference
# ---------------------------------------------------------------------------------------------
def node_parents(plan, n):
    order, ppos = plan.array("order"), plan.array("parent_pos")
    par = np.full(n, -1, dtype=np.int32)
    for ui in range(n):
        if ppos[ui] >= 0:
            par[order[ui]] = order[ppos[ui]]
    return par


def test_m3500_ordering_and_tree_match_golden(m3500):
    g = golden("m3500_batch.npz")
    ftype, fa, fb, _, _ = factor_arrays(m3500)
    p = HostPlan().build(m3500.n_nodes, ftype, fa, fb)
    assert np.array_equal(p.array("order"), g["ordering"])
    assert np.array_equal(node_parents(p, m3500.n_nodes), g["tree_parents"])
    info = p.info()
    assert info["nsn"] <= info["N"] and info["n_slots"] == 5453


@pytest.mark.parametrize("n", [1, 2, 3, 4, 7, 13, 64, 257, 900])
def test_subgraph_ordering_matches_reference(m3500, n):
    want = refcases.load(f"head{n}")
    sub = m3500.head(n)
    ref_order, ref_par = want["order"], want["parents"]
    ftype, fa, fb, _, _ = factor_arrays(sub)
    p = HostPlan().build(n, ftype, fa, fb)
    assert np.array_equal(p.array("order"), ref_order)
    assert np.array_equal(node_parents(p, n), ref_par)


def test_synthetic_ordering_matches_reference():
    d = datasets.manhattan_dense(1500, seed=3)
    ref_order = refcases.load("synth1500")["order"]
    ftype, fa, fb, _, _ = factor_arrays(d)
    p = HostPlan().build(d.n_nodes, ftype, fa, fb)
    assert np.array_equal(p.array("order"), ref_order)


def test_quotient_graph_ordering_equals_explicit_elimination():
    """The production ordering keeps the elimination graph implicitly (elements + exact degrees on
    demand); it must give the permutation of the explicit-clique implementation on any graph."""
    from support.hostplan import ref_ordering
    rng = np.random.default_rng(11)
    for n, extra in [(1, 0), (2, 1), (7, 5), (40, 60), (300, 200), (300, 2000), (2500, 4000)]:
        lo = list(range(n - 1))
        hi = list(range(1, n))
        for _ in range(extra):
            a, b = rng.integers(0, n, 2)
            if a != b:
                lo.append(int(min(a, b)))
                hi.append(int(max(a, b)))
        lo, hi = np.array(lo, dtype=np.int64), np.array(hi, dtype=np.int64)
        if n == 1:
            continue
        assert np.array_equal(ref_ordering(n, lo, hi), ref_ordering(n, lo, hi, explicit=True)), (n, extra)
    for d in (datasets.manhattan_dense(4000, seed=9), datasets.manhattan_sparse(9000, seed=4)):
        lo, hi = np.minimum(d.ea, d.eb), np.maximum(d.ea, d.eb)
        assert np.array_equal(ref_ordering(d.n_nodes, lo, hi), ref_ordering(d.n_nodes, lo, hi, explicit=True))


# ---------------------------------------------------------------------------------------------
# plan + emulated kernels == reference solution
# ---------------------------------------------------------------------------------------------
def emulate_batch(d):
    n = d.n_nodes
    ftype, fa, fb, fz, fW = factor_arrays(d)
    p = HostPlan().build(n, ftype, fa, fb)
    info = p.info()
    Hs = emul.Hessian(n, info["n_slots"])
    Hs.reset(n, 1e-4)
    lp = d.init.copy()
    node2q = p.array("node2q")
    Hs.linearize(range(len(ftype)), ftype, fa, fb, fz, fW, lp, lp, node2q, p.array("fslot"))
    fr = emul.Fronts()
    fr.ensure(n)
    desc, ipool = p.descs(), p.array("ipool")
    leaf = p.array("leaf_tasks")  # large graphs: k_factor_leaf runs these first (children first)
    if len(leaf):
        emul.factor(fr, Hs, desc, ipool, p.array("q2node"), leaf, None)
    emul.factor(fr, Hs, desc, ipool, p.array("q2node"), p.array("tasks"), p.array("nwait"), prior=leaf)
    emul.backsolve(fr, desc, ipool, p.array("btasks"))
    x = np.stack([fr.x[3 * node2q[i]:3 * node2q[i] + 3] for i in range(n)])
    st = lp + x
    st[:, 2] = emul.mod2pi(st[:, 2])
    return st


def test_emulated_batch_matches_golden_m3500(m3500):
    g = golden("m3500_batch.npz")
    st = emulate_batch(m3500)
    assert np.abs(st - g["states"][0]).max() < 1e-7


def test_emulated_batch_synthetic_vs_reference():
    d = datasets.manhattan_dense(600, seed=2)
    ref = refcases.load("synth600")["states"]
    assert np.abs(emulate_batch(d) - ref).max() < 1e-6 * max(1.0, np.abs(ref).max())


def test_large_plan_leaf_set_and_merged_chains():
    """12 k-pose dense world: the schedule splits into the leaf set (warp-per-front kernel) and the
    rest, chains of team-sized fronts are merged into wide supernodes; the emulated kernels on that
    plan still solve the normal equations (checked against a sparse direct solve)."""
    import scipy.sparse.linalg as spl
    d = datasets.manhattan_dense(12000, seed=5)
    n = d.n_nodes
    ftype, fa, fb, fz, fW = factor_arrays(d)
    p = HostPlan().build(n, ftype, fa, fb)
    D = p.descs()
    leaf, tasks, nwait = p.array("leaf_tasks"), p.array("tasks"), p.array("nwait")
    assert len(leaf) >= 4096 and (3 * D["mb"][leaf]).max() <= 63
    in_leaf = np.zeros(len(D["mb"]), bool)
    in_leaf[leaf] = True
    par = D["parent"]
    assert all(in_leaf[c] for c in range(len(par)) if par[c] >= 0 and in_leaf[par[c]]), "leaf set is downward closed"
    assert sorted(set(leaf) | set(tasks)) == list(range(len(par))) and not (set(leaf) & set(tasks))
    wide = D["cb"] > 32
    assert wide.any(), "fundamental chains of team-sized fronts are merged past the 32-pose cap"
    m = 3 * D["mb"][wide]
    assert ((((m + 2) // 2) * 2) * m > 25600).all(), "only fronts of the team path may be wider than the cap"
    st = emulate_batch(d)
    # exact Gauss-Newton step from the same Hessian
    Hs = emul.Hessian(n, p.info()["n_slots"])
    Hs.reset(n, 1e-4)
    Hs.linearize(range(len(ftype)), ftype, fa, fb, fz, fW, d.init, d.init, p.array("node2q"), p.array("fslot"))
    fslot = p.array("fslot")
    pairs = {}
    for f in range(len(ftype)):
        if ftype[f] == 1:
            pairs[fslot[f]] = (min(fa[f], fb[f]), max(fa[f], fb[f]))
    A = Hs.dense([pairs[s] for s in range(p.info()["n_slots"])])
    x = spl.spsolve(A.tocsc(), Hs.B.reshape(-1)).reshape(n, 3)
    want = d.init + x
    want[:, 2] = emul.mod2pi(want[:, 2])
    assert np.abs(st - want).max() < 1e-6 * max(1.0, np.abs(want).max())


def test_team_front_merge_and_backsolve_order(monkeypatch):
    """Team-sized fronts absorb their chain parent while the explicit zero rows stay below ASAM_TEAM_MERGE_PCT per cent
    (plan.c, supernode formation): fewer, wider supernodes, the same solution.  The back-substitution list (ordered by
    modelled chain time) must stay parents-first, blocks of a wide supernode last block first."""
    d = datasets.manhattan_dense(9000, seed=11)
    n = d.n_nodes
    ftype, fa, fb, fz, fW = factor_arrays(d)
    monkeypatch.setenv("ASAM_TEAM_MERGE_PCT", "0")
    p0 = HostPlan().build(n, ftype, fa, fb)
    st0 = emulate_batch(d)
    monkeypatch.setenv("ASAM_TEAM_MERGE_PCT", "40")
    p1 = HostPlan().build(n, ftype, fa, fb)
    st1 = emulate_batch(d)
    D0, D1 = p0.descs(), p1.descs()
    assert len(D1["mb"]) < len(D0["mb"]), "merging removes supernodes"
    assert np.array_equal(p0.array("node2q"), p1.array("node2q")), "the elimination order is untouched"
    lblocks = lambda D: int((D["cb"].astype(np.int64) * D["mb"] - D["cb"].astype(np.int64) * (D["cb"] - 1) // 2).sum())
    assert lblocks(D1) > lblocks(D0), "explicit zero blocks were added to L"
    assert np.abs(st1 - st0).max() < 1e-9 * max(1.0, np.abs(st0).max())
    for p in (p0, p1):
        bt, par = p.array("btasks"), p.descs()["parent"]
        sn, blk = bt & 0xFFFFFF, bt >> 24
        first = {}
        for k, s in enumerate(sn):
            first.setdefault(int(s), k)
        assert all(par[s] < 0 or first[int(par[s])] < first[s] for s in first), "parents first"
        for s in set(int(x) for x in sn[blk > 0]):
            b = blk[sn == s]
            assert (np.diff(b) < 0).all(), "last block first"


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_schedule_emulated(world):
    """Multi-GPU schedule (SURVEY.md section 8e): every rank factors its shards, the shard roots' trailing
    columns are exchanged, every rank factors the top, back-solves top + own shards, solution segments
    are exchanged.  Emulated with one numpy arena per rank; the result must equal the single-rank one."""
    d = datasets.manhattan_dense(6000, seed=7)
    n = d.n_nodes
    ftype, fa, fb, fz, fW = factor_arrays(d)
    ref = emulate_batch(d)
    plans = [HostPlan().build(n, ftype, fa, fb, world=world, rank=r) for r in range(world)]
    desc, ipool, q2node, node2q = plans[0].descs(), plans[0].array("ipool"), plans[0].array("q2node"), plans[0].array("node2q")
    nsn = len(desc["mb"])
    own = plans[0].array("shard_owner")
    q0, qn = plans[0].array("shard_q0"), plans[0].array("shard_qn")
    off, cnt = plans[0].array64("shard_off"), plans[0].array64("shard_cnt")
    assert len(own) >= world and set(own) == set(range(world)), "every rank gets work"
    for p in plans[1:]:  # the cut is the same on every rank
        assert np.array_equal(p.array("shard_owner"), own) and np.array_equal(p.array64("shard_off"), off)
        assert np.array_equal(p.array("top_tasks"), plans[0].array("top_tasks"))
    top = set(int(t) for t in plans[0].array("top_tasks"))
    seen = set(top)
    for r, p in enumerate(plans):
        mine = set(int(t) for t in p.array("tasks")) | set(int(t) for t in p.array("leaf_tasks"))
        assert not (mine & seen), "shards are disjoint from each other and from the top"
        seen |= mine
        assert set(int(t) & 0xffffff for t in p.array("btasks")) == mine | top
    assert seen == set(range(nsn)), "top + shards cover the tree"
    # shard intervals are disjoint position ranges
    iv = sorted(zip(q0, q0 + qn))
    assert all(a[1] <= b[0] for a, b in zip(iv, iv[1:]))
    root_of = {}  # shard root front offset -> shard
    for s_ in range(nsn):
        m_, c_ = 3 * int(desc["mb"][s_]), 3 * int(desc["cb"][s_])
        for i in range(len(own)):
            ld_ = (m_ + 2) & ~1  # ASAM_LD: leading dimension rounded up to even
            if int(desc["f_off"][s_]) + c_ * ld_ == off[i] and (m_ - c_) * ld_ == cnt[i]:
                root_of[s_] = i
    assert len(root_of) == len(own), "every exchanged range is the trailing part of one root front"

    Hs = emul.Hessian(n, plans[0].info()["n_slots"])
    Hs.reset(n, 1e-4)
    Hs.linearize(range(len(ftype)), ftype, fa, fb, fz, fW, d.init, d.init, node2q, plans[0].array("fslot"))
    arenas = []
    for r, p in enumerate(plans):  # phase 1: own shards
        fr = emul.Fronts()
        fr.ensure(n)
        leaf = p.array("leaf_tasks")
        if len(leaf):
            emul.factor(fr, Hs, desc, ipool, q2node, leaf, None)
        emul.factor(fr, Hs, desc, ipool, q2node, p.array("tasks"), p.array("nwait"), prior=leaf)
        arenas.append(fr)
    for s_, i in root_of.items():  # exchange: root fronts of the shards
        o = int(desc["f_off"][s_])
        for r in range(world):
            if r != own[i]:
                arenas[r].F[o] = arenas[own[i]].F[o]
                arenas[r].rhs[o] = arenas[own[i]].rhs[o]
    xs = []
    for r, p in enumerate(plans):  # phase 2: top (redundantly) + back-solve of top and own shards
        done_before = [s_ for s_ in range(nsn) if s_ not in top]
        emul.factor(arenas[r], Hs, desc, ipool, q2node, p.array("top_tasks"), p.array("top_nwait"), prior=done_before,
                    count_prior=False)
        emul.backsolve(arenas[r], desc, ipool, p.array("btasks"))
        xs.append(arenas[r].x.copy())
    x = xs[0].copy()
    for i in range(len(own)):  # exchange: solution segments
        x[3 * q0[i]:3 * (q0[i] + qn[i])] = xs[own[i]][3 * q0[i]:3 * (q0[i] + qn[i])]
    st = d.init + np.stack([x[3 * node2q[i]:3 * node2q[i] + 3] for i in range(n)])
    st[:, 2] = emul.mod2pi(st[:, 2])
    assert np.abs(st - ref).max() < 1e-9 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("n0,n1,step", [(1, 40, 1), (120, 200, 1), (300, 330, 3)])
def test_emulated_incremental_append(m3500, n0, n1, step):
    """plan_append: re-factoring only the marked supernodes reproduces the full solution."""
    db, estart = m3500.bucketed()
    ftype, fa, fb, fz, fW = factor_arrays(db, estart[n0])
    p = HostPlan().build(n0, ftype, fa, fb)
    Hs = emul.Hessian(n0, p.info()["n_slots"])
    Hs.reset(n0, 1e-4)
    lp = m3500.init.copy()
    Hs.linearize(range(len(ftype)), ftype, fa, fb, fz, fW, lp, lp, p.array("node2q"), p.array("fslot"))
    fr = emul.Fronts()
    fr.ensure(n0)
    emul.factor(fr, Hs, p.descs(), p.array("ipool"), p.array("q2node"), p.array("tasks"), p.array("nwait"))
    F0, N0 = len(ftype), n0
    for n in range(n0 + step, n1 + 1, step):
        ftype, fa, fb, fz, fW = factor_arrays(db, estart[n])
        order, pos, ppos = p.array("order"), p.array("pos"), p.array("parent_pos")
        marked = set()
        for f in range(F0, len(ftype)):
            for v in ([fa[f], fb[f]] if ftype[f] == 1 else [fa[f]]):
                while v < N0 and v not in marked:
                    marked.add(int(v))
                    pp = ppos[pos[v]]
                    if pp < 0:
                        break
                    v = order[pp]
        r = p.append(n, ftype, fa, fb, sorted(marked))
        assert r is not None
        tasks, nwait = r
        info = p.info()
        Hs.grow(n, info["n_slots"])
        fr.ensure(n)
        node2q = p.array("node2q")
        Hs.linearize(range(F0, len(ftype)), ftype, fa, fb, fz, fW, lp, lp, node2q, p.array("fslot"))
        desc, ipool = p.descs(), p.array("ipool")
        emul.factor(fr, Hs, desc, ipool, p.array("q2node"), tasks, nwait, keep=p.last_keep)  # checks the kept columns
        F0, N0 = len(ftype), n
    emul.backsolve(fr, desc, ipool, np.arange(info["nsn"] - 1, -1, -1))
    fslot = p.array("fslot")
    pairs = {}
    for f in range(len(ftype)):
        if ftype[f] == 1:
            pairs[fslot[f]] = (min(fa[f], fb[f]), max(fa[f], fb[f]))
    A = Hs.dense([pairs[s] for s in range(info["n_slots"])])
    xs = spl.spsolve(A.tocsc(), Hs.B.reshape(-1))
    x_node = np.concatenate([fr.x[3 * node2q[i]:3 * node2q[i] + 3] for i in range(N0)])
    assert np.abs(x_node - xs).max() < 1e-8 * max(1.0, np.abs(xs).max())
    assert getattr(fr, "kept_cols", 0) > 0, "some step kept the leading columns of a marked supernode"


def test_append_rejects_edge_between_old_poses(m3500):
    sub = m3500.head(50)
    ftype, fa, fb, _, _ = factor_arrays(sub)
    p = HostPlan().build(50, ftype, fa, fb)
    ftype2 = np.r_[ftype, 1].astype(np.int32)
    fa2 = np.r_[fa, 3].astype(np.int32)
    fb2 = np.r_[fb, 40].astype(np.int32)
    assert p.append(50, ftype2, fa2, fb2, [3, 40]) is None  # rc == 2: caller falls back


# ---------------------------------------------------------------------------------------------
# oracle pinned against the golden vectors; data generators
# ---------------------------------------------------------------------------------------------
def test_reference_oracle_reproduces_golden(m3500):
    if not H.available("reference"):
        pytest.skip("reference oracle not built")
    g = golden("m3500_batch.npz")
    with H.Harness("reference") as h:
        h.load_full(m3500)
        assert abs(h.chi2() - g["chi2"][0]) < 1e-9 * g["chi2"][0]
        h.batch()
        assert np.array_equal(h.states(), g["states"][0])
    r = golden("m3500_replay.npz")
    with H.Harness("reference") as h:
        h.replay_begin(m3500)
        chi2, _, info = h.replay_to(150)
        assert np.array_equal(chi2, r["chi2"][:150])
        assert np.array_equal(info[:, 0], r["naffected"][:150])


def test_golden_known_answers():
    """Values quoted in SURVEY.md section 8c."""
    g = golden("m3500_batch.npz")
    assert abs(g["chi2"][0] - 1283333.8296) < 1e-3
    assert abs(g["chi2"][1] - 127723.205936) < 1e-5
    assert abs(g["chi2"][6] - 70.1644936267) < 1e-8
    r = golden("m3500_replay.npz")
    assert abs(r["chi2"][-1] - 68.965607796) < 1e-8
    assert abs(r["chi2"][499] - 8.330019947) < 1e-8


def test_generators_are_seeded():
    a, b = datasets.manhattan_dense(800, 1), datasets.manhattan_dense(800, 1)
    assert np.array_equal(a.ea, b.ea) and np.array_equal(a.ez, b.ez) and np.array_equal(a.init, b.init)
    c = datasets.manhattan_dense(800, 2)
    assert not np.array_equal(a.ez[:10], c.ez[:10])
    assert 3.5 * 800 < a.n_edges < 4.5 * 800
    s = datasets.manhattan_sparse(2000, 1)
    assert 2000 - 1 < s.n_edges < 2000 * 1.1
    key = np.maximum(s.ea, s.eb)
    assert np.all(np.diff(key) >= 0) and np.all(s.ea < s.eb)


# ---------------------------------------------------------------------------------------------
# the plain-C oracle port, pinned against the golden vectors of the real reference
# ---------------------------------------------------------------------------------------------
def test_oracle_port_matches_golden(m3500):
    sys.path.insert(0, ROOT)
    from oracle import port
    g = golden("m3500_batch.npz")
    assert abs(port.chi2(m3500, m3500.init) - g["chi2"][0]) < 1e-9 * g["chi2"][0]
    st = m3500.init
    for it in range(2):
        st = port.batch_step(m3500, st)
        assert np.abs(st - g["states"][it]).max() < 1e-7, it
        assert abs(port.chi2(m3500, st) - g["chi2"][it + 1]) < 1e-7 * g["chi2"][it + 1]


def test_oracle_port_small_graphs_vs_reference(m3500):
    sys.path.insert(0, ROOT)
    from oracle import port
    for n in (1, 2, 3, 11, 150):
        sub = m3500.head(n)
        want = refcases.load(f"head{n}")
        ref, c = want["states"], float(want["chi2"])
        st = port.batch_step(sub, sub.init)
        assert np.abs(st - ref).max() < 1e-9, n
        assert abs(port.chi2(sub, st) - c) <= 1e-9 * max(1.0, c)


# ---------------------------------------------------------------------------------------------
# ".graph" files and attributes (SURVEY.md section 8f items 1-2)
# ---------------------------------------------------------------------------------------------
def _same_graph(x, y):
    assert x.n_nodes == y.n_nodes and x.n_factors == y.n_factors
    assert np.array_equal(x.states(), y.states())
    for f in range(x.n_factors):
        fx, fy = x.factor(f), y.factor(f)
        assert fx[:3] == fy[:3] and np.array_equal(fx[3], fy[3]) and np.array_equal(fx[4], fy[4])
        if f > 0:
            assert x.attr_get(x.FACTOR, f, "type") == y.attr_get(y.FACTOR, f, "type") != None  # noqa: E711
    assert x.attr_get(x.GRAPH, 0, "name") == y.attr_get(y.GRAPH, 0, "name") == "M3500 head"
    assert x.attr_get(x.GRAPH, 0, "poses", "uint64") == y.attr_get(y.GRAPH, 0, "poses", "uint64") == x.n_nodes
    assert x.attr_get(x.NODE, 3, "tag") == y.attr_get(y.NODE, 3, "tag") == "third"
    assert x.attr_get(x.NODE, 4, "tag") is None and y.attr_get(y.NODE, 4, "tag") is None


def test_graph_file_round_trip(m3500, tmp_path):
    """april_graph_save -> april_graph_create_from_file gives the same graph, attributes included."""
    path = str(tmp_path / "small.graph")
    with H.Harness("b200") as a, H.Harness("b200") as b:
        refcases.build_small(a, m3500)
        assert a.save(path)
        assert b.load(path) == a.n_nodes
        _same_graph(a, b)
        assert b.load(str(tmp_path / "missing.graph")) == -1


def test_graph_file_interchange_with_reference(m3500, tmp_path):
    """Files written by this library load in the reference and vice versa (same stype framing): the file the
    reference writes for this graph (tests/golden/m3500_head40.graph) loads here, and ours is the same file
    byte for byte but for the 8-byte object cookies, which count up per process in both libraries."""
    ours, theirs = str(tmp_path / "ours.graph"), os.path.join(ROOT, "tests", "golden", "m3500_head40.graph")
    with H.Harness("b200") as a, H.Harness("b200") as a2:
        refcases.build_small(a, m3500)
        assert a.save(ours)
        assert a2.load(theirs) == a.n_nodes, "we read the reference's file"
        _same_graph(a, a2)
    cookie = bytes.fromhex("7b287f8a1579")  # high bytes of the cookie sequence (serial.c next_magic)

    def masked(path):
        b = bytearray(open(path, "rb").read())
        i = b.find(cookie)
        while i >= 0:
            b[i + 6:i + 8] = b"\0\0"
            i = b.find(cookie, i + 8)
        return bytes(b)

    x, y = masked(ours), masked(theirs)
    assert len(x) == len(y) and y.count(cookie) > 0
    assert x == y, [i for i in range(len(x)) if x[i] != y[i]][:20]


def test_reference_examples_link_unchanged(built, tmp_path):
    """SURVEY.md section 8(f) item 1: the reference's four example programs compile and link against this library
    without a source change (oracle/Makefile builds them into oracle/_ref/ where the reference sources are
    present); the two that do not solve anything run here on the CPU, save + load included (the upstream simple
    example dies in the reference's own decoder because it forgets april_graph_stype_init(); this library
    registers the built-in types itself)."""
    names = ["aprilsam_graph_save_simple", "aprilsam_graph_save_with_attributes", "aprilsam_tutorial", "aprilsam_demo"]
    exe = {n: os.path.join(ROOT, "oracle", "_ref", "ref_" + n) for n in names}
    if not all(os.path.exists(p) for p in exe.values()):
        pytest.skip("the reference's example programs were not built (no reference sources at build time)")
    for n in names[:2]:
        r = subprocess.run([exe[n], "--path", str(tmp_path / (n + ".graph"))], capture_output=True, text=True, timeout=60)
        assert r.returncode == 0, (n, r.stdout[-500:], r.stderr[-500:])
        out = r.stdout
        a, b = out.split("Load graph")
        assert [l for l in a.splitlines() if l.startswith("node_")] == [l for l in b.splitlines() if l.startswith("node_")]
    assert "Graph name: AprilSAM-Graph" in out and out.count("factor type: geopin") == 2


def test_host_plan_under_sanitizers(tmp_path):
    """plan.c + ordering.c under AddressSanitizer / UBSan / LeakSanitizer: batch plan (leaf set, merged chains, team sizes),
    the schedules of 3 and 8 ranks, and 40 incremental appends on top of a batch plan."""
    csan = os.path.join(ROOT, "tests", "support", "csan")
    exe = str(tmp_path / "plan_san")
    inc = ["-I" + os.path.join(ROOT, p) for p in ("include", "include/aprilsam", "aprilsam_b200/host")]
    r = subprocess.run(["gcc", "-g", "-O1", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-std=gnu11"] + inc +
                       ["-o", exe, os.path.join(csan, "plan_driver.c"), os.path.join(csan, "device_stubs.c"),
                        os.path.join(ROOT, "aprilsam_b200", "host", "plan.c"), os.path.join(ROOT, "aprilsam_b200", "host", "ordering.c"), "-lm"],
                       capture_output=True, text=True)
    if r.returncode != 0 and "sanitize" in r.stderr:
        pytest.skip("no sanitizer runtime in this toolchain")
    assert r.returncode == 0, r.stderr[-2000:]
    for args in (["3000", "1"], ["20000", "1"], ["20000", "3"], ["30000", "8"]):
        r = subprocess.run([exe] + args, capture_output=True, text=True, timeout=600, env=dict(os.environ, ASAN_OPTIONS="detect_leaks=1"))
        assert r.returncode == 0 and "ERROR" not in r.stderr and "runtime error" not in r.stderr, (args, r.stderr[-1500:])
        assert "rank 0/" in r.stdout
