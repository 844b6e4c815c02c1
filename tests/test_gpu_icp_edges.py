"""The ICP kernel's fallback and limit paths against the oracle.

test_gpu_icp.py pins the kernel on the inputs it is tuned for: street scans, odometry-close initial guesses, a few
uniform problems per launch and the whole device.  The branches below are written to be "slower, still exact" and are
the ones production reaches first (a big map, a bad odometry jump, a wide batch).  Every test first asserts that its
input really reaches the branch it names, then asserts bit equality -- with the oracle (T, T_iter after every
iteration, ids / d2 of the last iteration, iterations, converged, last_kept, last_limit) or with the same call made
where the branch is not taken.

- Table-pool overflow: a 7.5 M-point map needs more than the 262144 fine tables the pool holds, so the cells beyond
  it stay leaves (stats.grid_overflow == 1, stats.grid_tables counts past the pool).  Pins the overflowing cells'
  leaf counts against the oracle and against the same registration with no overflow.
- Uncapped search: an initial guess 25 m off puts the trimmed quantile of iteration 0 beyond 12.8 m, so the search
  cap grows through every step (0.04 .. 163.84 m^2) to infinity.  Alone (static scheduling) and in a batch (dynamic
  scheduling).  A CPU test pins the oracle itself on this input against the float64 restatement of test_oracle.py.
- Ties at the trimmed limit: a lattice read at a half-cell offset gives thousands of exactly equal d2 at the limit,
  so `d2 <= limit` (not `<`) decides last_kept; plus trim ratios 0.001 and 0.3.
- The differential checker's ring at smooth_length 1, 2 and 15 (kMaxSmooth), with runs that stop on convergence
  and runs that stop on the counter.
- Independence from the CTA count: 1, 2, 3, 5, 37 CTAs for one problem and 1, 2, 3 CTAs per problem in a batch give
  the bits of the whole device.
- Wide, ragged batches: 17, 75, 149 and 160 (kMaxBatch) problems in one launch, readings of 1..131072 points,
  sub-maps of 1..16 (kMaxParts) parts; each equals its own single call, a sample equals the oracle; 161 problems and
  17 parts are refused without harming the context.
- Workspace reuse: one context run through builds of changing size and geometry (including the overflow build and
  the error paths) gives what a fresh context gives for every call.
- Normals strides 3, 4, 8 and 12 give identical bits; a stride the ABI refuses raises LsError.
"""
import contextlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_oracle import _independent_icp  # noqa: E402

THREADS = os.cpu_count() or 1
POOL_TABLES = 262144           # fine tables in the pool: 1.5 GB / (LS_FB3 = 512 cells * 12 bytes)
LAST_FINITE_CAP = 163.84       # m^2: the last search cap before the uncapped search (0.04 * 4^6)
I4 = np.eye(4, dtype=np.float32)
ORACLE_FIELDS = ("max_iterations", "trim_ratio", "use_differential", "min_diff_rot", "min_diff_trans", "smooth_length")


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _params(oracle_mod, **kw):
    """(device params, oracle params) of the same chain; grid tuning only exists on the device."""
    import laser_slam_b200 as ls
    return ls.default_params(**kw), oracle_mod.default_params(num_threads=THREADS,
                                                              **{k: v for k, v in kw.items() if k in ORACLE_FIELDS})


def _stats(s):
    return (s.iterations, s.converged, s.max_iter_reached, s.last_kept, s.last_limit)


def _assert_equals_oracle(g, r, what=""):
    """Full comparison of an icp_register(want_ids, want_hist) result with oracle.icp(want_hist)."""
    assert g["rc"] == r["rc"] == 0, what
    assert _stats(g["stats"]) == _stats(r["stats"]), what
    assert np.array_equal(g["T_iter_hist"], r["T_iter_hist"]), what
    assert np.array_equal(g["ids"], r["ids_hist"][-1]) and np.array_equal(g["d2"], r["d2_last"]), what
    assert np.array_equal(g["T"], r["T"]), what


def _assert_same_outcome(a, b, what=""):
    """Two device results of the same registration (any entry point): same rc, transform and stats."""
    assert a["rc"] == b["rc"], what
    assert np.array_equal(a["T"], b["T"]), what
    assert _stats(a["stats"]) == _stats(b["stats"]), what


def _assert_identical(a, b, what=""):
    """Two device results of the same call, every output that both carry."""
    _assert_same_outcome(a, b, what)
    for k in ("ids", "d2", "T_iter_hist"):
        if k in a or k in b:
            assert np.array_equal(a[k], b[k]), (what, k)
    sa, sb = a["stats"], b["stats"]
    assert (sa.grid_cells, sa.grid_tables, sa.grid_overflow) == (sb.grid_cells, sb.grid_tables, sb.grid_overflow), what


@contextlib.contextmanager
def _new_context():
    import laser_slam_b200 as ls
    ctx = ls.Context(0)
    try:
        yield ctx
    finally:
        ctx.close()


def _moved(T, dt, deg):
    """T with a yaw of `deg` degrees and a translation (dt, -dt/2, dt/4) applied on the left."""
    a = np.deg2rad(deg)
    M = np.eye(4)
    M[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    M[:3, 3] = [dt, -dt / 2, dt / 4]
    return (M @ np.asarray(T, np.float64)).astype(np.float32)


def _unit_rows(rng, m):
    v = rng.normal(size=(m, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def _ones4(xyz):
    out = np.ones((len(xyz), 4), np.float32)
    out[:, :3] = xyz
    return out


def _iteration0(oracle_mod, reading, ref, T0, ratio):
    """d2 of every reading point and the trimmed limit of iteration 0, from the oracle's pieces."""
    mu = oracle_mod.mean(ref)
    Tpre = np.asarray(T0, np.float32).copy()
    Tpre[:3, 3] -= mu
    q = oracle_mod.transform_points(Tpre, reading)[:, :3].copy()
    _, d2 = oracle_mod.nn_kdtree(q, (ref[:, :3] - mu).astype(np.float32), THREADS)
    limit, _ = oracle_mod.trim_limit(d2, ratio)
    return d2, limit


class _Pool:
    """A few synthetic sequences, their scans sub-sampled to 8192 points, pushed into one map on demand.  Problems are
    (reading id, part ids, part transforms, T0) tuples plus what the oracle needs (reading and assembled sub-map)."""

    def __init__(self, synth_mod, scans, traj, mp, seqs, n_scans=6):
        self.mp, self.seqs, self.n_scans = mp, seqs, n_scans
        self.seq = {}
        for s in seqs:
            if s == 0:
                (truth, odom), full = traj, scans[:n_scans]
            else:
                truth, odom = synth_mod.trajectory(s, n_scans)
                full = [synth_mod.scan(truth[k], s, k) for k in range(n_scans)]
            self.seq[s] = (truth, odom, [synth_mod.subsample(*f, 16) for f in full], full)
        self.ids = {}

    def _push(self, key, pts, nrm):
        if key not in self.ids:
            self.ids[key] = self.mp.push_scan(pts, nrm)
        return self.ids[key]

    def problem(self, oracle_mod, b, n_parts, n_read, dt=0.0, deg=0.0):
        s = self.seqs[b % len(self.seqs)]
        truth, odom, sub, full = self.seq[s]
        k = 1 + (b // len(self.seqs)) % (self.n_scans - 1)          # reading scan; the sub-map is centred on k-1
        ref = k - 1
        ks = [(ref - j) % self.n_scans for j in range(n_parts)]     # more parts than scans: scans repeat
        Ts = [I4.copy() if kk == ref else (np.linalg.inv(truth[ref]) @ truth[kk]).astype(np.float32) for kk in ks]
        if n_read == len(full[k][0]):
            rd_pts, rd_nrm = full[k]
        else:
            sel = np.linspace(0, len(sub[k][0]) - 1, n_read).astype(np.int64) if n_read < len(sub[k][0]) else slice(None)
            rd_pts, rd_nrm = np.ascontiguousarray(sub[k][0][sel]), np.ascontiguousarray(sub[k][1][sel])
        rid = self._push(("rd", s, k, n_read), rd_pts, rd_nrm)
        pids = [self._push(("part", s, kk), *sub[kk]) for kk in ks]
        T0 = _moved(np.linalg.inv(truth[ref]) @ odom[k], dt, deg)
        parts = [sub[kk] if np.array_equal(T, I4) else oracle_mod.transform_cloud(T, *sub[kk]) for kk, T in zip(ks, Ts)]
        host = dict(reading=rd_pts, ref=np.concatenate([p[0] for p in parts]), ref_normals=np.concatenate([p[1] for p in parts]))
        return (rid, pids, Ts, T0), host


def _small_batch(oracle_mod, pool, count):
    """`count` problems of 8192 points against sub-maps of 1..4 parts, T0 up to 0.4 m / 2 deg from odometry."""
    out = [pool.problem(oracle_mod, b, 1 + b % 4, 8192, dt=[0.0, 0.1, 0.4][b % 3], deg=[0.0, 1.0, 2.0][b % 3])
           for b in range(count)]
    return [p for p, _ in out], [h for _, h in out]


# ---- fixtures --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def overflow_problem():
    """About 7.5 M points uniform in a 70 x 70 x 60 m box: ~294 k one-metre cells of ~25 points, so with leaf_split 16
    well over the pool's 262144 cells need a fine table.  The reading is 16384 of the points under a small motion."""
    import oracle
    rng = np.random.default_rng(17)
    m = 7_500_000
    ref = _ones4(rng.uniform([-35.0, -35.0, -30.0], [35.0, 35.0, 30.0], (m, 3)).astype(np.float32))
    nrm = _unit_rows(rng, m)
    pick = np.sort(rng.choice(m, 16384, replace=False))
    motion = _moved(I4, 0.08, 1.5)
    reading = oracle.transform_points(np.linalg.inv(motion.astype(np.float64)).astype(np.float32), ref[pick])
    return dict(reading=reading, ref=ref, ref_normals=nrm, T0=I4.copy())


@pytest.fixture(scope="module")
def lattice():
    """Reference: the integer lattice 20 x 20 x 10 (mean exactly (9.5, 9.5, 4.5), so centring is exact).  Reading: the
    lattice shifted by (0.5, 0, 0) -- every point exactly 0.5 m from two lattice points, d2 == 0.25 -- and 1200 lattice
    points moved by less than 0.45 m (d2 < 0.25), in shuffled order."""
    rng = np.random.default_rng(23)
    g = np.stack(np.meshgrid(np.arange(20), np.arange(20), np.arange(10), indexing="ij"), -1).reshape(-1, 3).astype(np.float64)
    pick = rng.choice(len(g), 1200, replace=False)
    v = rng.normal(size=(1200, 3))
    v *= rng.uniform(0.0, 0.45, (1200, 1)) / np.linalg.norm(v, axis=1, keepdims=True)
    rd = np.concatenate([g + [0.5, 0.0, 0.0], g[pick] + v])[rng.permutation(len(g) + 1200)]
    return dict(reading=_ones4(rd.astype(np.float32)), ref=_ones4(g.astype(np.float32)), ref_normals=_unit_rows(rng, len(g)),
                T0=I4.copy())


def _far_off(small_pair):
    """small_pair with T0 25 m off along y: the trimmed quantile of iteration 0 lies beyond 12.8 m.  (Along y the normal
    equations stay well conditioned, cond(A) ~ 2e4, so the float64 restatement is a fair judge of the oracle there.)"""
    T0 = small_pair["T0"].copy()
    T0[1, 3] += 25.0
    return T0


# ---- 1. table-pool overflow ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_table_pool_overflow_equals_oracle_and_the_unsplit_build(gpu_ctx, oracle_mod, overflow_problem):
    P = overflow_problem
    pg, po = _params(oracle_mod, max_iterations=5, use_differential=0, leaf_split=16)
    g = gpu_ctx.icp_register(P["reading"], P["ref"], P["ref_normals"], P["T0"], pg, want_ids=True, want_hist=True)
    assert g["stats"].grid_overflow == 1                      # precondition: the pool ran out ...
    assert g["stats"].grid_tables > POOL_TABLES               # ... and the counter kept counting past it
    r = oracle_mod.icp(P["reading"], P["ref"], P["ref_normals"], P["T0"], po, want_hist=True)
    assert r["stats"].iterations == 5
    _assert_equals_oracle(g, r, "overflowing build")
    d = gpu_ctx.icp_register(P["reading"], P["ref"], P["ref_normals"], P["T0"],
                             _params(oracle_mod, max_iterations=5, use_differential=0)[0], want_ids=True, want_hist=True)
    assert d["stats"].grid_overflow == 0 and d["stats"].grid_tables < POOL_TABLES
    _assert_same_outcome(g, d, "default leaf_split")
    assert np.array_equal(g["ids"], d["ids"]) and np.array_equal(g["T_iter_hist"], d["T_iter_hist"])


# ---- 2. uncapped search ----------------------------------------------------------------------------------------------
def test_oracle_agrees_with_the_float64_restatement_at_a_far_off_guess(oracle_mod, small_pair):
    sp = small_pair
    T0 = _far_off(sp)
    _, limit = _iteration0(oracle_mod, sp["reading"], sp["ref"], T0, 0.75)
    assert limit > LAST_FINITE_CAP
    for iters in (1, 3):
        r = oracle_mod.icp(sp["reading"], sp["ref"], sp["ref_normals"], T0,
                           oracle_mod.default_params(max_iterations=iters, use_differential=0))
        T = _independent_icp(sp["reading"], sp["ref"], sp["ref_normals"], T0, iters)
        assert r["rc"] == 0 and r["stats"].iterations == iters
        assert np.abs(r["T"][:3, 3] - T[:3, 3]).max() < 1e-4, iters
        dR = r["T"][:3, :3].astype(np.float64) @ T[:3, :3].T
        assert np.linalg.norm([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]]) / 2 < 1e-5, iters


@pytest.mark.gpu
def test_uncapped_search_alone_and_in_a_batch_equals_oracle(gpu_ctx, oracle_mod, synth_mod, small_pair, scans, traj):
    sp = small_pair
    T0 = _far_off(sp)
    _, limit = _iteration0(oracle_mod, sp["reading"], sp["ref"], T0, 0.75)
    assert limit > LAST_FINITE_CAP                            # precondition: only the uncapped search finds the quantile
    mp = gpu_ctx.create_map(16, 131072)
    pool = _Pool(synth_mod, scans, traj, mp, seqs=(0,))
    normal, _ = _small_batch(oracle_mod, pool, 4)
    rid = mp.push_scan(sp["reading"], np.zeros((len(sp["reading"]), 3), np.float32))
    sid = mp.push_scan(sp["ref"], sp["ref_normals"])
    for iters in (1, 3):
        pg, po = _params(oracle_mod, max_iterations=iters, use_differential=0)
        r = oracle_mod.icp(sp["reading"], sp["ref"], sp["ref_normals"], T0, po, want_hist=True)
        assert r["stats"].last_limit > LAST_FINITE_CAP or iters > 1
        g = gpu_ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], T0, pg, want_ids=True, want_hist=True)
        _assert_equals_oracle(g, r, f"alone, {iters} iterations")
        far = (rid, [sid], [I4], T0)
        batch = mp.register_batch([normal[0], far, normal[1], normal[2]], pg)
        _assert_same_outcome(batch[1], g, f"in a batch, {iters} iterations")
        for b, pr in zip((0, 2, 3), (normal[0], normal[1], normal[2])):
            _assert_same_outcome(batch[b], mp.register(*pr, pg), f"neighbour {b}, {iters} iterations")
    mp.close()


# ---- 3. ties at the trimmed limit ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [0.75, 0.5, 1.0])
def test_exact_ties_at_the_trimmed_limit_equal_oracle(gpu_ctx, oracle_mod, lattice, ratio):
    L = lattice
    n = len(L["reading"])
    d2, limit = _iteration0(oracle_mod, L["reading"], L["ref"], L["T0"], ratio)
    assert limit == 0.25 and (d2 == limit).sum() > 1          # precondition: many d2 exactly at the limit ...
    if ratio < 1.0:                                           # ... straddling the quantile (at ratio 1 it is the maximum)
        assert (d2 <= limit).sum() > int(np.float32(n) * np.float32(ratio)) + 1
    pg, po = _params(oracle_mod, max_iterations=5, use_differential=0, trim_ratio=ratio)
    r = oracle_mod.icp(L["reading"], L["ref"], L["ref_normals"], L["T0"], po, want_hist=True)
    g = gpu_ctx.icp_register(L["reading"], L["ref"], L["ref_normals"], L["T0"], pg, want_ids=True, want_hist=True)
    _assert_equals_oracle(g, r, f"lattice, ratio {ratio}")
    one = gpu_ctx.icp_register(L["reading"], L["ref"], L["ref_normals"], L["T0"],
                               _params(oracle_mod, max_iterations=1, use_differential=0, trim_ratio=ratio)[0])
    assert one["stats"].last_kept == int((d2 <= limit).sum()) and one["stats"].last_limit == limit


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [0.001, 0.3])
def test_extreme_trim_ratios_equal_oracle(gpu_ctx, oracle_mod, small_pair, ratio):
    sp = small_pair
    pg, po = _params(oracle_mod, max_iterations=5, use_differential=0, trim_ratio=ratio)
    r = oracle_mod.icp(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], po, want_hist=True)
    g = gpu_ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], pg, want_ids=True, want_hist=True)
    assert r["stats"].last_kept >= int(np.float32(len(sp["reading"])) * np.float32(ratio)) + 1
    _assert_equals_oracle(g, r, f"small_pair, ratio {ratio}")


# ---- 4. the differential checker's ring ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_checker_ring_lengths_equal_oracle(gpu_ctx, oracle_mod, small_pair):
    sp = small_pair
    outcomes = []
    for L in (1, 2, 15):
        for rot, trans in ((0.001, 0.01), (0.05, 0.5)):
            pg, po = _params(oracle_mod, use_differential=1, smooth_length=L, min_diff_rot=rot, min_diff_trans=trans)
            r = oracle_mod.icp(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], po, want_hist=True)
            g = gpu_ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], pg, want_ids=True, want_hist=True)
            _assert_equals_oracle(g, r, (L, rot, trans))
            outcomes.append((g["stats"].iterations, g["stats"].converged))
    assert len({it for it, _ in outcomes}) >= 2, outcomes                     # precondition: the ring decides ...
    assert any(c == 1 and it < pg.max_iterations for it, c in outcomes), outcomes  # ... and stops some runs early


# ---- 5. independence from the CTA count ------------------------------------------------------------------------------
@pytest.mark.gpu
def test_results_do_not_depend_on_the_cta_count(oracle_mod, synth_mod, config2, scans, traj):
    import laser_slam_b200 as ls
    c2 = config2
    p = ls.default_params(max_iterations=8, use_differential=0)
    with _new_context() as ctx:
        full = ctx.set_icp_cta_budget(0)
        assert full >= 37
        want = ctx.icp_register(c2["reading"], c2["ref"], c2["ref_normals"], c2["T0"], p, want_ids=True, want_hist=True)
        for budget in (1, 2, 3, 5, 37):
            assert ctx.set_icp_cta_budget(budget) == budget      # precondition: one problem on `budget` CTAs
            got = ctx.icp_register(c2["reading"], c2["ref"], c2["ref_normals"], c2["T0"], p, want_ids=True, want_hist=True)
            _assert_identical(got, want, f"single problem, {budget} CTAs")
        mp = ctx.create_map(16, 131072)
        problems, _ = _small_batch(oracle_mod, _Pool(synth_mod, scans, traj, mp, seqs=(0,)), 8)
        pb = ls.default_params(max_iterations=12, use_differential=0)
        assert ctx.set_icp_cta_budget(0) == full
        want_b = mp.register_batch(problems, pb)
        for per in (1, 2, 3):
            assert ctx.set_icp_cta_budget(8 * per) // len(problems) == per   # precondition: `per` CTAs per problem
            got = mp.register_batch(problems, pb)
            for b in range(len(problems)):
                _assert_same_outcome(got[b], want_b[b], f"batch of 8, {per} CTAs per problem, problem {b}")
        mp.close()


# ---- 6. wide, ragged batches -----------------------------------------------------------------------------------------
READING_SIZES = (1, 31, 32, 33, 1000, 8192)


@pytest.fixture(scope="module")
def wide(synth_mod, scans, traj):
    """Its own context (up to 160 workspaces, freed at the end of the module) and a map holding three sequences."""
    with _new_context() as ctx:
        mp = ctx.create_map(128, 131072)
        yield ctx, mp, _Pool(synth_mod, scans, traj, mp, seqs=(0, 1, 2))
        mp.close()


def _wide_problems(oracle_mod, pool, B):
    """Problem b: reading size READING_SIZES[b % 6] (problem B // 2: a full 131072-point scan), 1 + b % 16 parts, T0 off
    odometry by 0 / 0.05 m 0.5 deg / 0.4 m 2 deg / 1.2 m 4 deg (b % 4)."""
    out = []
    for b in range(B):
        n_read = 131072 if b == B // 2 else READING_SIZES[b % len(READING_SIZES)]
        out.append(pool.problem(oracle_mod, b, 1 + b % 16, n_read, dt=[0.0, 0.05, 0.4, 1.2][b % 4], deg=[0, 0.5, 2, 4][b % 4]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("B", [17, 75, 149, 160])
def test_wide_ragged_batch_equals_single_calls_and_oracle(oracle_mod, wide, B):
    _, mp, pool = wide
    probs = _wide_problems(oracle_mod, pool, B)
    pg, po = _params(oracle_mod, max_iterations=12)
    got = mp.register_batch([p for p, _ in probs], pg)
    seen_n, seen_parts = set(), set()
    for b, ((pr, host), res) in enumerate(zip(probs, got)):
        single = mp.register(*pr, pg, raise_on_convergence=False)
        _assert_same_outcome(res, single, f"B={B}, problem {b}")
        n, k = len(host["reading"]), len(pr[1])
        if b % 8 == 0 or n not in seen_n or k not in seen_parts:
            r = oracle_mod.icp(host["reading"], host["ref"], host["ref_normals"], pr[3], po)
            assert res["rc"] == r["rc"], (B, b, n, k)
            assert np.array_equal(res["T"], r["T"]), (B, b, n, k)
            assert _stats(res["stats"]) == _stats(r["stats"]), (B, b, n, k)
        seen_n.add(n)
        seen_parts.add(k)
    assert seen_n == set(READING_SIZES) | {131072} and seen_parts == set(range(1, 17))
    ok = [r["stats"] for r in got if r["rc"] == 0]
    assert any(s.converged == 1 and s.iterations < 12 for s in ok)        # precondition: some stop on the checker ...
    assert any(s.max_iter_reached == 1 and s.converged == 0 for s in ok)  # ... and some on the counter


@pytest.mark.gpu
def test_batch_limits_are_refused_and_leave_the_context_usable(oracle_mod, wide):
    import laser_slam_b200 as ls
    ctx, mp, pool = wide
    probs = [p for p, _ in _wide_problems(oracle_mod, pool, 161)]
    pg = ls.default_params(max_iterations=12)
    want = mp.register(*probs[0], pg)
    with pytest.raises(ls.LsError):
        mp.register_batch(probs, pg)                                       # 161 > kMaxBatch
    _assert_same_outcome(mp.register(*probs[0], pg), want, "after B = 161")
    rid, pids, Ts, T0 = probs[0]
    too_many = (rid, [pids[0]] * 17, [Ts[0]] * 17, T0)
    with pytest.raises(ls.LsError):
        mp.register_batch([probs[1], too_many], pg)                        # 17 > kMaxParts
    with pytest.raises(ls.LsError):
        mp.register(*too_many, pg)
    _assert_same_outcome(mp.register(*probs[0], pg), want, "after 17 parts")
    again = mp.register_batch(probs[:2], pg)
    _assert_same_outcome(again[0], want, "batch after the refusals")


# ---- 7. workspace reuse ----------------------------------------------------------------------------------------------
def _error_calls(ctx, small_pair):
    """The calls of test_gpu_icp.py::test_error_paths."""
    import laser_slam_b200 as ls
    sp = small_pair
    empty4, empty3 = np.zeros((0, 4), np.float32), np.zeros((0, 3), np.float32)
    with pytest.raises(ls.ConvergenceError):
        ctx.icp_register(empty4, sp["ref"], sp["ref_normals"], sp["T0"])
    out = ctx.icp_register(sp["reading"], empty4, empty3, sp["T0"], raise_on_convergence=False)
    assert out["rc"] == ls.LS_ERR_CONVERGENCE and np.array_equal(out["T"], sp["T0"])
    with pytest.raises(ls.LsError):
        ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], ls.default_params(max_iterations=0))
    with pytest.raises(ls.LsError):
        ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], ls.default_params(trim_ratio=1.5))
    return None


@pytest.mark.gpu
def test_workspace_reuse_equals_a_fresh_context(oracle_mod, synth_mod, config2, small_pair, overflow_problem, lattice,
                                                scans, traj):
    import laser_slam_b200 as ls
    c2, sp, ov, L = config2, small_pair, overflow_problem, lattice

    def one(P, p):
        return lambda ctx: ctx.icp_register(P["reading"], P["ref"], P["ref_normals"], P["T0"], p, want_ids=True, want_hist=True)

    def batch16(ctx):
        mp = ctx.create_map(16, 131072)
        problems, _ = _small_batch(oracle_mod, _Pool(synth_mod, scans, traj, mp, seqs=(0,)), 16)
        out = mp.register_batch(problems, ls.default_params(max_iterations=12))
        mp.close()
        return out

    coarse = ls.default_params(max_iterations=6, use_differential=0, cell_size=0.25, max_cells=4096)
    steps = [("config 2", one(c2, ls.default_params(max_iterations=8, use_differential=0))),
             ("small_pair, 0.25 m cells in at most 4096", one(sp, coarse)),
             ("overflowing build", one(ov, ls.default_params(max_iterations=5, use_differential=0, leaf_split=16))),
             ("lattice", one(L, ls.default_params(max_iterations=5, use_differential=0))),
             ("batch of 16", batch16),
             ("error paths", lambda ctx: _error_calls(ctx, sp)),
             ("config 2 again", one(c2, ls.default_params(max_iterations=8, use_differential=0))),
             ("small_pair again", one(sp, coarse))]
    with _new_context() as ctx:
        for name, call in steps:
            got = call(ctx)
            with _new_context() as fresh:
                want = call(fresh)
            if name == "overflowing build":
                assert got["stats"].grid_overflow == 1
            if name.startswith("small_pair"):     # the level-0 cell had to grow: 0.25 m cells would need far more
                ext = sp["ref"][:, :3].max(0) - sp["ref"][:, :3].min(0)
                assert got["stats"].grid_cells <= 4096 and np.prod(ext / 0.25) > 64 * 4096
            if isinstance(got, list):
                for b, (x, y) in enumerate(zip(got, want)):
                    _assert_same_outcome(x, y, (name, b))
            elif got is not None:
                _assert_identical(got, want, name)


# ---- 8. normals stride -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_normals_stride_gives_identical_bits(gpu_ctx, small_pair):
    import laser_slam_b200 as ls
    sp = small_pair
    m = len(sp["ref"])
    p = ls.default_params(max_iterations=8, use_differential=0)

    def padded(cols):
        a = np.full((m, cols), np.nan, np.float32)     # garbage in the extra columns: NaN poisons any stray read
        a[:, :3] = sp["ref_normals"]
        return a

    want = gpu_ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"], sp["T0"], p, want_ids=True, want_hist=True)
    for cols in (4, 8, 12):
        got = gpu_ctx.icp_register(sp["reading"], sp["ref"], padded(cols), sp["T0"], p, want_ids=True, want_hist=True)
        _assert_identical(got, want, f"icp_register, stride {cols}")
    with pytest.raises(ls.LsError):
        gpu_ctx.icp_register(sp["reading"], sp["ref"], sp["ref_normals"][:, :2], sp["T0"], p)
    mp = gpu_ctx.create_map(8, 8192)
    rid = mp.push_scan(sp["reading"], np.zeros((len(sp["reading"]), 3), np.float32))
    ref_ids = {cols: mp.push_scan(sp["ref"], padded(cols)) for cols in (3, 4, 8, 12)}
    for cols, sid in ref_ids.items():
        got = mp.register(rid, [sid], [I4], sp["T0"], p, want_ids=True, want_hist=True)
        assert np.array_equal(got["T"], want["T"]) and np.array_equal(got["ids"], want["ids"]), cols
        assert np.array_equal(got["T_iter_hist"], want["T_iter_hist"]), cols
    f = np.ascontiguousarray(sp["ref"])
    n2, n12 = np.ascontiguousarray(padded(4)[:, :2]), padded(12)
    with pytest.raises(ls.LsError):
        mp.push_scan_raw(f.ctypes.data, n2.ctypes.data, 2, m)              # stride < 3
    with pytest.raises(ls.LsError):
        mp.push_scan_raw_async(f.ctypes.data, n12.ctypes.data, 12, m)      # the asynchronous upload takes 3..8
    mp.close()
