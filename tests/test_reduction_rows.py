"""Per-scenario reduction rows and the plane gather against exact references.

`mpcf_cost_residual_batch` (closed-form F0 torque bound) and `mpcf_cost_residual_table_batch` (per-node, per-joint bound table)
write out[4][B] = (cost, defect, torque-bound, fatigue-bound) per scenario: the only per-scenario result that leaves a GPU
(all-gathered by the multi-GPU runner, returned by `HostStepPipeline(outputs="reduced")`).  `mpcf_gather_planes` packs what the
host pipeline sends back.

The reference (`reduce_ref`) restates both reductions in numpy.  The three maxima are of single double operations (|a - b|,
lb - tau, tau - ub, f+ - f_max), so numpy reproduces them exactly and they are compared bit for bit; a NaN in any entry a row
reads makes the row NaN.  The cost is compared with the exact sum of exact products (fractions.Fraction) within the bound of
sequential summation.  The CPU tests check the reference against a literal loop and show that mutants of it (the bugs the GPU
tests are meant to catch) differ from it on the very inputs the GPU tests use.  The reduction kernels read only n from the
model, so the GPU tests feed hand-built planes.
"""
import ctypes as C
import math
from fractions import Fraction

import mpmath
import numpy as np
import pytest

GAP = 512  # canary doubles on each side of every carved buffer
CANARY = -7.25e300
U53 = 2.0 ** -53
# CUDA C++ Programming Guide, "Mathematical Functions", double precision: exp(x) has a maximum error of 1 ulp.  The reference
# bound rounds the exact exponential (0.5 ulp), so the two exponentials are at most 1 ulp apart as doubles; tau0 * e and
# |tau| - bound each add one rounding.  The closed-form r1 row is therefore within 3 ulp of max(|tau|, bound).
EXP_R1_ULPS = 3
SMEM_TABLE_MAX = 200 * 1024  # bytes of the bound table the table entry accepts (2 n N doubles)
MODELS = {3: "pilz3", 6: "pilz6", 16: "generic16", 64: "generic64"}


def _carve(pool, sizes):
    """views of `pool` separated by GAP canary doubles; returns (views, gap slices, total length)"""
    views, gaps, off = [], [], 0
    for sz in sizes:
        gaps.append(slice(off, off + GAP))
        off += GAP
        off = (off + 15) // 16 * 16  # 128-byte alignment of every buffer
        views.append(pool[off:off + sz])
        off += sz
    gaps.append(slice(off, off + GAP))
    return views, gaps, off + GAP


# ------------------------------------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------------------------------------
def _rowmax(vals, nan_drop=False):
    """The kernels' running maximum from +0.0 over the leading axes of vals [..., B]: NaN when any value is NaN, otherwise the
    largest value, and +0.0 when none exceeds 0 (-0.0 included).  nan_drop: fmax semantics, where a NaN operand is ignored."""
    vals = vals.reshape(-1, vals.shape[-1])
    if vals.shape[0] == 0:
        return np.zeros(vals.shape[-1])
    if nan_drop:
        vals = np.where(np.isnan(vals), -np.inf, vals)
    m = vals.max(axis=0)  # np.max propagates NaN
    return np.where(np.isnan(m), np.nan, np.where(m > 0.0, m, 0.0))


def f0_bounds(N, dt, tau0, alpha, tau_floor):
    """bound_k = max(tau0 exp((-alpha k) dt), tau_floor) as the kernel forms it, with the exponential correctly rounded"""
    mpmath.mp.prec = 200
    return np.array([max(tau0 * float(mpmath.exp(mpmath.mpf((-alpha * float(k)) * dt))), tau_floor) for k in range(N)])


def reduce_ref(case, mut=frozenset()):
    """(cost, r0, r1, r2) [4][B] of `case` (see _case).  The cost is the kernel's sequential sum (k outer, i inner) without
    fused multiply-adds; it is compared with the exact cost, not with this.  `mut` selects deliberate bugs (MUTANTS)."""
    n, N, B = case["n"], case["N"], case["B"]
    q, qd, f, tau, qn, qdn, fn = (case[k].reshape(n, N, B) for k in ("q", "qd", "f", "tau", "qn", "qdn", "fn"))
    nj = n - 1 if "joints_n_minus_1" in mut else n
    drop = "fmax" in mut
    w_qd, w_tau = (case["w_tau"], case["w_qd"]) if "swap_w" in mut else (case["w_qd"], case["w_tau"])
    cost = np.zeros(B)
    for k in range(N):
        for i in range(nj):
            v, t = qd[i, k], tau[i, k]
            cost = cost + (w_qd * v * v + w_tau * t * t)
    npair = N - 2 if "pairs_N_minus_2" in mut else N - 1
    blocks = [(qn, q, "drop_q"), (qdn, qd, "drop_qd"), (fn, f, "drop_f")]
    d = [np.abs(a[:nj, :npair] - b[:nj, 1:npair + 1]) for a, b, tag in blocks if tag not in mut and npair > 0]
    r0 = _rowmax(np.concatenate(d) if d else np.zeros((0, B)), drop)
    t = tau[:nj]
    if case["table"] is None:
        r1 = _rowmax(np.abs(t) - case["bounds"][None, :, None], drop)
    else:
        tab = case["table"].reshape(-1)
        tab = tab.reshape(n, N, 2).transpose(1, 0, 2) if "table_nN" in mut else tab.reshape(N, n, 2)
        lb, ub = tab[:, :nj, 0].T[:, :, None], tab[:, :nj, 1].T[:, :, None]
        if "swap_lb_ub" in mut:
            lb, ub = ub, lb
        inner = np.fmax(lb - t, t - ub) if drop else np.maximum(lb - t, t - ub)
        r1 = _rowmax(inner, drop)
    r2 = _rowmax(fn[:nj] - case["f_max"], drop)
    return np.stack([cost, r0, r1, r2])


def reduce_loop(case):
    """The same reduction as a literal loop over (k, i, b), statement for statement as the kernels run it."""
    n, N, B = case["n"], case["N"], case["B"]
    U = N * B
    q, qd, f, tau, qn, qdn, fn = (case[k].reshape(-1) for k in ("q", "qd", "f", "tau", "qn", "qdn", "fn"))

    def mx(r, x):
        return x if (x > r or math.isnan(x)) else r
    out = np.zeros((4, B))
    for b in range(B):
        cost, r0, r1, r2 = 0.0, 0.0, 0.0, 0.0
        for k in range(N):
            u = k * B + b
            for i in range(n):
                o = i * U + u
                v, t = float(qd[o]), float(tau[o])
                cost += case["w_qd"] * v * v + case["w_tau"] * t * t
                if case["table"] is None:
                    r1 = mx(r1, abs(t) - float(case["bounds"][k]))
                else:
                    tb = case["table"].reshape(-1)
                    r1 = mx(r1, mx(float(tb[2 * (k * n + i)]) - t, t - float(tb[2 * (k * n + i) + 1])))
                r2 = mx(r2, float(fn[o]) - case["f_max"])
                if k + 1 < N:
                    o1 = o + B
                    r0 = mx(r0, abs(float(qn[o]) - float(q[o1])))
                    r0 = mx(r0, abs(float(qdn[o]) - float(qd[o1])))
                    r0 = mx(r0, abs(float(fn[o]) - float(f[o1])))
        out[:, b] = (cost, r0, r1, r2)
    return out


def write_ref(buf, rows, col0, ld_out, mut=frozenset()):
    """Where the table entry puts the rows of a chunk in a [4][ld_out] buffer (flat `buf`): columns [col0, col0 + B)."""
    B = rows.shape[1]
    ld = B if "ignore_ld_out" in mut else ld_out
    out = buf.copy()
    for j in range(4):
        out[j * ld + col0:j * ld + col0 + B] = rows[j]
    return out


def _cost_bound_check(case, got_cost, scenarios):
    """|cost - exact| <= (2 n N + 2) 2^-53 sum |terms| (sequential summation of 2 n N products of two roundings each), with the
    exact sum of exact products in rational arithmetic.  NaN / inf inputs are the NaN tests' business."""
    n, N, B = case["n"], case["N"], case["B"]
    qd, tau = case["qd"].reshape(n, N, B), case["tau"].reshape(n, N, B)
    wq, wt = Fraction(case["w_qd"]), Fraction(case["w_tau"])
    bad = []
    for b in scenarios:
        exact, mag = Fraction(0), Fraction(0)
        for v in qd[:, :, b].reshape(-1).tolist():
            x = wq * Fraction(v) ** 2
            exact += x
            mag += abs(x)
        for t in tau[:, :, b].reshape(-1).tolist():
            x = wt * Fraction(t) ** 2
            exact += x
            mag += abs(x)
        err = abs(Fraction(float(got_cost[b])) - exact)
        if not err <= (2 * n * N + 2) * Fraction(U53) * mag:
            bad.append((b, float(got_cost[b]), float(exact)))
    assert not bad, bad[:5]


def _sample(case, budget=60000):
    """every scenario when their products fit the budget, otherwise an even sample that includes the first and the last"""
    B, per = case["B"], 2 * case["n"] * case["N"]
    k = max(2, budget // per)
    return list(range(B)) if B <= k else sorted(set(np.linspace(0, B - 1, k).astype(int).tolist()))


def _same_bits(a, b):
    """equal bit for bit, with any NaN matching any NaN (the payload of a device NaN is not specified)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64)))


def assert_rows(got, case, scenarios=None):
    """maxima bit for bit (closed-form r1: within EXP_R1_ULPS of max(|tau|, bound)); cost within the summation bound"""
    ref = reduce_ref(case)
    got = np.asarray(got)
    assert _same_bits(got[1], ref[1]), ("defect row", np.flatnonzero(~_eq(got[1], ref[1]))[:8])
    assert _same_bits(got[3], ref[3]), ("fatigue-bound row", np.flatnonzero(~_eq(got[3], ref[3]))[:8])
    if case["table"] is None and case["alpha"] != 0.0:
        n, N, B = case["n"], case["N"], case["B"]
        scale = np.maximum(np.abs(case["tau"].reshape(n, N, B)), case["bounds"][None, :, None]).max(axis=(0, 1))
        nan = np.isnan(ref[2])
        assert np.array_equal(np.isnan(got[2]), nan)
        assert np.all(np.abs(got[2] - ref[2])[~nan] <= EXP_R1_ULPS * np.spacing(scale[~nan])), "torque-bound row"
        assert not np.signbit(got[2]).any()
    else:
        assert _same_bits(got[2], ref[2]), ("torque-bound row", np.flatnonzero(~_eq(got[2], ref[2]))[:8])
    assert np.array_equal(np.isnan(got[0]), np.isnan(ref[0]))
    fin = [b for b in (range(case["B"]) if scenarios is None else scenarios) if np.isfinite(ref[0, b])]
    _cost_bound_check(case, got[0], fin)


def _eq(a, b):
    return (a == b) | (np.isnan(a) & np.isnan(b))


# ------------------------------------------------------------------------------------------------------------------------------
# cases: planes [n][N*B] with node-major units u = k*B + b, built on the CPU so the CPU tests see the GPU tests' inputs
# ------------------------------------------------------------------------------------------------------------------------------
def _case(n, N, B, seed, *, w_qd=1.0, w_tau=1e-2, f_max=50.0, table=None, dt=0.05, tau0=50.0, alpha=2.0, tau_floor=15.0,
          tau_scale=60.0):
    """Random states whose defects are exactly zero: x+_k is a copy of x_{k+1} for k < N - 1; x+ at the last node is random
    (there is no node N).  The caller plants defects, NaNs and bounds in the arrays."""
    rng = np.random.default_rng(seed)
    q, qd = rng.uniform(-2.0, 2.0, (n, N, B)), rng.uniform(-1.5, 1.5, (n, N, B))
    f, tau = rng.uniform(20.0, 60.0, (n, N, B)), rng.uniform(-tau_scale, tau_scale, (n, N, B))
    qn, qdn, fn = (np.empty_like(a) for a in (q, qd, f))
    for nxt, cur, lo, hi in ((qn, q, -2.0, 2.0), (qdn, qd, -1.5, 1.5), (fn, f, 20.0, 60.0)):
        nxt[:, :-1] = cur[:, 1:]
        nxt[:, -1] = rng.uniform(lo, hi, (n, B))
    c = dict(n=n, N=N, B=B, w_qd=w_qd, w_tau=w_tau, f_max=f_max, table=table, dt=dt, tau0=tau0, alpha=alpha, tau_floor=tau_floor)
    c.update(q=q, qd=qd, f=f, tau=tau, qn=qn, qdn=qdn, fn=fn)
    c["bounds"] = f0_bounds(N, dt, tau0, alpha, tau_floor)
    return c


def _flat(case):
    """the [n][N*B] contiguous planes of a case (reshapes of the [n][N][B] arrays, which share memory with them)"""
    for k in ("q", "qd", "f", "tau", "qn", "qdn", "fn"):
        case[k] = np.ascontiguousarray(case[k]).reshape(case["n"], -1)
    return case


def _view3(case, k):
    return case[k].reshape(case["n"], case["N"], case["B"])


def planted_defects(n, N, with_table=False, plant=True):
    """One defect per scenario, each of a distinct magnitude: in every block (q+, qd+, f+), at joint 0 and n - 1, at node pair 0
    and N - 2; plus mismatches of q+ / qd+ at the last node, which no row reads.  Returns (case, {b: (block, i, k)});
    plant=False: the same states without the defects."""
    sites = [(blk, i, k) for blk in ("qn", "qdn", "fn") for i in sorted({0, n - 1}) for k in sorted({0, N - 2})]
    sites += [("qn", n - 1, N - 1), ("qdn", 0, N - 1)]
    B = 2 * len(sites) + 3
    c = _case(n, N, B, seed=100 + n + N, f_max=61.0)  # f_max above every f+: the fatigue row stays +0.0 but for the plants
    if with_table:
        c["table"] = _random_table(n, N, seed=7)
    where = {}
    for j, (blk, i, k) in enumerate(sites):
        b = 2 * j + 1  # unplanted neighbours on both sides
        if plant:
            _view3(c, blk)[i, k, b] += 0.125 * (j + 1) + 1e-3 * j
        where[b] = (blk, i, k)
    return _flat(c), where


def _random_table(n, N, seed):
    """distinct (lb, ub) per (k, i), lb < 0 < ub, so a transposed index or swapped bounds changes the row"""
    rng = np.random.default_rng(seed)
    lb = -rng.uniform(5.0, 55.0, (N, n)) - 1e-3 * np.arange(N * n).reshape(N, n)
    ub = rng.uniform(5.0, 55.0, (N, n)) + 1e-3 * np.arange(N * n).reshape(N, n)
    return np.ascontiguousarray(np.stack([lb, ub], axis=-1))


# (array, node) -> rows that must become NaN for a NaN there, N >= 3.  q and f at node 0 are read by no row (the defect
# compares x+_k with x_{k+1}); q+ and qd+ at the last node are read by no row (there is no node N); f+ at the last node only by
# the fatigue-bound row; qd by the cost at every node.
NAN_NODES = ("first", "middle", "last")
EXPECTED_NAN = {
    ("q", "first"): (), ("q", "middle"): ("r0",), ("q", "last"): ("r0",),
    ("qd", "first"): ("cost",), ("qd", "middle"): ("cost", "r0"), ("qd", "last"): ("cost", "r0"),
    ("f", "first"): (), ("f", "middle"): ("r0",), ("f", "last"): ("r0",),
    ("tau", "first"): ("cost", "r1"), ("tau", "middle"): ("cost", "r1"), ("tau", "last"): ("cost", "r1"),
    ("qn", "first"): ("r0",), ("qn", "middle"): ("r0",), ("qn", "last"): (),
    ("qdn", "first"): ("r0",), ("qdn", "middle"): ("r0",), ("qdn", "last"): (),
    ("fn", "first"): ("r0", "r2"), ("fn", "middle"): ("r0", "r2"), ("fn", "last"): ("r2",),
}
ROWS = ("cost", "r0", "r1", "r2")


def nan_case(n, arr, node, with_table=False, B=9, N=5, b=4, i=None):
    c = _case(n, N, B, seed=300 + n, f_max=45.0, alpha=0.0 if not with_table else 2.0, tau0=40.0)
    if with_table:
        c["table"] = _random_table(n, N, seed=8)
    k = {"first": 0, "middle": N // 2, "last": N - 1}[node]
    _view3(c, arr)[n // 2 if i is None else i, k, b] = np.nan
    return _flat(c)


def weights_case(n, w):
    return _flat(_case(n, 9, 37, seed=500 + n, w_qd=w[0], w_tau=w[1]))


def ld_out_case(n):
    c = _flat(_case(n, 6, 45, seed=600 + n))
    c["table"] = _random_table(n, 6, seed=9)
    return c


LD_OUT = dict(col0=5, ld=45 + 5 + 11)


def f0_case(n):
    """dt, alpha, tau0, tau_floor such that the floor takes over at node KF = 13 of 20 (50 e^{-0.1 k}: 15.06 at k = 12, 13.6 at
    k = 13).  Scenarios 1..5 carry tau = +/-(floor + j ulp), j = -2..2, at node KF (alternating sign); scenarios 7..9 carry
    tau at the exponential bound of node KF - 1 and 1 ulp either side; scenario 11 has f+ = f_max exactly, scenario 12
    f+ = f_max + 1 ulp.  Every other |tau| < 5 and f+ < f_max, so those rows are +0.0 but for the plants."""
    N, B, KF = 20, 16, 13
    c = _case(n, N, B, seed=700 + n, dt=0.05, tau0=50.0, alpha=2.0, tau_floor=15.0, f_max=61.0, tau_scale=5.0)
    tau, fn = _view3(c, "tau"), _view3(c, "fn")
    for j, b in zip(range(-2, 3), range(1, 6)):
        tau[n - 1, KF, b] = (-1) ** b * (15.0 + j * np.spacing(15.0))
    bk = c["bounds"][KF - 1]
    for j, b in zip((-1, 0, 1), (7, 8, 9)):
        tau[0, KF - 1, b] = -(bk + j * np.spacing(bk)) if b == 8 else bk + j * np.spacing(bk)
    fn[n // 2, N - 1, 11] = 61.0
    fn[0, 3, 12] = 61.0 + np.spacing(61.0)
    return _flat(c), KF


# mutants of the reference, and the planted cases on which each must differ from it
MUTANTS = ("fmax", "drop_q", "drop_qd", "drop_f", "joints_n_minus_1", "pairs_N_minus_2", "swap_w", "table_nN", "swap_lb_ub",
           "ignore_ld_out")


# ------------------------------------------------------------------------------------------------------------------------------
# CPU tests
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("n,N,B", [(3, 1, 4), (3, 2, 3), (6, 5, 7), (4, 3, 2)])
def test_reference_equals_literal_loop(n, N, B, table):
    c = _case(n, N, B, seed=n * 100 + N * 10 + B, tau_scale=60.0, w_qd=0.7, w_tau=3.0)
    rng = np.random.default_rng(1)
    if table:
        c["table"] = _random_table(n, N, seed=2)
        c["table"][rng.integers(0, N), rng.integers(0, n)] = (-np.inf, np.inf)
    for arr in ("q", "qd", "f", "tau", "qn", "qdn", "fn"):  # perturb some entries so that defects are non-zero
        a = _view3(c, arr)
        a[rng.integers(0, n), rng.integers(0, N), rng.integers(0, B)] += 0.3
    _view3(c, "tau")[0, 0, 0] = -0.0
    _view3(c, "fn")[0, N - 1, B - 1] = np.nan
    _flat(c)
    assert _same_bits(reduce_ref(c), reduce_loop(c))


def test_planted_constructor_gives_zero_defects_except_where_planted():
    for n, N in ((3, 2), (6, 7), (16, 3)):
        c, where = planted_defects(n, N)
        ref = reduce_ref(c)
        for b in range(c["B"]):
            if b in where and where[b][2] < N - 1:
                assert ref[1, b] > 0.0, (n, N, b, where[b])
            else:  # unplanted, or planted at the last node, which no defect reads
                assert ref[1, b] == 0.0 and not np.signbit(ref[1, b]), (n, N, b)
        for blk, cur in (("qn", "q"), ("qdn", "qd"), ("fn", "f")):
            clean = _case(n, N, c["B"], seed=100 + n + N)  # x+_k is a copy of x_{k+1}
            assert np.array_equal(clean[blk][:, :-1], clean[cur][:, 1:])


def test_expected_nan_rows_follow_from_the_reference():
    for (arr, node), rows in EXPECTED_NAN.items():
        for table in (False, True):
            ref = reduce_ref(nan_case(6, arr, node, table))
            assert [r for j, r in enumerate(ROWS) if np.isnan(ref[j, 4])] == list(rows), (arr, node, table)
            assert not np.isnan(np.delete(ref, 4, axis=1)).any()
    c = _flat(_case(6, 5, 3, seed=1, f_max=45.0))
    _view3(c, "fn")[2, 1, 1] = np.inf
    ref = reduce_ref(c)
    assert ref[3, 1] == np.inf and ref[1, 1] == np.inf


def _differs(case, mut):
    a, b = reduce_ref(case), reduce_ref(case, frozenset([mut]))
    return not _same_bits(a, b)


@pytest.mark.parametrize("mut", MUTANTS)
def test_reference_mutants_are_caught_by_the_gpu_cases(mut):
    """Each mutant differs from the reference on the inputs of the GPU test that is meant to catch it, so that test can fail."""
    for n in MODELS:
        if mut in ("drop_q", "drop_qd", "drop_f", "joints_n_minus_1", "pairs_N_minus_2"):
            for N in (2, 7):
                assert _differs(planted_defects(n, N)[0], mut), (n, N)
        elif mut == "fmax":
            for (arr, node), rows in EXPECTED_NAN.items():
                if set(rows) & {"r0", "r1", "r2"}:
                    for table in (False, True):
                        assert _differs(nan_case(n, arr, node, table), mut), (n, arr, node, table)
        elif mut == "swap_w":
            for w in ((1.0, 0.0), (0.0, 1.0), (0.3, 7.0)):
                c = weights_case(n, w)
                assert not np.allclose(reduce_ref(c)[0], reduce_ref(c, frozenset([mut]))[0], rtol=1e-6), (n, w)
        elif mut in ("table_nN", "swap_lb_ub"):
            c, _ = planted_defects(n, 7, with_table=True)
            assert _differs(c, mut), n
        else:  # ignore_ld_out
            c = ld_out_case(n)
            rows = reduce_ref(c)
            buf = np.full(4 * LD_OUT["ld"], CANARY)
            assert not np.array_equal(write_ref(buf, rows, LD_OUT["col0"], LD_OUT["ld"]),
                                      write_ref(buf, rows, LD_OUT["col0"], LD_OUT["ld"], frozenset([mut])))


def test_pair_guard_mutant_needs_the_last_pair():
    """k + 1 < N - 1 drops only node pair N - 2: the planted cases put a defect there in every block."""
    c, where = planted_defects(6, 7)
    ref, mut = reduce_ref(c), reduce_ref(c, frozenset(["pairs_N_minus_2"]))
    changed = {b for b in range(c["B"]) if ref[1, b] != mut[1, b]}
    assert changed == {b for b, (blk, i, k) in where.items() if k == 5}


def test_f0_case_puts_the_floor_in_the_middle_of_the_horizon():
    c, KF = f0_case(6)
    b = f0_bounds(20, 0.05, 50.0, 2.0, 15.0)
    assert b[KF] == 15.0 and b[KF - 1] > 15.0 * (1 + 1e-3) and 50.0 * math.exp(-2.0 * KF * 0.05) < 15.0 * (1 - 1e-3)
    ref = reduce_ref(c)
    ulp = np.spacing(15.0)
    assert [float(x) for x in ref[2, 1:6]] == [0.0, 0.0, 0.0, ulp, 2 * ulp]
    assert ref[3, 11] == 0.0 and not np.signbit(ref[3, 11]) and ref[3, 12] == np.spacing(61.0)
    assert ref[2, 8] == 0.0 and ref[2, 9] == np.spacing(b[KF - 1])


# ------------------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------------------------------------
_model_cache = {}


def _model(n):
    from mpc_fatigue_b200.model import Model, data_urdf
    if n not in _model_cache:
        if n in (3, 6):
            m = Model.from_urdf(data_urdf(MODELS[n]), armature=1e-2)
        else:
            m = Model.synthetic("chain", n, seed=5, armature=1e-2)
        assert m.n == n and m.kernel_family == ("chain%d" % n if n < 16 else MODELS[n])
        _model_cache[n] = m
    return _model_cache[n]


def _ev(n):
    from mpc_fatigue_b200.evaluator import BatchEvaluator
    return BatchEvaluator(_model(n), "cuda:0")


def _dev(case):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(case[k])).cuda() for k in ("q", "qd", "f", "tau", "qn", "qdn", "fn")]


def run_entry(case, entry, out=None, out_col0=0):
    """the rows of `case` from the closed-form ("closed") or the table ("table") entry, as [4][B] numpy"""
    import torch
    ev, B, N = _ev(case["n"]), case["B"], case["N"]
    args = _dev(case)
    if entry == "closed":
        r = ev.cost_residual(B, N, *args, case["dt"], w_qd=case["w_qd"], w_tau=case["w_tau"], tau0=case["tau0"], alpha=case["alpha"],
                             tau_floor=case["tau_floor"], f_max=case["f_max"], out=out)
    else:
        r = ev.cost_residual_table(B, N, *args, torch.from_numpy(np.ascontiguousarray(case["table"])).cuda(), w_qd=case["w_qd"], w_tau=case["w_tau"],
                                   f_max=case["f_max"], out=out, out_col0=out_col0)
    torch.cuda.synchronize()
    return r.cpu().numpy()


def _as_table(case):
    """the case with the closed-form schedule turned into the table the table entry reads (exactly -b_k <= tau <= b_k)"""
    c = dict(case)
    if c["table"] is None:
        c["table"] = np.ascontiguousarray(np.stack([-c["bounds"][:, None].repeat(c["n"], 1), c["bounds"][:, None].repeat(c["n"], 1)], -1))
    return c


def check_both(case, entries=("closed", "table"), scenarios=None):
    rows = {}
    for e in entries:
        c = case if e == "closed" else _as_table(case)
        got = run_entry(c, e)
        assert_rows(got, c, scenarios)
        rows[e] = got
    return rows


gpu = pytest.mark.gpu
ENTRIES = ["closed", "table"]
_TABLE = None


# ------------------------------------------------------------------------------------------------------------------------------
# GPU tests: both reduction entries
# ------------------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("N", [2, 7])
@pytest.mark.parametrize("n", list(MODELS))
def test_planted_defects(n, N, entry):
    c, where = planted_defects(n, N, with_table=(entry == "table"))
    if entry == "closed":
        c["alpha"], c["bounds"] = 0.0, f0_bounds(N, c["dt"], c["tau0"], 0.0, c["tau_floor"])  # bound = tau0 exactly: r1 bitwise
    got = run_entry(c, entry)
    assert_rows(got, c)
    for b in range(c["B"]):
        if not (b in where and where[b][2] < N - 1):
            assert got[1, b] == 0.0 and not np.signbit(got[1, b]), (b, where.get(b))
    # the mismatches at the last node changed nothing: the rows equal those of the unplanted states
    last = [b for b, (blk, i, k) in where.items() if k == N - 1]
    clean, _ = planted_defects(n, N, with_table=(entry == "table"), plant=False)
    clean_rows = run_entry(dict(clean, alpha=c["alpha"], bounds=c["bounds"]), entry)
    assert _same_bits(got[:, last], clean_rows[:, last])


@gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("n", [3, 16])
def test_single_node_has_no_defect(n, entry):
    c = _flat(_case(n, 1, 40, seed=11))
    rng = np.random.default_rng(4)
    for k in ("qn", "qdn", "fn"):  # x+ of the only node compares with nothing
        c[k] += rng.uniform(1.0, 2.0, c[k].shape)
    got = run_entry(c if entry == "closed" else _as_table(c), entry)
    assert np.all(got[1] == 0.0) and not np.signbit(got[1]).any()
    assert_rows(got, c if entry == "closed" else _as_table(c))


@gpu
@pytest.mark.parametrize("N", [1, 2, 100])
@pytest.mark.parametrize("B", [1, 31, 255, 256, 257, 1000])
def test_shapes(B, N):
    c = _flat(_case(6, N, B, seed=B * 7 + N, f_max=55.0))
    rng = np.random.default_rng(B + N)
    for k in ("qn", "qdn", "fn"):  # non-zero defects of varied size
        c[k] += rng.normal(0.0, 1e-3, c[k].shape) * (rng.random(c[k].shape) < 0.05)
    check_both(c, scenarios=_sample(c))


@gpu
@pytest.mark.parametrize("w", [(1.0, 0.0), (0.0, 1.0), (0.3, 7.0)])
@pytest.mark.parametrize("n", [6, 64])
def test_cost_weights(n, w):
    c = weights_case(n, w)
    rows = check_both(c)
    for got in rows.values():
        assert np.all(got[0] > 0.0)


@gpu
@pytest.mark.parametrize("n", [3, 6])
def test_f0_closed_form(n):
    c, KF = f0_case(n)
    got = run_entry(c, "closed")
    assert_rows(got, c)
    ulp = np.spacing(15.0)
    # at the first floor node the bound is tau_floor exactly: |tau| - bound is exact, so the row is too
    assert [float(x) for x in got[2, 1:6]] == [0.0, 0.0, 0.0, ulp, 2 * ulp]
    assert not np.signbit(got[2, 1:6]).any()
    assert got[3, 11] == 0.0 and not np.signbit(got[3, 11]) and got[3, 12] == np.spacing(61.0)
    assert np.all(got[3, [b for b in range(c["B"]) if b not in (11, 12)]] == 0.0)
    # large torques over the whole horizon: within the exp allowance of every node's bound
    big = _flat(_case(n, 20, 300, seed=9, tau_scale=70.0, f_max=61.0))
    assert_rows(run_entry(big, "closed"), big)


@gpu
@pytest.mark.parametrize("n", [3, 6, 16])
def test_table_bounds(n):
    c, _ = planted_defects(n, 7, with_table=True)
    assert_rows(run_entry(c, "table"), c)
    # an unbounded joint (+/-inf) gives +0.0 for finite torques; every joint unbounded: the row is +0.0
    u = dict(c, table=c["table"].copy())
    u["table"][:, :, 0], u["table"][:, :, 1] = -np.inf, np.inf
    got = run_entry(u, "table")
    assert np.all(got[2] == 0.0) and not np.signbit(got[2]).any()
    assert_rows(got, u)
    half = dict(c, table=c["table"].copy())
    half["table"][:, ::2, 0], half["table"][:, ::2, 1] = -np.inf, np.inf
    assert_rows(run_entry(half, "table"), half)


@gpu
@pytest.mark.parametrize("entry", ENTRIES)
def test_negative_zero_violations_keep_the_row_at_plus_zero(entry):
    """Violations of -0.0 (lb = -0.0 against tau = +0.0, f+ = -0.0 against f_max = +0.0) and below: the rows stay +0.0."""
    n, N, B = 6, 4, 8
    c = _case(n, N, B, seed=12, f_max=0.0, tau0=0.0, alpha=0.0, tau_floor=0.0)
    _view3(c, "tau")[:] = 0.0
    _view3(c, "fn")[:] = -0.0
    _view3(c, "fn")[:, :, 1::2] = -1.0
    c = _flat(c)
    if entry == "table":
        c["table"] = np.ascontiguousarray(np.stack([np.full((N, n), -0.0), np.full((N, n), 3.0)], axis=-1))
    got = run_entry(c, entry)
    assert np.all(got[2:] == 0.0) and not np.signbit(got[2:]).any()
    assert_rows(got, c)


@gpu
@pytest.mark.parametrize("n,N,B", [(16, 400, 33), (16, 800, 9), (64, 200, 5)])
def test_table_sizes_across_the_shared_memory_limits(n, N, B):
    """102,400 B needs the raised shared-memory limit; 204,800 B (n = 16, N = 800 and n = 64, N = 200) is the largest table
    accepted.  One node more is MPCF_ELIMIT and writes nothing."""
    import torch
    c = _flat(_case(n, N, B, seed=n + N))
    c["table"] = _random_table(n, N, seed=n)
    assert_rows(run_entry(c, "table"), c, scenarios=_sample(c))
    if 2 * n * N * 8 == SMEM_TABLE_MAX:
        over = _flat(_case(n, N + 1, 2, seed=1))
        over["table"] = _random_table(n, N + 1, seed=1)
        out = torch.full((4, 2), CANARY, dtype=torch.float64, device="cuda")
        with pytest.raises(ValueError, match="200 KB"):
            run_entry(over, "table", out=out)
        assert bool((out == CANARY).all())


@gpu
def test_table_small_after_large_and_large_after_small():
    """The shared-memory limit is raised once per device and kept: tables on either side of 48 KB in any order."""
    cs = []
    for N in (30, 800, 30, 400, 800):
        c = _flat(_case(16, N, 17, seed=N + 1))
        c["table"] = _random_table(16, N, seed=N)
        cs.append(c)
    for c in cs:
        assert_rows(run_entry(c, "table"), c, scenarios=[0, 8, 16])


@gpu
def test_table_writes_only_its_columns_of_the_send_buffer():
    import torch
    n = 6
    c = ld_out_case(n)
    B, col0, ld = c["B"], LD_OUT["col0"], LD_OUT["ld"]
    pool = torch.full((_carve(np.empty(0), [4 * ld])[2],), CANARY, dtype=torch.float64, device="cuda")
    (buf,), gaps, _ = _carve(pool, [4 * ld])
    got = run_entry(c, "table", out=buf.view(4, ld), out_col0=col0)
    rows = reduce_ref(c)
    assert_rows(got[:, col0:col0 + B], c)
    expect = write_ref(np.full(4 * ld, CANARY), got[:, col0:col0 + B], col0, ld)
    assert np.array_equal(buf.cpu().numpy(), expect)
    assert all(bool((pool[g] == CANARY).all()) for g in gaps)
    assert _same_bits(got[:, col0:col0 + B][1:], rows[1:])
    # the closed-form entry writes exactly its [4][B]
    (o2,), gaps2, _ = _carve(pool, [4 * B])
    pool.fill_(CANARY)
    closed = dict(c, table=None)
    got2 = run_entry(closed, "closed", out=o2.view(4, B))
    assert_rows(got2, closed)
    assert all(bool((pool[g] == CANARY).all()) for g in gaps2)


@gpu
@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("n", [6, 16])
def test_nan_reaches_exactly_the_rows_that_read_it(n, entry):
    clean_case = nan_case(n, "q", "first", entry == "table")
    _view3(clean_case, "q")[n // 2, 0, 4] = 0.5
    clean = run_entry(clean_case, entry)
    for (arr, node), rows in EXPECTED_NAN.items():
        c = nan_case(n, arr, node, entry == "table")
        got = run_entry(c, entry)
        assert_rows(got, c)
        assert [r for j, r in enumerate(ROWS) if np.isnan(got[j, 4])] == list(rows), (arr, node)
        assert _same_bits(np.delete(got, 4, axis=1), np.delete(clean, 4, axis=1)), (arr, node)
    c = _flat(_case(n, 5, 9, seed=3, f_max=45.0, alpha=0.0))
    if entry == "table":
        c = _as_table(c)
    _view3(c, "fn")[0, 4, 2] = np.inf
    got = run_entry(c, entry)
    assert got[3, 2] == np.inf
    assert_rows(got, c)


def _capi_call(entry, m, B, N, ptrs, out, ld_out=0, table=True):
    import torch
    from mpc_fatigue_b200 import _capi
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if entry == "closed":
        return _capi.lib.mpcf_cost_residual_batch(m.handle, B, N, *ptrs, 0.05, 1.0, 1e-2, 50.0, 2.0, 15.0, 80.0, out, s)
    tb = C.c_void_p(_TABLE.data_ptr()) if table else None
    return _capi.lib.mpcf_cost_residual_table_batch(m.handle, B, N, *ptrs, 1.0, 1e-2, tb, 80.0, out, ld_out, s)


@gpu
@pytest.mark.parametrize("entry", ENTRIES)
def test_reduction_arguments(entry):
    import torch
    from mpc_fatigue_b200 import _capi
    m = _model(6)
    c = _flat(_case(6, 3, 4, seed=1))
    d = _dev(c)
    ptrs = [C.c_void_p(t.data_ptr()) for t in d]
    global _TABLE
    _TABLE = torch.from_numpy(_random_table(6, 3, seed=1)).cuda()
    pool = torch.full((_carve(np.empty(0), [16])[2],), CANARY, dtype=torch.float64, device="cuda")
    (o,), gaps, _ = _carve(pool, [16])
    out = C.c_void_p(o.data_ptr())
    assert _capi_call(entry, m, -1, 3, ptrs, out) == _capi.EINVAL
    assert _capi_call(entry, m, 4, 0, ptrs, out) == _capi.EINVAL
    assert _capi_call(entry, m, 4, -2, ptrs, out) == _capi.EINVAL
    for j in range(7):
        p = list(ptrs)
        p[j] = None
        assert _capi_call(entry, m, 4, 3, p, out) == _capi.EINVAL, j
    assert _capi_call(entry, m, 4, 3, ptrs, None) == _capi.EINVAL
    if entry == "table":
        assert _capi_call(entry, m, 4, 3, ptrs, out, ld_out=3) == _capi.EINVAL  # ld_out < B
        assert _capi_call(entry, m, 4, 3, ptrs, out, table=False) == _capi.EINVAL
        assert _capi_call(entry, m, 4, 3, ptrs, out, ld_out=4) == _capi.OK  # the same call with valid arguments runs
        torch.cuda.synchronize()
        assert bool((o[:16] != CANARY).all())
        pool.fill_(CANARY)
    assert _capi_call(entry, m, 0, 3, ptrs, out) == _capi.OK
    assert _capi_call(entry, m, 0, 3, [None] * 7, None, table=False) == _capi.OK
    torch.cuda.synchronize()
    assert bool((pool == CANARY).all())


@gpu
def test_nan_torque_through_the_jacobian_and_the_reduction():
    """A NaN torque in one unit of a pilz6 batch: that scenario's rows are NaN as the reference says, and every other unit's
    states, Jacobian planes and rows are bit-identical to the clean run, including the units that share the NaN unit's 32-unit
    workspace tile.  Then the same batch through HostStepPipeline."""
    import torch
    from mpc_fatigue_b200.ocp import f0_bound_table
    from mpc_fatigue_b200.pipeline import HostStepPipeline
    from mpc_fatigue_b200.synth import synth_batch
    n, B, N, dt = 6, 67, 5, 0.02
    m, ev = _model(6), _ev(6)
    lim = {k: m.export(k) for k in ("q_lo", "q_hi", "v_max", "tau_max")}
    q, qd, tau, f = synth_batch(lim, 0, B, N, seed=21, device="cuda")
    bs, ks = 13, 2
    us = ks * B + bs
    tau_nan = tau.clone()
    tau_nan[3, us] = float("nan")
    tb = torch.from_numpy(f0_bound_table(N, n, dt, 50.0, 2.0, 15.0)).cuda()
    runs = []
    for t in (tau, tau_nan):
        qn, qdn, fn, jac = ev.step_rk4_jvp(q, qd, t, f, dt)
        red = ev.cost_residual_table(B, N, q, qd, f, t, qn, qdn, fn, tb, f_max=60.0)
        torch.cuda.synchronize()
        runs.append([x.cpu().numpy() for x in (qn, qdn, fn, jac, red)])
    (cq, cqd, cf, cj, cr), (nq, nqd, nf, nj, nr) = runs
    others = np.ones(B * N, dtype=bool)
    others[us] = False
    assert us // 32 == (us - 1) // 32 == (us + 1) // 32  # neighbours in the same workspace tile are among the units compared
    for a, b in ((cq, nq), (cqd, nqd), (cf, nf)):
        assert _same_bits(a[:, others], b[:, others])
    assert _same_bits(cj[..., others], nj[..., others])
    assert np.isnan(nq[:, us]).any() or np.isnan(nqd[:, us]).any()
    case = dict(n=n, N=N, B=B, w_qd=1.0, w_tau=1e-2, f_max=60.0, table=f0_bound_table(N, n, dt, 50.0, 2.0, 15.0), alpha=2.0)
    h = lambda x: x.cpu().numpy()
    case.update(q=h(q), qd=h(qd), f=h(f), tau=h(tau_nan), qn=nq, qdn=nqd, fn=nf)
    ref = reduce_ref(case)
    assert _same_bits(nr[1:], ref[1:]) and np.isnan(nr[0, bs]) and np.isnan(nr[:, bs]).all()
    keep = np.arange(B) != bs
    assert _same_bits(nr[:, keep], cr[:, keep])
    # the host-facing pipeline: the same rows come back (chunks of 20 scenarios; the NaN one in the first)
    pipe = HostStepPipeline(m, "cuda:0", chunk_units=20 * N)
    host = [x.cpu().pin_memory() for x in (q, qd, tau_nan, f)]
    got = {}
    pipe.run(*host, dt, B, N, consume=lambda v, b0, b1: got.__setitem__((b0, b1), v.clone()))
    direct = ev.cost_residual(B, N, q, qd, f, tau_nan, *[torch.from_numpy(x).cuda() for x in (nq, nqd, nf)], dt)
    assert _same_bits(pipe.h_red.numpy(), direct.cpu().numpy())
    full = np.concatenate([nq, nqd, nf, nj.reshape(-1, B * N)]).reshape(-1, N, B)
    for (b0, b1), v in got.items():
        assert _same_bits(v.numpy(), full[:, :, b0:b1])


# ------------------------------------------------------------------------------------------------------------------------------
# GPU tests: mpcf_gather_planes (reference: src[map] by torch indexing, bit for bit)
# ------------------------------------------------------------------------------------------------------------------------------
def _gather(src, ld_src, pmap, nplanes, U, dst):
    import torch
    from mpc_fatigue_b200 import _capi
    p = lambda t: None if t is None else C.c_void_p(t if isinstance(t, int) else t.data_ptr())
    return _capi.lib.mpcf_gather_planes(p(src), ld_src, p(pmap), nplanes, U, p(dst), C.c_void_p(torch.cuda.current_stream().cuda_stream))


@gpu
@pytest.mark.parametrize("pad", [0, 1, 2])
@pytest.mark.parametrize("U", [1, 2, 3, 511, 512, 513, 303105, 606210])
def test_gather_planes(U, pad):
    """U = 303,105 (odd: scalar path) and 606,210 (even: 16-byte path at pad 0) make the grid-stride loop wrap: the grid is at
    most 592 blocks of 256 threads."""
    import torch
    from mpc_fatigue_b200 import _capi
    ld = U + pad
    nsrc = 5
    src = torch.arange(nsrc * ld, dtype=torch.float64, device="cuda") * 1.25 - 3.0
    maps = {"identity": list(range(nsrc)), "reversed": list(range(nsrc))[::-1], "repeated": [3, 0, 3, 3, 4, 0, 1], "single": [2]}
    for name, mp in maps.items():
        k = len(mp)
        pool = torch.full((_carve(np.empty(0), [k * U])[2],), CANARY, dtype=torch.float64, device="cuda")
        (dst,), gaps, _ = _carve(pool, [k * U])
        pm = torch.tensor(mp, dtype=torch.int32, device="cuda")
        assert _gather(src, ld, pm, k, U, dst) == _capi.OK, _capi.last_error()
        torch.cuda.synchronize()
        ref = src.view(-1)[:nsrc * ld].view(nsrc, ld)[:, :U][pm.long()].reshape(-1)
        assert torch.equal(dst.view(torch.int64), ref.view(torch.int64)), (U, pad, name)
        assert all(bool((pool[g] == CANARY).all()) for g in gaps), (U, pad, name)


@gpu
def test_gather_planes_limits_and_arguments():
    import torch
    from mpc_fatigue_b200 import _capi
    U = 4
    src = torch.arange(3 * U, dtype=torch.float64, device="cuda")
    pool = torch.full((_carve(np.empty(0), [65535 * U + 16])[2],), CANARY, dtype=torch.float64, device="cuda")
    (dst,), gaps, _ = _carve(pool, [65535 * U + 16])
    pm = torch.arange(65536, dtype=torch.int32, device="cuda") % 3
    # nothing to do: OK, nothing written
    assert _gather(src, U, pm, 0, U, dst) == _capi.OK
    assert _gather(src, U, pm, 3, 0, dst) == _capi.OK
    torch.cuda.synchronize()
    assert bool((pool == CANARY).all())
    # 65,535 planes (the grid's y limit) are accepted; 65,536 are MPCF_ELIMIT
    assert _gather(src, U, pm, 65535, U, dst) == _capi.OK, _capi.last_error()
    torch.cuda.synchronize()
    assert torch.equal(dst[:65535 * U], src.view(3, U)[pm[:65535].long()].reshape(-1))
    assert bool((dst[65535 * U:] == CANARY).all()) and all(bool((pool[g] == CANARY).all()) for g in gaps)
    pool.fill_(CANARY)
    assert _gather(src, U, pm, 65536, U, dst) == _capi.ELIMIT
    # misaligned src or dst, ld_src < U, negative sizes, NULL arrays: MPCF_EINVAL, nothing written
    assert _gather(src.data_ptr() + 8, U, pm, 2, U, dst) == _capi.EINVAL
    assert _gather(src, U, pm, 2, U, dst.data_ptr() + 8) == _capi.EINVAL
    assert _gather(src, U - 1, pm, 2, U, dst) == _capi.EINVAL
    assert _gather(src, U, pm, -1, U, dst) == _capi.EINVAL
    assert _gather(src, U, pm, 2, -1, dst) == _capi.EINVAL
    assert _gather(src, U, None, 2, U, dst) == _capi.EINVAL
    assert _gather(None, U, pm, 2, U, dst) == _capi.EINVAL
    assert _gather(src, U, pm, 2, U, None) == _capi.EINVAL
    torch.cuda.synchronize()
    assert bool((pool == CANARY).all())
