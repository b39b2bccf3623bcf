"""Top-k ranking against inputs built to defeat the tensor-core screening.

ibl_l2dist_topk screens every database row on the tensor cores and re-scores only the candidates it keeps in exact
fp32.  Its answer is the exact fp32 ranking only if a guard notices every query for which a row that was not kept
could still belong to the top-k.  The inputs below make one row T lose to the screening: its representation
error points the same way in every coordinate, so its screened distance is far larger than its exact one, and enough
decoys sit in between to push it out of the candidate set.

The CPU part emulates the two screening representations (the power-of-two-scaled fp16 plane of rows_f16_kernel and the
bf16 hi/lo planes of planes_sqnorm_kernel), uses them to build the inputs, checks that the inputs mean what they
should, and checks the formula of the guard's bound (screen_guard_bound in common.cuh) against the emulated
screening.  The GPU part checks each path of the kernels against an fp64 ranking (ties to the lowest index)."""
import os

import numpy as np
import pytest
import torch

# ---------------------------------------------------------------------------------------------
# emulation of the screening representations
# ---------------------------------------------------------------------------------------------


def f16_plane(x):
    """rows_f16_kernel: x = plane * 2^e per row, row max scaled into [0.5, 1), fp16 round-to-nearest-even.
    Returns the represented values (fp64)."""
    x = np.asarray(x, dtype=np.float32)
    m = np.abs(x).max(axis=1)
    _, e = np.frexp(m)
    e = np.where(m > 0, e, 0).astype(np.int32)
    inv = np.ldexp(np.float32(1), -e).astype(np.float32)[:, None]
    plane = (x * inv).astype(np.float16)
    return np.ldexp(plane.astype(np.float64), e[:, None])


def bf16_rn(x):
    """fp32 -> bf16 round-to-nearest-even on the bit pattern (finite inputs); returned as fp32."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def bf16_planes(x):
    """planes_sqnorm_kernel: hi = bf16(x), lo = bf16(x - hi) (x - hi is exact in fp32).  fp64 hi, lo."""
    x = np.asarray(x, dtype=np.float32)
    hi = bf16_rn(x)
    lo = bf16_rn((x - hi).astype(np.float32))
    return hi.astype(np.float64), lo.astype(np.float64)


def sqnorm(x):
    return (np.asarray(x, dtype=np.float64) ** 2).sum(axis=1)


def screened(q, db, path):
    """Screened distances [m, n]: exact |q|^2 + |d|^2 minus twice the dot product the tensor cores see (fp64 sums)."""
    if path == "f16":
        dot = f16_plane(q) @ f16_plane(db).T
    else:                                          # bf16x3: hi.hi + hi.lo + lo.hi, lo.lo dropped
        qh, ql = bf16_planes(q)
        dh, dl = bf16_planes(db)
        dot = qh @ dh.T + qh @ dl.T + ql @ dh.T
    return sqnorm(q)[:, None] + sqnorm(db)[None, :] - 2 * dot


def exact64(q, db):
    q, db = np.asarray(q, dtype=np.float64), np.asarray(db, dtype=np.float64)
    return ((q[:, None, :] - db[None, :, :]) ** 2).sum(-1) if q.shape[0] * db.shape[0] * q.shape[1] < 2 ** 24 else \
        sqnorm(q)[:, None] + sqnorm(db)[None, :] - 2 * (q @ db.T)


def rep_err(x, path):
    x64 = np.asarray(x, dtype=np.float64)
    if path == "f16":
        return np.linalg.norm(x64 - f16_plane(x), axis=1)
    hi, lo = bf16_planes(x)
    return np.linalg.norm(x64 - hi - lo, axis=1)


def new_bound(q, db, path):
    """screen_guard_bound (common.cuh) per query, with the maxima over the database rows."""
    d = q.shape[1]
    an, qe = sqnorm(q), rep_err(q, path)
    dmax_sq, dmax_err = sqnorm(db).max(), rep_err(db, path).max()
    n_mma = d // 16 if path == "f16" else 3 * (d // 16)
    lolo = 0.0 if path == "f16" else 1.5411377e-5
    nq, nd = np.sqrt(an) * 1.001, np.sqrt(dmax_sq) * 1.001
    rep = qe * nd + nq * dmax_err + qe * dmax_err
    rel = lolo + n_mma * 2.3841858e-7 * 1.01 + (d // 32 + 8) * 5.9604645e-8
    return 1.001 * (2 * (rep + rel * nq * nd) + 4.7683716e-7 * (an + dmax_sq))


def old_bound_f16(q, db):
    """The guard this project used before: 8 sigma of a random fp16 rounding model from the rows' 4-norms, plus a
    term for fp16 subnormals."""
    q, db = np.asarray(q, dtype=np.float64), np.asarray(db, dtype=np.float64)
    c = 8 * 2 * 1.41421356 * 0.41 * 2.0 ** -11
    n4 = lambda x: (x ** 4).sum(axis=1) ** 0.25
    sub = 2 * 2.0 ** -24 * np.sqrt(q.shape[1]) * (np.abs(db).max() * np.sqrt(sqnorm(q)) +
                                                  np.abs(q).max(axis=1) * np.sqrt(sqnorm(db).max()))
    return c * n4(q) * n4(db).max() + sub


def fp32_err(q, db):
    """Size of the fp32 rounding of |q|^2 + |d|^2 - 2 q.d: a few units of the last place of |q|^2 + |d|^2."""
    return 2.0 ** -23 * (sqnorm(q)[:, None] + sqnorm(db)[None, :])


def kept_count(path, k):
    return 16 if k <= 12 else min(k + 8, 128)


# ---------------------------------------------------------------------------------------------
# the adversarial inputs
# ---------------------------------------------------------------------------------------------
# Per path: the dimension, the query value (every coordinate), T's value (every coordinate) and the decoy levels.
# A decoy of level a is q +/- a * step in `count` coordinates, half of them +: exactly representable in both
# representations, so it screens at its exact distance.  Levels: N (k - 1 copies, in the true top-k next to T),
# B1 (2 copies, the first rows after the true top-k) and B2 (enough copies to fill the candidate set).  The fp16 levels
# are chosen so that B2 - B1 exceeds the old statistical bound: without T, that guard saw nothing wrong.
SPEC = {
    # fp16: q = 2^-5 (0.5 after scaling), T = (0.5 + 0.49 * 2^-11) / 16 loses 0.49 ulp in every coordinate
    "f16": dict(D=1024, qv=2.0 ** -5, tv=(0.5 + 0.49 * 2.0 ** -11) / 16, step=2.0 ** -15, count=1024,
                levels=dict(N=4, B1=16, B2=28)),
    # bf16x3: q = 2^-6, T = 2^-6 + j 2^-29: hi = 2^-6, the lo plane drops 63 units of 2^-29 in every coordinate
    "bf16": dict(D=4096, qv=2.0 ** -6, tv=2.0 ** -6 + (2 ** 15 - 2 ** 7 + 2 ** 6 - 1) * 2.0 ** -29, step=2.0 ** -12,
                 levels=dict(N=100, B1=300, B2=420)),        # count: decoy coordinates (distance = count * step^2)
}


def decoy(spec, level, rng):
    D, qv, step = spec["D"], spec["qv"], spec["step"]
    row = np.full(D, qv, dtype=np.float64)
    if "count" in spec:                              # fp16: every coordinate moves by level * step
        idx, amp = rng.permutation(D), level * step
    else:                                            # bf16: `level` coordinates move by one step
        idx, amp = rng.permutation(D)[:level], step
    sign = np.ones(len(idx))
    sign[len(idx) // 2:] = -1
    row[idx] += sign * amp
    return row.astype(np.float32)


def build(path, k, n_rand=1200, pad=5, seed=0):
    """Returns (q [1, D], db [n, D] fp32 with `pad` padding rows at the end that are copies of q, n_valid, t_row)."""
    spec = SPEC[path]
    rng = np.random.default_rng(seed)
    D = spec["D"]
    q = np.full((1, D), spec["qv"], dtype=np.float32)
    t = np.full(D, spec["tv"], dtype=np.float32)
    kc = kept_count(path, k)
    lv = spec["levels"]
    # copies of one row per level: equal distances come from identical rows, which every evaluation ties
    rows = [t] + [decoy(spec, lv["N"], rng)] * (k - 1) + [decoy(spec, lv["B1"], rng)] * 2 + [decoy(spec, lv["B2"], rng)] * kc
    rand = rng.standard_normal((n_rand, D)).astype(np.float32)
    rand /= np.linalg.norm(rand, axis=1, keepdims=True)
    n_valid = n_rand + len(rows)
    # spread the special rows over the database: different 256-row tiles and work items; T in the last tile
    pos = np.sort(rng.choice(np.arange(0, n_valid - 256), size=len(rows) - 1, replace=False))
    pos = np.concatenate([[n_valid - 7], pos])
    db = np.empty((n_valid + pad, D), dtype=np.float32)
    free = np.setdiff1d(np.arange(n_valid), pos)
    db[pos] = np.stack(rows)
    db[free] = rand
    db[n_valid:] = q                                 # padding: would rank first if it leaked in
    return q, db, n_valid, int(pos[0])


def fp64_topk(q, db, k):
    d = exact64(q, db)
    idx = np.argsort(d, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(d, idx, axis=1), idx


CASES = [("f16", 1), ("f16", 10), ("f16", 12), ("bf16", 1), ("bf16", 10), ("bf16", 12), ("bf16", 20), ("bf16", 120)]


# ---------------------------------------------------------------------------------------------
# CPU: the inputs mean what they should, and the bound holds
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path,k", CASES)
def test_crafted_inputs_defeat_the_screening(path, k):
    q, db, n_valid, t = build(path, k)
    dbv = db[:n_valid]
    ex = exact64(q, dbv)[0]
    sc = screened(q, dbv, path)[0]
    order = np.argsort(ex, kind="stable")
    # T is in the true top-k ...
    assert t in order[:k]
    # ... but not among the candidates the path keeps
    kc = kept_count(path, k)
    kept = np.argsort(sc, kind="stable")[:kc]
    assert t not in kept
    assert sc[t] > np.sort(sc)[kc - 1]
    # the true top-k is unambiguous at fp32 resolution: distinct distances are 10x the fp32 error apart, and equal
    # ones belong to identical rows (so any fp32 evaluation ties them too, broken by the index)
    err = fp32_err(q, dbv)[0]
    top = order[:k + 1]
    for a, b in zip(top[:-1], top[1:]):
        if ex[a] == ex[b]:
            assert np.array_equal(dbv[a], dbv[b])
        else:
            assert ex[b] - ex[a] >= 10 * max(err[a], err[b]), (a, b, ex[a], ex[b])
    # the guard: with T gone, the k-th exact distance of the kept candidates and their largest screened distance
    e_k = np.sort(ex[kept])[k - 1]
    s_kc = sc[kept].max()
    assert not (s_kc - new_bound(q, dbv, path)[0] > e_k), "the bound of screen_guard_bound must flag this query"
    if path == "f16":
        assert s_kc - old_bound_f16(q, dbv)[0] > e_k, "the old statistical guard did not flag this query"


@pytest.mark.parametrize("path", ["f16", "bf16"])
@pytest.mark.parametrize("D", [64, 1024, 4096, 32768])
def test_screening_bound_covers_every_pair(path, D):
    """|screened - exact| <= B for random unit rows, sparse rows, rows with fp16 subnormals after scaling and the
    crafted rows (the bound's accumulator term is not emulated here: the emulated dot products are exact)."""
    rng = np.random.default_rng(D)
    n = 64 if D == 32768 else 256
    rand = rng.standard_normal((n, D)).astype(np.float32)
    rand /= np.linalg.norm(rand, axis=1, keepdims=True)
    sparse = np.zeros((n // 4, D), dtype=np.float32)
    for r in range(n // 4):
        j = rng.choice(D, size=max(2, D // 64), replace=False)
        sparse[r, j] = rng.standard_normal(len(j))
    spread = (rng.standard_normal((n // 4, D)) * np.exp(rng.uniform(-25, 0, (n // 4, D)))).astype(np.float32)
    spread[:, 0] = 1.0                               # row max 1: most coordinates are fp16 subnormals after scaling
    crafted = []
    for p in ("f16", "bf16"):
        spec = SPEC[p]
        t = np.resize(np.float32(spec["tv"]), D)
        crafted += [t, np.resize(np.float32(spec["qv"]), D), decoy(dict(spec, D=D), spec["levels"]["B2"] % D, rng)]
    db = np.concatenate([rand, sparse, spread, np.stack(crafted).astype(np.float32)])
    q = np.concatenate([db[::7], (rand[:8] + 0.01 * rng.standard_normal((8, D))).astype(np.float32)])
    gap = np.abs(screened(q, db, path) - exact64(q, db))
    bound = new_bound(q, db, path)
    assert (gap <= bound[:, None]).all(), float((gap / bound[:, None]).max())


def test_bound_rarely_trips_on_descriptor_like_data():
    """Emulated on the benchmark's kind of data (unit 4096-d rows, planted positives, 10k database rows): the bound
    is ~1e-3 for the fp16 plane and ~4e-4 for bf16x3, the k-th-to-16th gap is usually several times larger, and the
    fraction of queries sent to the exact brute force stays small (0.2 % fp16, none bf16x3 on this subset)."""
    from openibl_b200 import synth
    q, db, _ = synth.make_gallery(10000, 500, 4096)
    q, db = q.numpy(), db.numpy()
    for path, limit in (("f16", 5), ("bf16", 0)):
        sc = screened(q, db, path)
        ex = exact64(q, db)
        kept = np.argsort(sc, axis=1, kind="stable")[:, :16]
        e_k = np.sort(np.take_along_axis(ex, kept, axis=1), axis=1)[:, 9]
        s16 = np.take_along_axis(sc, kept, axis=1).max(axis=1)
        flagged = int((~(s16 - new_bound(q, db, path) > e_k)).sum())
        assert flagged <= limit, (path, flagged)


# ---------------------------------------------------------------------------------------------
# GPU: every path of ibl_l2dist_topk against the fp64 ranking
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    from openibl_b200.engine import Engine
    return Engine.get(0)


def taken_path(m, k):
    """The screening ibl_l2dist_topk applies (engine.cu): the single fp16 pass for m > 128, k <= 12 unless
    IBL_DIST_SCREEN=3, else bf16x3."""
    return "f16" if (m > 128 and k <= 12 and os.environ.get("IBL_DIST_SCREEN", "1") != "3") else "bf16"


GPU_CASES = [("f16", 1, 256), ("f16", 10, 256), ("f16", 12, 256),       # single pass (m > 128)
             ("bf16", 1, 100), ("bf16", 10, 100), ("bf16", 12, 100),    # bf16x3 top-16 (m <= 128)
             ("bf16", 20, 64), ("bf16", 120, 64)]                        # bf16x3 dense tiles (k > 12)


@pytest.mark.gpu
@pytest.mark.parametrize("path,k,m", GPU_CASES, ids=[f"{p}-k{k}-m{m}" for p, k, m in GPU_CASES])
def test_topk_ranks_crafted_rows_like_fp64(eng, path, k, m):
    q1, db, n_valid, t = build(path, k)
    q = np.repeat(q1, m, axis=0)
    base = 1000
    wd, wi = fp64_topk(q1, db[:n_valid], k)
    qd, dbd = torch.from_numpy(q).cuda(), torch.from_numpy(db).cuda()
    dk, ik = eng.l2dist_topk(qd, dbd, k, idx_base=base, n_valid=n_valid)
    flagged = eng.dist_flagged()
    got_i = ik.cpu().numpy() - base
    assert (got_i == wi).all(), (got_i[0].tolist(), wi[0].tolist(), t)
    assert np.abs(dk.cpu().numpy() - wd).max() <= 2e-6
    run = taken_path(m, k)
    sc = screened(q1, db[:n_valid], run)[0]
    if np.argsort(sc, kind="stable").tolist().index(t) >= kept_count(run, k):   # the screening loses T on this path
        assert flagged > 0
    # control: the CUDA-core path computes every distance in fp32 without screening and finds the same rows (T among
    # them); its summation order rounds T's distance differently, so only the set of rows is compared
    eng.set_gemm_mode(0)
    try:
        dk0, ik0 = eng.l2dist_topk(qd, dbd, k, idx_base=base, n_valid=n_valid)
        assert eng.dist_flagged() == -1
    finally:
        eng.set_gemm_mode(1)
    assert (np.sort(ik0.cpu().numpy() - base, axis=1) == np.sort(wi, axis=1)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k,m", [(10, 256), (10, 100), (20, 64)])
def test_topk_padding_rows_never_win(eng, k, m):
    """Rows at and beyond n_valid are exact copies of the queries: they would rank first if any path read them."""
    gen = torch.Generator().manual_seed(11)
    n, n_valid, d = 1500, 1300, 512
    db = torch.nn.functional.normalize(torch.randn(n, d, generator=gen), dim=1)
    q = torch.nn.functional.normalize(torch.randn(m, d, generator=gen), dim=1)
    db[n_valid:n_valid + m] = q[: n - n_valid]
    wd, wi = fp64_topk(q.numpy(), db[:n_valid].numpy(), k)
    dk, ik = eng.l2dist_topk(q.cuda(), db.cuda(), k, idx_base=7, n_valid=n_valid)
    assert np.array_equal(ik.cpu().numpy() - 7, wi)
    assert np.abs(dk.cpu().numpy() - wd).max() <= 2e-6


@pytest.mark.gpu
def test_dist_flagged_reports_the_last_call(eng):
    """The flag count belongs to the last call, whichever path it took: a flagged call with 256 queries (single pass)
    followed by a bf16x3 call with 50 queries on clean data reads 0, and a CUDA-core call reads -1."""
    from openibl_b200 import synth
    q1, db, n_valid, _ = build(taken_path(256, 10), 10)
    dbd = torch.from_numpy(db).cuda()
    q = torch.from_numpy(np.repeat(q1, 256, axis=0)).cuda()
    eng.l2dist_topk(q, dbd, 10, n_valid=n_valid)
    assert eng.dist_flagged() > 0
    q2, db2, _ = synth.make_gallery(2000, 50, db.shape[1])
    eng.l2dist_topk(q2.cuda(), db2.cuda(), 10)
    assert eng.dist_flagged() == 0
    eng.set_gemm_mode(0)
    try:
        eng.l2dist_topk(q2.cuda(), db2.cuda(), 10)
        assert eng.dist_flagged() == -1
    finally:
        eng.set_gemm_mode(1)
