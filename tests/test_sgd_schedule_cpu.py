"""The schedule reference of the stratified SGD kernel (tests/sgd_schedule.py), without a GPU.

* Its own invariants: a permutation; cells of a stratum disjoint in users and items; waves without a repeated row;
  the tail only where the greedy colouring ran out of colours; every cell pairs the user block with the item block
  that the kernel's ring traversal (csrc/sgd.cu, dsgd_body) holds in that stratum.
* A literal per-rating transcription of dsgd_key_kernel and dsgd_color_kernel gives the same order.
* Discrimination: schedules that a subtly wrong kernel would apply (strata swapped, colour order ignored, tail
  reversed, a rating lost, the wrong cluster size in the key) move the oracle's factors by at least MARGIN x ATOL,
  the tolerance of the element-wise GPU comparison (tests/test_gpu_sgd_schedule.py).  For SVD++ the same order
  mutants and the y_j-side ones (y_j frozen, the decay not integrated, 1/|I_u|, z_u not advanced, c_j counting
  raters, a chunk count off by one, g_u kept across chunks) move the relaxation by at least MARGIN x ATOL.
* The SVD++ relaxation (oracle.svdpp_relaxed_sgd) equals its pseudo-code transcribed in numpy, and the reference
  (oracle.svdpp_sgd) where the two must agree: on a conflict-free input, and with lr_yj = 0 in the same order.
* The planner's shared-memory arithmetic: the item counts at which capping B at the co-resident clusters used to
  leave a clustered plan without item buffers.
"""
import numpy as np
import pytest

import oracle
import sgd_schedule as S


def _random_case(seed, P, C, dense=0):
    rng = np.random.default_rng(seed)
    B = C * int(rng.integers(1, 4))
    nu, ni = int(rng.integers(max(P, 40), 300)), int(rng.integers(max(P, 30), 200))
    if dense:
        ni = 500                                                 # 300 items per dense user
    n = int(rng.integers(max(nu, ni) + 50, min(nu * ni // 3, 6000)))
    u, i, r, _, _ = S.draw(nu, ni, n, seed, dense_users=dense, dense_share=0.6)
    return u, i, r, B


@pytest.mark.parametrize("P", (1, 2, 3, 4))
@pytest.mark.parametrize("C", (1, 2, 16))
def test_reference_invariants(P, C):
    for seed in range(3):
        u, i, r, B = _random_case(100 * P + C + seed, P, C, dense=3 if seed == 2 else 0)
        sc = S.schedule(u, i, B, C, P)
        o, col = sc["order"], sc["colour"]
        assert np.array_equal(np.sort(o), np.arange(len(u)))
        # the emission is sorted by (stratum, rank, user block, colour)
        key = np.stack((sc["stratum"][o], sc["rank"][o], sc["ub"][o], col[o]))
        assert (np.diff(key[0]) >= 0).all()
        for a in range(1, 4):
            same = (key[:a, 1:] == key[:a, :-1]).all(axis=0)
            assert (np.diff(key[a])[same] >= 0).all()
        # the item block of a cell is the one the kernel's two-level ring holds in that stratum
        K = B // C
        ub, s = sc["ub"], sc["stratum"]
        Sx, sl = s // B, s % B
        T, t = sl // C, sl % C
        D = (ub // C + T) % K
        j = (ub % C + t) % C
        assert np.array_equal((i.astype(np.int64) // P) % B, D * C + j)
        assert np.array_equal(i % P, (sc["rank"] + Sx) % P)           # the rank's item super-block in sub-epoch S
        assert np.array_equal(sc["rank"], u % P)
        # a stratum's cells (over all ranks) share no user and no item
        for st in np.unique(s):
            m = s == st
            for rows in (u[m], i[m]):
                cells_per_row = {}
                for x, c in zip(rows.tolist(), sc["cell"][m].tolist()):
                    assert cells_per_row.setdefault(x, c) == c
        # a wave repeats no row; the tail only when the colours ran out, first free colour otherwise
        n_tail = 0
        for c in np.unique(sc["cell"]):
            ks = np.nonzero(sc["cell"] == c)[0]                    # input order
            seen_u, seen_i = {}, {}
            for k in ks.tolist():
                taken = seen_u.get(u[k], set()) | seen_i.get(i[k], set())
                if col[k] == S.TAIL:
                    n_tail += 1
                    assert taken >= set(range(S.TAIL))
                else:
                    assert col[k] not in taken and all(x in taken for x in range(col[k]))
                    seen_u.setdefault(u[k], set()).add(col[k])
                    seen_i.setdefault(i[k], set()).add(col[k])
        if seed == 2 and P * B <= 4:
            assert n_tail > 0, "the dense users of this case reach the tail"


def _literal_order(u, i, B, C, P):
    """dsgd_key_kernel + stable radix sort + dsgd_color_kernel, one rating at a time, for every rank; then the
    cells in the order the ranks' kernels apply them (stratum, rank, user block)."""
    n_cells = P * B * B
    cells = {}
    for rank in range(P):
        keys = []
        for k in range(len(u)):
            uu, ii = int(u[k]), int(i[k])
            if uu % P != rank:
                keys.append(n_cells)
                continue
            Sx = ((ii % P) - rank + P) % P
            ub, ibk = (uu // P) % B, (ii // P) % B
            K = B // C
            Cl, c, D, j = ub // C, ub % C, ibk // C, ibk % C
            T, t = (D - Cl + K) % K, (j - c + C) % C
            keys.append((Sx * B + T * C + t) * B + ub)
        val = sorted(range(len(u)), key=lambda k: keys[k])      # Python's sort is stable
        for k in val:
            if keys[k] < n_cells:
                cells.setdefault((rank, keys[k]), []).append(k)
    out = []
    for (rank, cell) in sorted(cells, key=lambda rc: (rc[1] // B, rc[0], rc[1] % B)):
        ks = cells[(rank, cell)]
        masks = {}
        colours = []
        for k in ks:
            ul, il = ("u", (int(u[k]) // P) // B), ("i", (int(i[k]) // P) // B)
            used = masks.get(ul, 0) | masks.get(il, 0)
            inv = ~used & ((1 << 64) - 1)
            c = (inv & -inv).bit_length() - 1 if inv else -1      # __ffsll(~used) - 1
            if c < 0 or c >= S.NW - 1:
                c = S.NW - 1
            else:
                masks[ul] = masks.get(ul, 0) | (1 << c)
                masks[il] = masks.get(il, 0) | (1 << c)
            colours.append(c)
        hist = [0] * (S.NW + 1)                                  # counting sort by colour (stable)
        for c in colours:
            hist[c + 1] += 1
        for c in range(S.NW):
            hist[c + 1] += hist[c]
        placed = [None] * len(ks)
        for k, c in zip(ks, colours):
            placed[hist[c]] = k
            hist[c] += 1
        out.extend(placed)
    return np.array(out)


@pytest.mark.parametrize("P,C", [(1, 1), (1, 2), (1, 16), (2, 2), (3, 1), (4, 2)])
def test_literal_transcription(P, C):
    u, i, r, B = _random_case(7 + P * 10 + C, P, C, dense=2)
    assert np.array_equal(_literal_order(u, i, B, C, P), S.schedule_order(u, i, B, C, P))


# --------------------------------------------------------------------------------------------------------------
# discrimination
def _mutants(u, i, B, C, P):
    sc = S.schedule(u, i, B, C, P)
    o = sc["order"]
    out = {}
    s = sc["stratum"][o]
    a = B // 2                                                   # strata a and a + 1 swapped
    out["adjacent strata swapped"] = np.concatenate((o[s < a], o[s == a + 1], o[s == a], o[s > a + 1]))
    pos = np.arange(len(u))
    out["input order inside a cell"] = np.lexsort((pos, sc["ub"], sc["rank"], sc["stratum"]))
    tail = sc["colour"][o] == S.TAIL
    if tail.any():
        m = o.copy()
        cell = sc["cell"][o]
        for c in np.unique(cell[tail]):
            w = np.nonzero(tail & (cell == c))[0]
            m[w] = m[w[::-1]]
        out["tail reversed"] = m
    out["one rating dropped"] = np.delete(o, len(o) // 3)
    if C > 1:
        out["C = 1 key formula"] = S.schedule_order(u, i, B, 1, P)
    return o, out


# (shape, B, C): the reduced ml-1M-like shape of the GPU tests at its default layout (7 clusters of 16 CTAs), and
# the dense-user shape at SB2_DSGD_BLOCKS=4 (two clusters of 2, colour tail, cells beyond the staged records)
DISCRIMINATION = {
    "default": (dict(n_users=3000, n_items=2000, n=400_000, seed=1), 112, 16, 20),
    "dense": (dict(n_users=300, n_items=2000, n=300_000, seed=2, dense_users=40, dense_share=0.6), 4, 2, 20),
}


def _pp_mutants():
    """SVD++ relaxations a subtly wrong kernel or host would apply: name -> (chunks of the exact schedule, chunks of
    the mutant, variant bits of oracle.svdpp_relaxed_sgd)."""
    return {
        "y_j frozen": (1, 1, oracle.PP_Y_FROZEN),
        "decay not integrated": (1, 1, oracle.PP_NO_DECAY),
        "1/|I_u|": (1, 1, oracle.PP_ISQ_INV_N),
        "z not advanced": (1, 1, oracle.PP_Z_FROZEN),
        "c_j from raters": (1, 1, oracle.PP_C_RATERS),
        "chunks 2 instead of 1": (1, 2, 0),
        "chunks 2 instead of 3": (3, 2, 0),
        "g_u not reset between chunks": (3, 3, oracle.PP_G_KEPT),
    }


@pytest.mark.parametrize("case", sorted(DISCRIMINATION))
def test_mutant_schedules_move_the_factors(case):
    """SVD, then SVD++ (the relaxation of tests/sgd_schedule.oracle_fit): the order mutants, and for SVD++ the
    mutants of the y_j side."""
    shape, B, C, f = DISCRIMINATION[case]
    u, i, r, nu, ni = S.draw(**shape)
    rng = np.random.RandomState(0)
    pu0, qi0 = rng.normal(0, S.INIT_STD, (nu, f)), rng.normal(0, S.INIT_STD, (ni, f))
    yj0 = rng.normal(0, S.INIT_STD, (ni, f))
    o, mutants = _mutants(u, i, B, C, 1)
    want = S.oracle_fit(u, i, r, o, pu0, qi0)
    if case == "dense":
        assert "tail reversed" in mutants
    report = []
    for name, m in mutants.items():
        got = S.oracle_fit(u, i, r, m, pu0, qi0)
        d = S.max_dist(want, got)
        report.append("%s: %.3g = %.0f x ATOL" % (name, d, d / S.ATOL))
        assert d >= S.MARGIN * S.ATOL, (case, name, d)
    print("\n%s (B=%d, C=%d, f=%d): %s" % (case, B, C, f, "; ".join(report)))

    stratum = S.schedule(u, i, B, C)["stratum"]

    def pp(order, chunks, variant=0):
        return S.oracle_fit(u, i, r, order, pu0, qi0, yj0=yj0, stratum=stratum, bounds=S.chunk_bounds(B, chunks),
                            variant=variant)
    exact = {1: pp(o, 1)}
    runs = [(name, exact[1], pp(m, 1)) for name, m in mutants.items()]
    for name, (base, chunks, variant) in _pp_mutants().items():
        if base not in exact:
            exact[base] = pp(o, base)
        runs.append((name, exact[base], pp(o, chunks, variant)))
    report, dists = [], []
    for name, a, b in runs:
        d = S.max_dist(a, b)
        dists.append(d / S.ATOL)
        report.append("%s: %.3g = %.0f x ATOL" % (name, d, d / S.ATOL))
        assert d >= S.MARGIN * S.ATOL, (case, "svdpp", name, d)
    print("%s SVD++: smallest %.0f x ATOL; %s" % (case, min(dists), "; ".join(report)))


def test_oracle_is_order_sensitive_only_through_the_order():
    """The same order twice gives bit-identical oracle factors (the distances above are the order's alone)."""
    u, i, r, nu, ni = S.draw(200, 150, 5000, seed=3)
    rng = np.random.RandomState(1)
    pu0, qi0 = rng.normal(0, .1, (nu, 8)), rng.normal(0, .1, (ni, 8))
    o = S.schedule_order(u, i, 8, 2)
    a, b = S.oracle_fit(u, i, r, o, pu0, qi0), S.oracle_fit(u, i, r, o.copy(), pu0, qi0)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    w = oracle.svd_sgd(u[o], i[o], r[o], pu0, qi0, S.EPOCHS, True, S.f32(np.mean(r)), *([S.f32(S.LR)] * 4),
                       *([S.f32(S.REG)] * 4))
    assert all(np.array_equal(x, y) for x, y in zip(a, w))


# --------------------------------------------------------------------------------------------------------------
# the SVD++ relaxation (oracle.svdpp_relaxed_sgd) and its link to the reference (oracle.svdpp_sgd)
LRS = (0.011, 0.013, 0.017, 0.019, 0.023)        # bu, bi, pu, qi, yj: a swapped pair moves the result
REGS = (0.029, 0.031, 0.037, 0.041, 0.043)


def _relaxed_py(u, i, r, order, stratum, bounds, pu0, qi0, yj0, epochs, mu, lr, reg):
    """The relaxation of DESIGN.md section 6, literally and slowly (small inputs only)."""
    (lbu, lbi, lpu, lqi, lyj), (rbu, rbi, rpu, rqi, ryj) = lr, reg
    nu, ni = len(pu0), len(qi0)
    pu, qi, yj, bu, bi = pu0.copy(), qi0.copy(), yj0.copy(), np.zeros(nu), np.zeros(ni)
    items = [i[u == x] for x in range(nu)]
    raters = [u[i == j] for j in range(ni)]
    isq = np.array([1 / np.sqrt(len(s)) if len(s) else 0. for s in items])
    d = 1 - lyj * ryj
    for _ in range(epochs):
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            z = np.stack([isq[x] * yj[items[x]].sum(0) for x in range(nu)])
            g, cnt = np.zeros_like(pu), np.zeros(nu)
            for k in order:
                if not lo <= stratum[k] < hi:
                    continue
                x, j = u[k], i[k]
                p, q, zz = pu[x].copy(), qi[j].copy(), z[x].copy()
                err = r[k] - (mu + bu[x] + bi[j] + q @ (p + zz))
                bu[x] += lbu * (err - rbu * bu[x])
                bi[j] += lbi * (err - rbi * bi[j])
                pu[x] = p + lpu * (err * q - rpu * p)
                qi[j] = q + lqi * (err * (p + zz) - rqi * q)
                z[x] = zz + lyj * (err * q - ryj * zz)
                g[x] += err * isq[x] * q
                cnt[x] += 1
            for j in range(ni):
                c = cnt[raters[j]].sum()
                if c == 0:
                    continue
                gain = lyj if d == 1 else lyj * (1 - d ** c) / (c * (1 - d))
                yj[j] = yj[j] * d ** c + gain * g[raters[j]].sum(0)
    return pu, qi, bu, bi, yj


@pytest.mark.parametrize("reg_yj", (REGS[4], 0.0))
@pytest.mark.parametrize("chunks", (1, 3))
def test_relaxed_oracle_literal_transcription(chunks, reg_yj):
    """The C relaxation equals its pseudo-code, transcribed in numpy, to fp64 rounding; reg_yj = 0 takes the plain
    sum (no 0 / 0)."""
    u, i, r, nu, ni = S.draw(40, 30, 500, seed=8)
    B, C = 4, 2
    sc = S.schedule(u, i, B, C)
    rng = np.random.RandomState(5)
    pu0, qi0, yj0 = (rng.normal(0, S.INIT_STD, (m, 6)) for m in (nu, ni, ni))
    reg = REGS[:4] + (reg_yj,)
    got = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, 2, lr=LRS, reg=reg, yj0=yj0, stratum=sc["stratum"],
                       bounds=S.chunk_bounds(B, chunks))
    want = _relaxed_py(u, i, r, sc["order"], sc["stratum"], S.chunk_bounds(B, chunks), pu0, qi0, yj0, 2,
                       S.f32(np.mean(r)), [S.f32(x) for x in LRS], [S.f32(x) for x in reg])
    assert all(np.isfinite(x).all() for x in got)
    assert S.max_dist(got, want) <= 1e-12, [float(np.abs(a - b).max()) for a, b in zip(got, want)]
    assert S.max_dist(got[4:], (yj0,)) > 1e-3                    # y_j moved


def _pp_reference(u, i, r, order, pu0, qi0, yj0, epochs, lr, reg):
    """oracle.svdpp_sgd on the ratings in `order`, as (pu, qi, bu, bi, yj)."""
    ptr, idx = S.ur_csr(u, i, len(pu0))
    pu, qi, yj, bu, bi = oracle.svdpp_sgd(u[order], i[order], r[order], ptr, idx, pu0, qi0, yj0, epochs,
                                          S.f32(np.mean(r)), *[S.f32(x) for x in lr], *[S.f32(x) for x in reg])
    return pu, qi, bu, bi, yj


@pytest.mark.parametrize("B,C,chunks", [(1, 1, 1), (4, 2, 1), (8, 2, 3)])
def test_relaxed_oracle_is_the_reference_on_a_conflict_free_input(B, C, chunks):
    """A permutation matrix of ratings: each y_j has one rater, who rates nothing else, so applying its gradient
    after the chunk is the reference's per-rating update."""
    n, f = 400, 12
    rng = np.random.RandomState(9)
    u = np.arange(n, dtype=np.int32)
    i = rng.permutation(n).astype(np.int32)
    r = rng.randint(1, 6, n).astype(np.float64)
    pu0, qi0, yj0 = (rng.normal(0, S.INIT_STD, (n, f)) for _ in range(3))
    sc = S.schedule(u, i, B, C)
    got = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, 3, lr=LRS, reg=REGS, yj0=yj0, stratum=sc["stratum"],
                       bounds=S.chunk_bounds(B, chunks))
    want = _pp_reference(u, i, r, sc["order"], pu0, qi0, yj0, 3, LRS, REGS)
    assert S.max_dist(got, want) <= 1e-12, [float(np.abs(a - b).max()) for a, b in zip(got, want)]
    assert S.max_dist(got[4:], (yj0,)) > 1e-3


@pytest.mark.parametrize("chunks", (1, 3))
def test_relaxed_oracle_without_lr_yj_is_the_reference_in_the_same_order(chunks):
    """lr_yj = 0: y_j and z_u never move, and the relaxation is the reference applied in the kernel's order."""
    u, i, r, nu, ni = S.draw(600, 400, 30_000, seed=1)
    B, C, f = 8, 2, 20
    sc = S.schedule(u, i, B, C)
    rng = np.random.RandomState(0)
    pu0, qi0, yj0 = (rng.normal(0, S.INIT_STD, (m, f)) for m in (nu, ni, ni))
    lr = LRS[:4] + (0.0,)
    got = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, lr=lr, reg=REGS, yj0=yj0, stratum=sc["stratum"],
                       bounds=S.chunk_bounds(B, chunks))
    want = _pp_reference(u, i, r, sc["order"], pu0, qi0, yj0, S.EPOCHS, lr, REGS)
    assert S.max_dist(got, want) <= 1e-12, [float(np.abs(a - b).max()) for a, b in zip(got, want)]
    assert np.array_equal(got[4], yj0)


def test_relaxed_oracle_reg_yj_zero_is_the_limit():
    """reg_yj = 0 (the plain sum lr_yj sum g_u) is the limit of the integrated decay as reg_yj -> 0."""
    u, i, r, nu, ni = S.draw(300, 200, 8000, seed=4)
    sc = S.schedule(u, i, 8, 2)
    rng = np.random.RandomState(1)
    pu0, qi0, yj0 = (rng.normal(0, S.INIT_STD, (m, 8)) for m in (nu, ni, ni))

    def fit(reg_yj, variant=0):
        return S.oracle_fit(u, i, r, sc["order"], pu0, qi0, yj0=yj0, stratum=sc["stratum"],
                            bounds=S.chunk_bounds(8), reg=(S.REG,) * 4 + (reg_yj,), variant=variant)
    plain = fit(0.0)
    assert S.max_dist(plain, fit(1e-9)) <= 1e-6
    assert S.max_dist(plain, fit(0.0, oracle.PP_NO_DECAY)) == 0.0
    assert S.max_dist(plain, fit(S.REG)) >= S.MARGIN * S.ATOL


# --------------------------------------------------------------------------------------------------------------
# the planner's shared-memory arithmetic
def test_plan_smem_at_the_config2_and_ml20m_shapes():
    # ml-1M (config 2), f = 100, 7 clusters of 16: 34 item rows per block, both blocks staged
    assert S.plan_smem(6040, 3706, 100, 112, 16)[:2] == (True, True)
    # ml-20M, f = 100: two item buffers fit at the B = 144 first tried, not at the B = 112 of 7 clusters
    assert S.plan_smem(138_000, 27_000, 100, 144, 16)[0]
    assert not S.plan_smem(138_000, 27_000, 100, 112, 16)[0]
    assert S.plan_smem(138_000, 27_000, 100, 112, 16)[3] == 24_444


@pytest.mark.parametrize("f,window", [(50, (51_521, 66_096)), (100, (26_993, 34_704)), (150, (17_809, 22_896)),
                                      (200, (13_553, 17_424))])
def test_cluster_cap_windows(f, window):
    """Item counts (2 000 users, 400 k ratings, 148 SMs, 7 co-resident clusters of 16) at which the unchecked cap
    of B produced a clustered plan without item buffers; tests/test_gpu_sgd_schedule.py creates plans inside and
    around these windows on the device."""
    assert S.clamp_window(f, 2000, 400_000, items=range(window[0] - 500, window[1] + 500)) == window
