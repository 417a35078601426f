"""TEST INFRASTRUCTURE: the order in which the stratified SGD kernel (csrc/sgd.cu) applies the rating updates.

Given the COO the plan was created from, in the order it received it (``Trainset.coo()``), and the plan's layout
(B blocks, cluster size C, P ranks of a ring), ``schedule_order`` returns the permutation of the ratings that one epoch
of ``dsgd_svd_kernel`` applies:

* every rating gets the cell key of ``dsgd_key_kernel``: rank ``g = u % P``, sub-epoch ``S``, user block ``ub``, item
  block ``ibk``, outer / inner step ``T`` / ``t``, stratum ``s = S B + T C + t``, ``cell = s B + ub``;
* the keys are sorted stably (input order inside a cell);
* each cell is coloured greedily in that order with 64-bit masks, as ``dsgd_color_kernel`` does: the lowest colour
  0..62 that neither the user's nor the item's mask holds, 63 (the sequential tail) when there is none;
* each cell is sorted stably by colour;
* cells are emitted by stratum ``s`` (sub-epoch first), then rank ``g``, then user block ``ub``.

Cells of one stratum share no user and no item, ratings of one colour share no row, and every row sees its cells in
stratum order, so applying the ratings in this sequence is equivalent to what the kernel does, provided that its
hand-offs of item blocks are correct.  ``oracle.svd_sgd(u[o], i[o], r[o], ...)`` on this order is then an
element-wise reference for the kernel's factors.  DEP mode (``SB2_DSGD_DEP=1``) applies the same order: its
dependency counts follow the colour-sorted records.

SVD++ runs the same kernel and order, but not the reference's per-rating ``y_j`` updates: the user row carries
``z_u = sum y_j / sqrt|I_u|`` and a gradient accumulator ``g_u``, and the accumulated gradients reach ``y_j`` once per
chunk of strata (DESIGN.md section 6).  ``oracle_fit(..., yj0=...)`` restates that relaxation in fp64
(``oracle.svdpp_relaxed_sgd``): the same order, each rating's stratum, and the chunks' strata (``chunk_bounds``: the
whole epoch by default and on a ring, ``SB2_SVDPP_CHUNKS`` of them on one GPU).  Its link to the reference is pinned
on the CPU (tests/test_sgd_schedule_cpu.py): on a conflict-free input, and with ``lr_yj = 0``, it equals
``oracle.svdpp_sgd`` to fp64 rounding.

``plan_smem`` restates the planner's shared-memory arithmetic (``svd_plan_create_dev``) for the layout tests.
"""
import numpy as np

NW = 64                 # waves per cell: colours 0..62 and the tail
TAIL = NW - 1
SMEM_BUDGET = 200 * 1024

# Hyper-parameters of the schedule-exact comparisons.  Learning rates this large make the update order a first-order
# effect, so that a lost, duplicated or reordered update moves the factors far beyond fp32 rounding.
LR, REG, INIT_STD, EPOCHS = 0.03, 0.02, 0.1, 2
# Largest element-wise |kernel - oracle| allowed on pu, qi, bu, bi (and yj of SVD++, against the relaxation).  Every
# mutant schedule of tests/test_sgd_schedule_cpu.py must move the oracle's factors by at least MARGIN times this.
ATOL = 2e-5
MARGIN = 20


def f32(x):
    """A scalar as the kernel sees it (DsgdArgs holds fp32 copies of mu and the hyper-parameters)."""
    return float(np.float32(x))


def ur_csr(u, i, n_users):
    """(u_ptr, ui_idx) of the ratings grouped by user, input order inside a user (Trainset.user_csr's layout)."""
    u = np.asarray(u, dtype=np.int64)
    o = np.argsort(u, kind="stable")
    return np.r_[0, np.cumsum(np.bincount(u, minlength=n_users))].astype(np.int64), np.asarray(i)[o].astype(np.int32)


def chunk_bounds(n_strata, chunks=1):
    """Strata of the y_j applications of one epoch: chunk c = [bounds[c], bounds[c + 1]) (svd_plan_run)."""
    return [n_strata * c // chunks for c in range(chunks + 1)]


def oracle_fit(u, i, r, order, pu0, qi0, epochs=EPOCHS, biased=True, lr=LR, reg=REG, yj0=None, stratum=None,
               bounds=None, mu=None, variant=0):
    """The fp64 oracle on the ratings in `order`, with the kernel's fp32 scalars.  lr / reg: one value for all, or
    (bu, bi, pu, qi[, yj]); mu: the global mean (default: the mean of r).

    SVD (yj0 None): the sequential reference; returns (pu, qi, bu, bi).
    SVD++ (yj0 given): the kernel's relaxation (oracle.svdpp_relaxed_sgd), always biased; `stratum` per rating
    (indexed like u), `bounds` the chunks' strata (chunk_bounds), `variant` a mutation of it; returns
    (pu, qi, bu, bi, yj)."""
    import oracle
    pp = yj0 is not None
    k = 5 if pp else 4
    lr = [f32(x) for x in (lr if np.ndim(lr) else [lr] * k)]
    reg = [f32(x) for x in (reg if np.ndim(reg) else [reg] * k)]
    assert len(lr) == len(reg) == k
    mu = f32(np.mean(r) if mu is None else mu) if biased or pp else 0.0
    if not pp:
        return oracle.svd_sgd(u[order], i[order], r[order], pu0, qi0, epochs, biased, mu, *lr, *reg)
    ptr, idx = ur_csr(u, i, len(pu0))
    pu, qi, yj, bu, bi = oracle.svdpp_relaxed_sgd(u, i, r, ptr, idx, stratum, order, bounds, pu0, qi0, yj0, epochs,
                                                  mu, *lr, *reg, variant=variant)
    return pu, qi, bu, bi, yj


def max_dist(a, b):
    return max(float(np.max(np.abs(x - y))) if x.size else 0.0 for x, y in zip(a, b))


def cell_keys(u, i, B, C, P=1):
    """(rank, stratum s of the epoch, user block ub, cell) per rating, as dsgd_key_kernel computes them."""
    u = np.asarray(u, dtype=np.int64)
    i = np.asarray(i, dtype=np.int64)
    if B % C:
        raise ValueError("B must be a multiple of C")
    g = u % P
    S = ((i % P) - g + P) % P
    ub, ibk = (u // P) % B, (i // P) % B
    K = B // C
    Cl, c, D, j = ub // C, ub % C, ibk // C, ibk % C
    T, t = (D - Cl + K) % K, (j - c + C) % C
    s = S * B + T * C + t
    return g, s, ub, s * B + ub


def greedy_colours(u, i, cell_sorted_order, cells):
    """Colour of every rating (indexed like u, i): ratings visited in `cell_sorted_order` (cell by cell, input order
    inside a cell); `cells[k]` identifies k's cell (rank included).  Lowest colour free in both rows' masks, else 63."""
    col = np.empty(len(u), dtype=np.int64)
    uu, ii, cc = u.tolist(), i.tolist(), cells.tolist()
    cur, mu, mi = None, {}, {}
    for k in cell_sorted_order.tolist():
        if cc[k] != cur:
            cur, mu, mi = cc[k], {}, {}
        a, b = uu[k], ii[k]
        used = mu.get(a, 0) | mi.get(b, 0)
        c = (~used & (used + 1)).bit_length() - 1      # lowest clear bit
        if c >= TAIL:
            c = TAIL
        else:
            mu[a] = mu.get(a, 0) | (1 << c)
            mi[b] = mi.get(b, 0) | (1 << c)
        col[k] = c
    return col


def schedule(u, i, B, C, P=1):
    """dict(order, colour, rank, stratum, ub, cell) of one epoch; order is the permutation the kernel applies."""
    u = np.asarray(u, dtype=np.int64)
    i = np.asarray(i, dtype=np.int64)
    g, s, ub, cell = cell_keys(u, i, B, C, P)
    gcell = g * (P * B * B) + cell                     # one key space over the ranks
    by_cell = np.argsort(gcell, kind="stable")
    col = greedy_colours(u, i, by_cell, gcell)
    pos = np.arange(len(u))
    order = np.lexsort((pos, col, ub, g, s))           # last key is the primary one
    return dict(order=order, colour=col, rank=g, stratum=s, ub=ub, cell=gcell)


def schedule_order(u, i, B, C, P=1):
    return schedule(u, i, B, C, P)["order"]


def plan_smem(n_users, n_items, f, B, C, P=1, with_yj=False, dep_mode=False):
    """(stage_i, stage_u, bytes used before the records, floats per item buffer): the planner's plan_smem."""
    fp = -(-f // 4) * 4
    us = 3 * fp if with_yj else fp
    nu_max, ni_max = -(-n_users // P), -(-n_items // P)
    mul, mil = -(-nu_max // B), -(-ni_max // B)
    fixed = (2 * (NW + 1) + 2 * P * B) * 4 + 64 + ((mul + mil) * 4 if dep_mode else 0)
    ibuf = -(-(mil * (fp + 1)) // 4) * 4
    need_i = (2 if C > 1 else 1) * ibuf * 4 + 16
    need_u = mul * (us + 3) * 4 + 16
    min_rec = 256 * 32
    stage_i = fixed + min_rec + need_i <= SMEM_BUDGET
    stage_u = stage_i and fixed + min_rec + need_i + need_u <= SMEM_BUDGET
    used = fixed + (need_i if stage_i else 0) + (need_u if stage_u else 0)
    return stage_i, stage_u, used, ibuf


def unclamped_cluster_blocks(n_users, n_items, n, n_sm, C, P=1):
    """B the planner first tries for cluster size C (before capping it at the co-resident clusters)."""
    b_cells = max(1, int(np.sqrt(max(n, 1) / 16.0)))
    b_tot = min(n_sm, b_cells)
    if P > 1:
        b_tot = max(b_tot // P, min(16, b_tot))
    b_lim = min(b_tot, -(-n_users // P), -(-n_items // P))
    return b_lim // C * C


def clamp_window(f, n_users, n, n_sm=148, C=16, max_clusters=7, P=1, items=range(1000, 200_001)):
    """Item counts at which the cluster size C fits two item buffers at the B it first tries but not at the B capped
    at `max_clusters` co-resident clusters: the plans the unchecked cap turned into clusters without item buffers.
    Returns (first, last) or None."""
    hit = []
    for ni in items:
        b0 = unclamped_cluster_blocks(n_users, ni, n, n_sm, C, P)
        if b0 < 2 * C or b0 // C <= max_clusters:
            continue
        b1 = max_clusters * C
        if plan_smem(n_users, ni, f, b0, C, P)[0] and not plan_smem(n_users, ni, f, b1, C, P)[0]:
            hit.append(ni)
    if not hit:
        return None
    assert hit == list(range(hit[0], hit[-1] + 1)), "the window is an interval"
    return hit[0], hit[-1]


def draw(n_users, n_items, n, seed, dense_users=0, dense_share=0.5, step=0.5):
    """Unique (u, i) pairs with ratings on a `step` grid from a planted rank-4 model, returned in Trainset.coo()
    order (u ascending, draw order inside a user); every user and item has a rating.  dense_users > 0: that many
    users rate `dense_share` of all items each (cells beyond the colour limit and beyond the staged records)."""
    rng = np.random.default_rng(seed)
    lin = []
    if dense_users:
        for x in range(dense_users):
            lin.append(x * n_items + rng.choice(n_items, int(dense_share * n_items), replace=False))
    # every user and every item once, then uniform pairs
    lin.append(np.arange(max(n_users, n_items)) % n_users * n_items + rng.permutation(max(n_users, n_items)) % n_items)
    lin.append(rng.integers(0, n_users * n_items, int(n * 1.2) + 64))
    lin = np.concatenate(lin)
    _, first = np.unique(lin, return_index=True)
    lin = lin[np.sort(first)]
    base = int(dense_users * int(dense_share * n_items)) + max(n_users, n_items)
    lin = np.concatenate((lin[:base], rng.permutation(lin[base:])[:max(0, n - base)]))
    u, i = lin // n_items, lin % n_items
    assert len(np.unique(u)) == n_users and len(np.unique(i)) == n_items
    p, q = rng.normal(0, .5, (n_users, 4)), rng.normal(0, .5, (n_items, 4))
    r = 3.5 + np.einsum("kf,kf->k", p[u], q[i]) + rng.normal(0, .7, len(u))
    r = np.clip(np.round(r / step) * step, 1.0, 5.0)
    o = np.argsort(u, kind="stable")
    return u[o].astype(np.int32), i[o].astype(np.int32), r[o], n_users, n_items
