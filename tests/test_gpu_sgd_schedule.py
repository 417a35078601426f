"""The stratified SGD kernel (csrc/sgd.cu) held to its exact update schedule, and the planner held to its layout rules.

* Layout sweep: plans are created and their layout read back (sb2_svd_plan_layout), never run, across factor
  counts, item counts inside and around the windows where capping B at the co-resident clusters used to leave a
  clustered plan without item buffers (tests/sgd_schedule.py: clamp_window), SVD and SVD++, and virtual rings.  A
  plan with clusters stages its item blocks, fits the device's shared memory and has at most one CTA per SM; a
  layout the kernel cannot run comes back as SB2_ERR_UNSUPPORTED, never as a plan.
* Schedule-exact factors: for every path of the kernel (staging variants, cluster sizes, both DSMEM hops, the
  colour tail, records beyond the staged ones, lane shapes, unbiased SVD, DEP mode, split launches, rings), the
  case first asserts the layout it is meant to reach, then runs a few epochs and requires pu, qi, bu, bi to equal
  the fp64 oracle applied in the kernel's schedule (sgd_schedule.schedule_order) to within sgd_schedule.ATOL.  A
  lost, duplicated or reordered update, a stale item block or a race on a hand-off moves the factors by at least
  MARGIN x ATOL (tests/test_sgd_schedule_cpu.py).
* SVD++ on the same paths (and SB2_SVDPP_CHUNKS, reg_yj = 0, rows without ratings): pu, qi, bu, bi and yj equal the
  fp64 restatement of the kernel's y_j relaxation (DESIGN.md section 6, sgd_schedule.oracle_fit with yj0) to within
  ATOL -- the z_u refresh, the item-side application (one GPU) and the ranks' partial sums + all-reduce (rings).
  SVDpp.fit with ten distinct learning rates / regularisations pins the host's parameter plumbing.
* The same plan reset and run again is bit-identical; SVD fits at the full ml-20M shape.
"""
import ctypes as C

import numpy as np
import pytest

import oracle
import sgd_schedule as S

pytestmark = pytest.mark.gpu

import surprise_b200 as sb  # noqa: E402
from surprise_b200 import _native as nat  # noqa: E402
from surprise_b200 import synth  # noqa: E402

MAX_ERR = {}       # case -> largest element-wise |kernel - oracle| (printed at the end of the module)


@pytest.fixture(scope="module", autouse=True)
def _report_max_errors():
    yield
    if MAX_ERR:
        worst = max(MAX_ERR.values())
        print("\nschedule-exact max |kernel - oracle|: %.3g (ATOL %.3g); %s" % (
            worst, S.ATOL, ", ".join("%s %.2g" % kv for kv in sorted(MAX_ERR.items()))))


def _prm(f, epochs, mu, biased=1, lr=S.LR, reg=S.REG, yj=False, reg_yj=None):
    reg_yj = reg if reg_yj is None else reg_yj
    return nat.SgdParams(n_factors=f, n_epochs=epochs, biased=int(biased), reserved=0, global_mean=mu, lr_bu=lr,
                         lr_bi=lr, lr_pu=lr, lr_qi=lr, lr_yj=lr if yj else 0., reg_bu=reg, reg_bi=reg, reg_pu=reg,
                         reg_qi=reg, reg_yj=reg_yj if yj else 0.)


def layout(plan):
    ints = [C.c_int() for _ in range(8)]
    smem, rec_cap, max_cell = C.c_int64(), C.c_int(), C.c_int()
    nat.check(nat.lib().sb2_svd_plan_layout(plan, *[C.byref(x) for x in ints], C.byref(smem), C.byref(rec_cap),
                                            C.byref(max_cell)))
    names = ("B", "C", "G", "CH", "W", "stage_u", "stage_i", "dep_mode")
    out = {k: v.value for k, v in zip(names, ints)}
    out.update(smem=smem.value, rec_cap=rec_cap.value, max_cell=max_cell.value)
    return out


def _device_limits():
    import torch
    p = torch.cuda.get_device_properties(torch.cuda.current_device())
    return p.multi_processor_count, p.shared_memory_per_block_optin


def create_layout(u, i, r, nu, ni, f, with_yj=False, rank=0, world=1):
    """Create a plan, read its layout, destroy it (nothing runs).  Returns (return code, layout or None, message)."""
    lib = nat.lib()
    d_u, d_i, d_r = nat.to_dev(u, np.int32), nat.to_dev(i, np.int32), nat.to_dev(r, np.float64)
    d_up = d_ui = None
    if with_yj:
        ptr, idx = S.ur_csr(u, i, nu)
        d_up, d_ui = nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32)
    prm = _prm(f, 1, float(np.mean(r)), yj=with_yj)
    plan = C.c_void_p()
    rc = lib.sb2_svd_ring_create_dev(nu, ni, len(r), nat.ptr(d_u), nat.ptr(d_i), nat.ptr(d_r), C.byref(prm),
                                     int(with_yj), nat.ptr(d_up), nat.ptr(d_ui), rank, world, nat.stream(),
                                     C.byref(plan))
    if rc != nat.OK:
        return rc, None, lib.sb2_last_error().decode()
    try:
        return rc, layout(plan), ""
    finally:
        import torch
        torch.cuda.synchronize()
        lib.sb2_svd_plan_destroy(plan)


def _uniform(nu, ni, n, seed):
    """Rating pairs for planning only (duplicates allowed), in user order."""
    rng = np.random.default_rng(seed)
    u = np.sort(rng.integers(0, nu, n)).astype(np.int32)
    i = rng.integers(0, ni, n).astype(np.int32)
    return u, i, rng.integers(1, 6, n).astype(np.float64)


def _check_layout(lay, rc, msg, n_sm, optin, where):
    """where: dict of the plan's shape, part of every message."""
    assert rc in (nat.OK, nat.ERR_UNSUPPORTED), (where, rc, msg)
    if rc != nat.OK:
        return
    assert lay["C"] == 1 or lay["stage_i"], ("clusters without item buffers", where, lay)
    assert lay["smem"] <= optin, (where, lay)
    assert 1 <= lay["B"] <= n_sm and lay["B"] % lay["C"] == 0, (where, lay)
    assert lay["stage_u"] <= lay["stage_i"], (where, lay)
    if where.get("world", 1) > 1:
        assert lay["stage_i"], (where, lay)


@pytest.mark.parametrize("f", (3, 8, 20, 50, 100, 150, 200, 300))
def test_layout_sweep(f):
    """Plans are only created: the layout is read on the host, no SGD kernel runs."""
    n_sm, optin = _device_limits()
    nu, n = 2000, 400_000
    w = S.clamp_window(f, nu, n, n_sm=n_sm, items=range(2000, 80_001))
    items = [27_000, 3706]          # the ml-20M and ml-1M item counts first
    if w is not None:
        lo, hi = w
        items += sorted({lo - 1, lo, (lo + hi) // 2, hi, hi + 1} - set(items))
    seen = []
    for k, ni in enumerate(items):
        u, i, r = _uniform(nu, ni, n, seed=k)
        for with_yj in (False, True):
            rc, lay, msg = create_layout(u, i, r, nu, ni, f, with_yj)
            seen.append((ni, with_yj, rc, lay))
            _check_layout(lay, rc, msg, n_sm, optin, dict(n_items=ni, f=f, svdpp=with_yj))
    assert any(rc == nat.OK for _, _, rc, _ in seen)
    print("\nf=%d: %s" % (f, "; ".join("%d%s: %s" % (ni, "++" if yj else "", "unsupported" if lay is None else
                                                   "B=%(B)d C=%(C)d su=%(stage_u)d si=%(stage_i)d" % lay)
                                      for ni, yj, rc, lay in seen)))


@pytest.mark.parametrize("world", (2, 3, 4))
@pytest.mark.parametrize("f", (20, 100, 300))
def test_layout_sweep_rings(world, f):
    n_sm, optin = _device_limits()
    for ni in (3706, 27_000):
        u, i, r = _uniform(2000, ni, 400_000, seed=ni)
        for with_yj in (False, True):
            for rank in range(world):
                rc, lay, msg = create_layout(u, i, r, 2000, ni, f, with_yj, rank, world)
                _check_layout(lay, rc, msg, n_sm, optin,
                              dict(n_items=ni, f=f, svdpp=with_yj, rank=rank, world=world))


# ------------------------------------------------------------------------------------------------------------------
# schedule-exact factors
def plan_fit(u, i, r, nu, ni, f, epochs, pu0, qi0, biased=True, runs=1, yj0=None, reg_yj=None):
    """Create -> layout -> (reset -> run -> read) x runs -> status -> destroy through the plan API.  yj0 given: an
    SVD++ plan (the ur CSR of the ratings, lr_yj = LR, reg_yj = REG unless given); each run returns
    (pu, qi, bu, bi[, yj])."""
    import torch
    lib = nat.lib()
    with_yj = yj0 is not None
    d_u, d_i, d_r = nat.to_dev(u, np.int32), nat.to_dev(i, np.int32), nat.to_dev(r, np.float64)
    d_pu0, d_qi0 = nat.to_dev(pu0, np.float64), nat.to_dev(qi0, np.float64)
    d_yj0 = d_up = d_ui = None
    if with_yj:
        ptr, idx = S.ur_csr(u, i, nu)
        d_yj0, d_up, d_ui = nat.to_dev(yj0, np.float64), nat.to_dev(ptr, np.int64), nat.to_dev(idx, np.int32)
    prm = _prm(f, epochs, float(np.mean(r)) if biased or with_yj else 0., biased, yj=with_yj, reg_yj=reg_yj)
    plan = C.c_void_p()
    nat.check(lib.sb2_svd_plan_create_dev(nu, ni, len(r), nat.ptr(d_u), nat.ptr(d_i), nat.ptr(d_r), C.byref(prm),
                                          int(with_yj), nat.ptr(d_up), nat.ptr(d_ui), nat.stream(), C.byref(plan)))
    try:
        lay = layout(plan)
        out = []
        for _ in range(runs):
            nat.check(lib.sb2_svd_plan_reset_dev(plan, nat.ptr(d_pu0), nat.ptr(d_qi0), nat.ptr(d_yj0), nat.stream()))
            nat.check(lib.sb2_svd_plan_run(plan, epochs, nat.stream()))
            t = [nat.empty_dev(s, np.float64) for s in ((nu, f), (ni, f), (nu,), (ni,))]
            t_yj = nat.empty_dev((ni, f), np.float64) if with_yj else None
            nat.check(lib.sb2_svd_plan_read_dev(plan, *[nat.ptr(x) for x in t], nat.ptr(t_yj), nat.stream()))
            nat.check(lib.sb2_svd_plan_status(plan, nat.stream()))
            out.append(tuple(x.cpu().numpy() for x in t + ([t_yj] if with_yj else [])))
        return lay, out
    finally:
        torch.cuda.synchronize()
        lib.sb2_svd_plan_destroy(plan)


SHAPES = {
    # the reduced ml-1M-like shape: 7 clusters of 16 CTAs, both blocks staged (config 2's layout)
    "default": dict(n_users=3000, n_items=2000, n=400_000, seed=1),
    # 536 users per block: the user rows stay in global memory
    "many_users": dict(n_users=60_000, n_items=2000, n=400_000, seed=3),
    # 800 items per block at the unclustered B: the item rows stay in global memory
    "many_items": dict(n_users=2000, n_items=20_000, n=200_000, seed=4),
    # 40 users rating 60 % of the items: with 4 blocks most of a dense user's cell is colour tail, and cells hold
    # several times the records staged in shared memory
    "dense": dict(n_users=300, n_items=2000, n=300_000, seed=2, dense_users=40, dense_share=0.6),
    # the item count of the ml-20M shape with 2 000 users: inside the f = 100 window of the cluster cap
    "fault": dict(n_users=2000, n_items=27_000, n=400_000, seed=5),
    # the default shape in a plan of 40 more users and 24 more items, which have no ratings
    "unrated": dict(n_users=3000, n_items=2000, n=400_000, seed=6),
}
UNRATED = {"unrated": (40, 24)}
_DRAWN, _SCHEDULES = {}, {}


def _shape(name):
    if name not in _DRAWN:
        u, i, r, nu, ni = S.draw(**SHAPES[name])
        du, di = UNRATED.get(name, (0, 0))
        _DRAWN[name] = u, i, r, nu + du, ni + di
    return _DRAWN[name]


def _schedule(name, B, C):
    if (name, B, C) not in _SCHEDULES:
        u, i = _shape(name)[:2]
        _SCHEDULES[(name, B, C)] = S.schedule(u, i, B, C)
    return _SCHEDULES[(name, B, C)]


def _is(**want):
    return lambda lay: all(lay[k] == v for k, v in want.items())


CASES = [
    # id, shape, f, environment, expected layout, biased, SVD++
    ("bulk_hop_c16", "default", 100, {}, _is(C=16, stage_u=1, stage_i=1, G=8, CH=4), True, False),
    ("st_hop_c16", "default", 100, {"SB2_DSGD_HOP": "st"}, _is(C=16, stage_u=1, stage_i=1), True, False),
    ("c8", "default", 100, {"SB2_DSGD_CLUSTER": "8"}, _is(C=8, stage_i=1), True, False),
    ("c4", "default", 100, {"SB2_DSGD_CLUSTER": "4"}, _is(C=4, stage_i=1), True, False),
    ("c2", "default", 100, {"SB2_DSGD_CLUSTER": "2"}, _is(C=2, stage_i=1), True, False),
    ("c1", "default", 100, {"SB2_DSGD_CLUSTER": "1"}, _is(C=1, stage_u=1, stage_i=1), True, False),
    ("users_in_global", "many_users", 100, {}, lambda l: l["C"] > 1 and not l["stage_u"] and l["stage_i"], True,
     False),
    ("items_in_global_c1", "many_items", 100, {"SB2_DSGD_CLUSTER": "1"}, _is(C=1, stage_u=0, stage_i=0), True, False),
    ("tail_and_records_beyond_rec_cap", "dense", 20, {"SB2_DSGD_BLOCKS": "4"},
     lambda l: l["B"] == 4 and l["C"] == 2 and l["max_cell"] > l["rec_cap"], True, False),
    ("lanes_f3", "default", 3, {}, _is(C=16, G=1, CH=1), True, False),
    ("lanes_f50", "default", 50, {}, _is(C=16, G=4, CH=4), True, False),
    ("lanes_f150", "default", 150, {}, _is(C=16, G=16, CH=3), True, False),
    ("lanes_f300", "default", 300, {}, _is(G=32, CH=0), True, False),
    ("unbiased", "default", 20, {}, _is(C=16), False, False),
    ("dep", "default", 100, {"SB2_DSGD_DEP": "1"}, _is(dep_mode=1, G=32, stage_u=1, stage_i=1), True, False),
    ("split3", "default", 100, {"SB2_DSGD_SPLIT": "3"}, _is(C=16), True, False),
    ("fault_shape", "fault", 100, {}, lambda l: l["C"] > 1 and l["stage_i"] == 1, True, False),
    # SVD++ (pu, qi, bu, bi and yj against the relaxation): user rows of [p | z | g] (3 FP floats) change the
    # staging -- the default shape still stages both blocks at C = 16 (27 users x 303 floats per block) and C = 1
    # (86 users), 60 000 users do not
    ("pp_bulk_hop_c16", "default", 100, {}, _is(C=16, stage_u=1, stage_i=1, G=8, CH=4, dep_mode=0), True, True),
    ("pp_st_hop_c16", "default", 100, {"SB2_DSGD_HOP": "st"}, _is(C=16, stage_u=1, stage_i=1), True, True),
    ("pp_c8", "default", 100, {"SB2_DSGD_CLUSTER": "8"}, _is(C=8, stage_u=1, stage_i=1), True, True),
    ("pp_c4", "default", 100, {"SB2_DSGD_CLUSTER": "4"}, _is(C=4, stage_u=1, stage_i=1), True, True),
    ("pp_c2", "default", 100, {"SB2_DSGD_CLUSTER": "2"}, _is(C=2, stage_u=1, stage_i=1), True, True),
    ("pp_c1", "default", 100, {"SB2_DSGD_CLUSTER": "1"}, _is(C=1, stage_u=1, stage_i=1), True, True),
    ("pp_users_in_global", "many_users", 100, {}, lambda l: l["C"] > 1 and not l["stage_u"] and l["stage_i"], True,
     True),
    ("pp_items_in_global_c1", "many_items", 100, {"SB2_DSGD_CLUSTER": "1"}, _is(C=1, stage_u=0, stage_i=0), True,
     True),
    ("pp_tail_and_records_beyond_rec_cap", "dense", 20, {"SB2_DSGD_BLOCKS": "4"},
     lambda l: l["B"] == 4 and l["C"] == 2 and l["stage_u"] and l["max_cell"] > l["rec_cap"], True, True),
    ("pp_lanes_f3", "default", 3, {}, _is(C=16, G=1, CH=1, stage_u=1, stage_i=1), True, True),
    ("pp_lanes_f50", "default", 50, {}, _is(C=16, G=4, CH=4, stage_u=1, stage_i=1), True, True),
    ("pp_lanes_f150", "default", 150, {}, _is(C=16, G=16, CH=3, stage_u=1, stage_i=1), True, True),
    ("pp_lanes_f300", "default", 300, {}, _is(G=32, CH=0), True, True),
    ("pp_split3", "default", 100, {"SB2_DSGD_SPLIT": "3"}, _is(C=16), True, True),
    ("pp_chunks2", "default", 100, {"SB2_SVDPP_CHUNKS": "2"}, _is(C=16), True, True),
    ("pp_chunks3", "default", 100, {"SB2_SVDPP_CHUNKS": "3"}, _is(C=16), True, True),
    ("pp_chunks_clamped_to_B", "default", 20, {"SB2_SVDPP_CHUNKS": "100000"}, _is(C=16), True, True),
    ("pp_dep_ignored", "default", 100, {"SB2_DSGD_DEP": "1"}, _is(dep_mode=0, G=8, CH=4), True, True),
    ("pp_reg_yj_0", "default", 20, {}, _is(C=16), True, True),
    ("pp_unrated_rows", "unrated", 100, {}, _is(C=16, stage_u=1, stage_i=1), True, True),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_schedule_exact_factors(case, monkeypatch):
    name, shape, f, env, expect, biased, with_yj = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    u, i, r, nu, ni = _shape(shape)
    rng = np.random.RandomState(7)
    pu0, qi0 = rng.normal(0, S.INIT_STD, (nu, f)), rng.normal(0, S.INIT_STD, (ni, f))
    yj0 = rng.normal(0, S.INIT_STD, (ni, f)) if with_yj else None
    reg_yj = 0.0 if name == "pp_reg_yj_0" else S.REG
    lay, (got,) = plan_fit(u, i, r, nu, ni, f, S.EPOCHS, pu0, qi0, biased, yj0=yj0, reg_yj=reg_yj)
    assert expect(lay), (name, lay)
    sc = _schedule(shape, lay["B"], lay["C"])
    if shape == "dense":
        assert (sc["colour"] == S.TAIL).any(), "the case reaches the colour tail"
    if with_yj:
        chunks = min(int(env.get("SB2_SVDPP_CHUNKS", 1)), lay["B"])    # the planner clamps the chunks to B
        want = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, S.EPOCHS, yj0=yj0, stratum=sc["stratum"],
                            bounds=S.chunk_bounds(lay["B"], chunks), reg=(S.REG,) * 4 + (reg_yj,))
    else:
        want = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, S.EPOCHS, biased)
    err = S.max_dist(got, want)
    MAX_ERR[name] = err
    # per array: the largest difference and the element where it is
    where = [(float(np.abs(a - b).max()), np.unravel_index(np.argmax(np.abs(a - b)), a.shape))
             for a, b in zip(got, want)]
    assert err <= S.ATOL, (name, lay, where)
    # rows without ratings: the fp32 rounding of their initial values, bit for bit, and zero biases
    ru, ri = np.setdiff1d(np.arange(nu), u), np.setdiff1d(np.arange(ni), i)
    if shape in UNRATED:
        assert len(ru) == UNRATED[shape][0] and len(ri) == UNRATED[shape][1]
    f32 = lambda a: a.astype(np.float32).astype(np.float64)
    assert np.array_equal(got[0][ru], f32(pu0[ru])) and np.array_equal(got[1][ri], f32(qi0[ri]))
    assert not got[2][ru].any() and not got[3][ri].any()
    if with_yj:
        assert np.array_equal(got[4][ri], f32(yj0[ri]))


@pytest.mark.parametrize("world,blocks", [(2, 32), (3, 32), (4, 16)])
def test_schedule_exact_virtual_ring(world, blocks, monkeypatch):
    """SVD, then SVD++: one persistent launch for SVD; for SVD++ svd_ring_epoch_local (z_u refresh, the P sub-epochs,
    the ranks' partial sums into xch), the all-reduce of xch and svdpp_item_apply_xch_kernel per epoch -- the
    relaxation with one chunk of P B strata, U_j over all ranks; every rank must hold the same y_j."""
    from test_gpu_ring import virtual_ring_fit
    monkeypatch.setenv("SB2_DSGD_BLOCKS", str(blocks))
    u, i, r, nu, ni = S.draw(2000, 1200, 150_000, seed=12)
    f = 24
    rng = np.random.RandomState(3)
    pu0, qi0, yj0 = (rng.normal(0, S.INIT_STD, (m, f)) for m in (nu, ni, ni))
    for with_yj in (False, True):
        rc, lay, msg = create_layout(u, i, r, nu, ni, f, with_yj, rank=0, world=world)
        assert rc == nat.OK, msg
        assert lay["B"] == blocks and lay["C"] > 1 and lay["stage_i"] and lay["stage_u"], (with_yj, lay)
        sc = S.schedule(u, i, lay["B"], lay["C"], world)
        prm = _prm(f, S.EPOCHS, float(np.mean(r)), yj=with_yj)
        if with_yj:
            got = virtual_ring_fit(world, nu, ni, u, i, r, prm, pu0, qi0, yj0, S.ur_csr(u, i, nu))
            want = S.oracle_fit(u, i, r, sc["order"], pu0, qi0, yj0=yj0, stratum=sc["stratum"],
                                bounds=S.chunk_bounds(world * lay["B"]))
            key = "pp_ring_P%d" % world
        else:
            got = virtual_ring_fit(world, nu, ni, u, i, r, prm, pu0, qi0)
            want = S.oracle_fit(u, i, r, sc["order"], pu0, qi0)
            key = "ring_P%d" % world
        err = S.max_dist(got, want)
        MAX_ERR[key] = err
        assert err <= S.ATOL, (world, with_yj, lay, [float(np.abs(a - b).max()) for a, b in zip(got, want)])


def test_svdpp_plumbing_vs_relaxation():
    """sb.SVDpp with ten distinct learning rates / regularisations and init_mean != 0: fit() must hand every one of
    them to the right place (SVDpp._sgd_params -> fill_args) and draw pu, qi, yj as the relaxation is fed them."""
    u, i, r, nu, ni = S.draw(1500, 900, 120_000, seed=21)
    ts = sb.Trainset.from_coo(u, i, r, nu, ni)
    f, epochs, seed, init_mean = 16, 2, 5, 0.05
    lr = dict(lr_bu=0.011, lr_bi=0.013, lr_pu=0.017, lr_qi=0.019, lr_yj=0.023)
    reg = dict(reg_bu=0.029, reg_bi=0.031, reg_pu=0.037, reg_qi=0.041, reg_yj=0.043)
    algo = sb.SVDpp(n_factors=f, n_epochs=epochs, init_mean=init_mean, init_std_dev=S.INIT_STD, random_state=seed,
                    **lr, **reg).fit(ts)
    uu, ii, rr = ts.coo()
    rc, lay, msg = create_layout(uu, ii, rr, nu, ni, f, with_yj=True)
    assert rc == nat.OK, msg
    rng = np.random.RandomState(seed)
    pu0, qi0, yj0 = (rng.normal(init_mean, S.INIT_STD, (m, f)) for m in (nu, ni, ni))
    sc = S.schedule(uu, ii, lay["B"], lay["C"])
    want = S.oracle_fit(uu, ii, rr, sc["order"], pu0, qi0, epochs, lr=list(lr.values()), reg=list(reg.values()),
                        yj0=yj0, stratum=sc["stratum"], bounds=S.chunk_bounds(lay["B"]), mu=ts.global_mean)
    got = (algo.pu, algo.qi, algo.bu, algo.bi, algo.yj)
    err = S.max_dist(got, want)
    MAX_ERR["pp_plumbing"] = err
    assert err <= S.ATOL, (lay, [float(np.abs(a - b).max()) for a, b in zip(got, want)])


def test_reset_and_rerun_bit_identical():
    u, i, r, nu, ni = _shape("default")
    f = 20
    rng = np.random.RandomState(11)
    pu0, qi0 = rng.normal(0, S.INIT_STD, (nu, f)), rng.normal(0, S.INIT_STD, (ni, f))
    _, (a, b) = plan_fit(u, i, r, nu, ni, f, 3, pu0, qi0, runs=2)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_ml20m_shape_svd_fit_vs_oracle():
    """SVD(n_factors=100) at the ml-20M shape: the fit completes (status OK) and its held-out RMSE / MAE are within
    0.005 of the sequential oracle on the same draw."""
    d = synth.shaped("ml-20m", seed=0)
    u, i, r = d["train"]
    ts = sb.Trainset.from_coo(u, i, r, d["n_users"], d["n_items"], (0.5, 5.0))
    algo = sb.SVD(n_factors=100, n_epochs=2, random_state=0).fit(ts)
    rng = np.random.RandomState(0)
    pu0 = rng.normal(0, .1, (ts.n_users, 100)); qi0 = rng.normal(0, .1, (ts.n_items, 100))
    uu, ii, rr = ts.coo()
    mu = float(ts.global_mean)
    w = oracle.svd_sgd(uu, ii, rr, pu0, qi0, 2, True, mu, *([.005] * 4), *([.02] * 4))
    tu, ti, tr = d["test"]
    want, _ = oracle.mf_estimate(tu, ti, True, mu, *w)
    got, _ = oracle.mf_estimate(tu, ti, True, mu, algo.pu, algo.qi, algo.bu, algo.bi)

    def scores(e):
        e = np.clip(e, 0.5, 5.0)
        return float(np.sqrt(np.mean((e - tr) ** 2))), float(np.mean(np.abs(e - tr)))
    (rw, mw), (rg, mg) = scores(want), scores(got)
    print("\nml-20M SVD f=100, 2 epochs: RMSE %.5f (oracle %.5f), MAE %.5f (oracle %.5f)" % (rg, rw, mg, mw))
    assert abs(rw - rg) <= 0.005 and abs(mw - mg) <= 0.005, (rw, rg, mw, mg)
