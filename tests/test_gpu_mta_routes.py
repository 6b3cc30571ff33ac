"""solve_mta on every route launch_mta can take, held to a float64 restatement of the reference (oracle/mta.py, the
same fp32 inputs and fp32-rounded parameters): the mode and its logits, and the solver state that jcb_mta_debug reads
back -- the squared bandwidths, the affinity A = P P^T and the final inlierness weights y.

The mode alone cannot see a subtly wrong solver.  MTA is a contraction: a bandwidth rank off by one, a softmax scale or
a lambda_y off by 1e-4 move the mode by less than its 2e-5 tolerance, while they move bw^2, A and y by 20x to 1e5x their
fp32 rounding.  test_tolerances_have_power (CPU, float64) pins that each tolerance below still sees such a mistake.

Routes (launch_mta's dispatch at a 220 KB shared-memory limit):
  tc+fast<N>   probabilities as a bf16 x 3-limb tensor-core GEMM (mta_split_x_kernel ...), then mta_fast_kernel<N>:
               D % 128 == 0 and the problem fits; N = 32 for V <= 4, 64 for V <= 12, 128 for V <= 32, 512 above.  At
               C = 403: V <= 82 at D = 512, V <= 62 at D = 768, V <= 47 at D = 1024 (D > 512 re-reads the mode from
               shared memory in the density passes)
  tc+smem      the same probabilities, mta_kernel<256> with the problem in shared memory: D % 128 == 64 (D = 64, 320),
               or V = 83..89 at C = 403, D = 512
  tc+big       the same probabilities, large-V pre-pass (mta_gram_big_kernel, mta_bw_big_kernel) + mta_kernel<1024>:
               V >= 90 at C = 403, D = 512
  simt+smem    fp32 SIMT mta_probs_kernel + mta_kernel<256>: D % 64 == 32 (D = 32, 96), V < 108
  simt+big     mta_probs_kernel + the large-V pre-pass: D = 96, V >= 108
  none+smem    C > 416: mta_kernel<256> computes logits and softmax itself, in shared memory (C = 1000: V < 52)
  none+scratch the same with its workspace in global scratch (C = 1000: V >= 52)

Largest error over the cases of this file with default-conditioned inputs (unit views, two clusters, the parameter
sets), per route, on a B200 at a 1000 W power limit (fp32 kernels vs the float64 oracle; y relative as defined below):
  route          mode     logits   bw^2     A        y
  tc+fast<32>    5.0e-8   1.2e-5   7.1e-7   1.1e-6   2.6e-5
  tc+fast<64>    2.0e-6   1.9e-4   8.4e-7   2.6e-6   2.4e-4   (k_frac = 0, i.e. one neighbour: 1.0e-3)
  tc+fast<128>   6.9e-7   5.0e-5   9.5e-7   1.8e-6   1.7e-4
  tc+fast<512>   1.5e-6   1.4e-4   1.1e-6   2.2e-6   2.4e-4
  tc+smem        3.9e-7   3.7e-5   1.4e-7   3.5e-6   6.5e-5
  tc+big         2.0e-7   2.4e-5   8.4e-7   2.8e-6   6.5e-5
  simt+smem      4.3e-6   3.5e-4   8.1e-8   4.7e-6   1.5e-4
  simt+big       1.8e-6   1.7e-4   3.9e-7   4.6e-6   2.9e-4
  none+smem      1.9e-6   2.4e-4   9.3e-8   5.4e-6   2.9e-4
  none+scratch   1.7e-6   1.4e-4   9.2e-8   3.8e-6   1.1e-4
Peaked text (temperature 0.01): A <= 2.7e-4, y <= 1.03e-3.  Near-duplicate views: mode <= 2.3e-8, A <= 3.8e-6.
The tc routes first measured A ~2e-5 and y up to 2e-3 (a mode 3.5e-5 off): the limb products were summed largest first,
see mta_split_x_kernel.  Route boundaries measured as listed; the fast kernel's at D > 512 are lower than at D = 512.

n_views = 1 is accepted (jcb_pipeline accepts it too) and pinned to what the reference computes: the bandwidth is the
mean of no distances, so the mode is all NaN, on every route that V = 1 can take.
"""
import re

import numpy as np
import pytest
import torch

from oracle import solve_mta as o_mta

# absolute unless noted; y: |y - y_ref| <= Y_RTOL (|y_ref| + Y_FLOOR), the floor because outlier views get weights
# near zero
MODE_TOL = 2e-5
LOGIT_TOL = 1e-2
BW2_TOL = 2e-6
A_TOL = 1e-5
Y_RTOL, Y_FLOOR = 3e-4, 1e-7
# peaked text (temperature 0.01): logits of O(1e3) whose fp32 rounding (~6e-5) is an error in the softmax exponent
A_TOL_PEAKED = 3e-4
Y_RTOL_PEAKED = 1.5e-3
# k_frac = 0 (k = 1): each bandwidth is one neighbour's distance, and the density's exponent scales with its inverse
Y_RTOL_ONE_NEIGHBOUR = 1.5e-3

TC = ("mta_split_x_kernel", "mta_split_t_kernel", "mta_softmax_rows_kernel")
BIG = ("mta_gram_big_kernel", "mta_bw_big_kernel", "mta_kernel<1024>")

# (V, C, D, route): one or more cases per route, and both sides of every boundary
CASES = [
    (1, 403, 512, "tc+fast<32>"), (2, 403, 512, "tc+fast<32>"), (4, 403, 512, "tc+fast<32>"),
    (5, 403, 512, "tc+fast<64>"), (12, 403, 512, "tc+fast<64>"), (13, 403, 512, "tc+fast<128>"),
    (32, 403, 512, "tc+fast<128>"), (33, 403, 512, "tc+fast<512>"), (82, 403, 512, "tc+fast<512>"),
    (83, 403, 512, "tc+smem"), (89, 403, 512, "tc+smem"), (90, 403, 512, "tc+big"), (513, 403, 512, "tc+big"),
    (9, 1, 512, "tc+fast<64>"), (9, 2, 512, "tc+fast<64>"), (9, 416, 512, "tc+fast<64>"),
    (9, 417, 512, "none+smem"), (9, 1000, 512, "none+smem"), (51, 1000, 512, "none+smem"),
    (52, 1000, 512, "none+scratch"),
    (9, 403, 32, "simt+smem"), (9, 403, 96, "simt+smem"), (107, 403, 96, "simt+smem"), (108, 403, 96, "simt+big"),
    (9, 403, 64, "tc+smem"), (33, 403, 320, "tc+smem"),
    (9, 403, 768, "tc+fast<64>"), (62, 403, 768, "tc+fast<512>"), (63, 403, 768, "tc+smem"),
    (2, 403, 1024, "tc+fast<32>"), (47, 403, 1024, "tc+fast<512>"), (48, 403, 1024, "tc+smem"),
    (50, 403, 1024, "tc+big"),
]
# one case per route for the input families and the parameters
REPS = [(9, 403, 512), (65, 403, 512), (85, 403, 512), (100, 403, 512), (9, 403, 96), (120, 403, 96), (20, 1000, 512),
        (60, 1000, 512), (20, 403, 768)]


def _case_id(c):
    return "V{}-C{}-D{}".format(*c[:3])


def _two_clusters(seed, I, V, D):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((I, 2, D))
    c /= np.linalg.norm(c, axis=-1, keepdims=True)
    x = c[:, (np.arange(V) >= (V + 1) // 2).astype(int)] + 0.3 * rng.standard_normal((I, V, D)) / np.sqrt(D)
    return (x / np.linalg.norm(x, axis=-1, keepdims=True)).astype(np.float32)


def _inputs(jb, family, V, C, D, seed=0):
    """feats [I, V, D] and text [D, C] fp32 (CPU) of an input family."""
    I = 2 if V > 200 else 3
    s = seed + 7 * V + C + D
    if family == "clusters":
        x = _two_clusters(s, I, V, D)
    else:
        spread = {"unit035": 0.35, "unit1": 1.0, "neardup": 1e-3, "peaked": 0.35}[family]
        x = jb.synth.make_unit_views(s, I, V, dim=D, spread=spread)
    t = jb.synth.make_text_features(seed=10 + s, num_classes=C, dim=D)
    return torch.from_numpy(x), torch.from_numpy(t).t().contiguous()


def _f32(v):
    return float(np.float32(v))


def _oracle_params(params):
    """the values the kernels see: jcb_mta_params holds fp32 fields (k_frac is a double)"""
    return {k: (v if k in ("k_frac", "max_iter") else _f32(v)) for k, v in params.items()}


def _y_err(y, y_ref):
    return float(((y - y_ref).abs() / (y_ref.abs() + Y_FLOOR)).max())


def _errors(jb, feats, text, params, cuda_dev):
    """jcb_mta_debug on (feats, text) vs the float64 oracle, image by image: {quantity: largest error}"""
    out = {k: v.cpu().double() for k, v in jb.blocks.mta_debug(feats.to(cuda_dev), text.to(cuda_dev), params).items()}
    err = {"mode": 0.0, "logits": 0.0, "bw2": 0.0, "A": 0.0, "y": 0.0}
    for i in range(feats.shape[0]):
        m, s = o_mta(feats[i], text, True, dtype=torch.float64, **_oracle_params(params))
        assert torch.isfinite(out["mode"][i]).all() and torch.isfinite(out["y"][i]).all()
        err["mode"] = max(err["mode"], float((out["mode"][i] - m[0]).abs().max()))
        err["logits"] = max(err["logits"], float((out["logits"][i] - m[0] @ text.double() * 100).abs().max()))
        err["bw2"] = max(err["bw2"], float((out["bw"][i] ** 2 - s["bandwidth"] ** 2).abs().max()))
        err["A"] = max(err["A"], float((out["affinity"][i] - s["affinity"]).abs().max()))
        err["y"] = max(err["y"], _y_err(out["y"][i], s["y"]))
    return err


def _assert_within(err, V, family="unit035", params=None):
    tol = {"mode": MODE_TOL, "logits": LOGIT_TOL, "bw2": BW2_TOL, "A": A_TOL, "y": Y_RTOL}
    if (params or {}).get("k_frac") == 0.0:
        tol.update(y=Y_RTOL_ONE_NEIGHBOUR)
    if family == "peaked":
        tol.update(A=A_TOL_PEAKED, y=Y_RTOL_PEAKED)
    if family == "neardup":
        # bw^2 ~ 9e-7 with ~6 % fp32 rounding in the cancelling cdist: bw^2 and y (through the density) have no
        # reference to agree with here; what must hold is a finite state and the mode
        del tol["bw2"], tol["y"]
    bad = {k: (err[k], t) for k, t in tol.items() if not err[k] <= t}
    assert not bad, f"error above tolerance: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c[0] > 1], ids=_case_id)
def test_route_matrix(jb, cuda_dev, case):
    V, C, D, _ = case
    feats, text = _inputs(jb, "unit035", V, C, D)
    _assert_within(_errors(jb, feats, text, {}, cuda_dev), V)


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["unit035", "unit1", "clusters", "neardup", "peaked"])
@pytest.mark.parametrize("shape", REPS, ids=_case_id)
def test_input_families(jb, cuda_dev, family, shape):
    V, C, D = shape
    feats, text = _inputs(jb, family, V, C, D, seed=1)
    params = {"temperature": 0.01} if family == "peaked" else {}
    _assert_within(_errors(jb, feats, text, params, cuda_dev), V, family)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(9, 1, 512), (40, 1, 512), (100, 1, 512), (9, 1, 96), (120, 1, 96)], ids=_case_id)
def test_single_class_affinity_is_one(jb, cuda_dev, shape):
    """C = 1: every softmax row is [1], so A == 1 everywhere and y follows the density alone."""
    V, C, D = shape
    feats, text = _inputs(jb, "unit035", V, C, D, seed=2)
    _assert_within(_errors(jb, feats, text, {}, cuda_dev), V)
    A = jb.blocks.mta_debug(feats.to(cuda_dev), text.to(cuda_dev))["affinity"]
    assert (A - 1).abs().max() <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("params", [
    {"th": 0.0, "max_iter": 1}, {"th": 0.0, "max_iter": 2}, {"th": 0.0, "max_iter": 8},
    {"k_frac": 0.0}, {"k_frac": 0.5}, {"k_frac": 1.0},
    {"lambda_y": 0.35}, {"lambda_q": 1.5}, {"lambda_y": 0.1, "lambda_q": 6.0, "th": 0.0, "max_iter": 3},
], ids=lambda p: "-".join(f"{k}={v}" for k, v in p.items()))
@pytest.mark.parametrize("shape", REPS, ids=_case_id)
def test_parameters(jb, cuda_dev, params, shape):
    """th = 0 fixes the iteration counts, so no early exit can flip between fp32 and float64."""
    V, C, D = shape
    feats, text = _inputs(jb, "unit035", V, C, D, seed=3)
    _assert_within(_errors(jb, feats, text, params, cuda_dev), V, params=params)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", REPS, ids=_case_id)
def test_debug_entry_point_returns_the_same_mode(jb, cuda_dev, shape):
    V, C, D = shape
    feats, text = (t.to(cuda_dev) for t in _inputs(jb, "unit035", V, C, D, seed=4))
    params = {"lambda_y": 0.3}
    mode, logits = jb.solve_mta_batched(feats, text, return_logits=True, params=params)
    dbg = jb.blocks.mta_debug(feats, text, params)
    assert torch.equal(dbg["mode"], mode) and torch.equal(dbg["logits"], logits)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in CASES if c[0] <= 2] + [(1, 403, 64, "tc+smem"), (1, 403, 96, "simt+smem"),
                                                                     (1, 1000, 512, "none+smem")], ids=_case_id)
def test_single_view_gives_the_references_nan(jb, cuda_dev, case):
    """V = 1: the reference's bandwidth averages sorted_dist[:, 1:2] of a 1 x 1 matrix, an empty slice: NaN, and so
    is everything after it.  The kernels divide 0 by 0 and land on the same; V = 2 next to it is finite."""
    V, C, D, _ = case
    feats, text = _inputs(jb, "unit035", V, C, D)
    mode = jb.solve_mta_batched(feats.to(cuda_dev), text.to(cuda_dev)).cpu()
    ref = torch.cat([o_mta(f, text, dtype=torch.float64) for f in feats])
    if V == 1:
        assert torch.isnan(ref).all() and torch.isnan(mode).all()
    else:
        assert (mode - ref).abs().max() <= MODE_TOL


def _kernels(prof):
    names = set()
    for e in prof.events():
        m = re.search(r"\b(mta_[a-z_]*kernel(?:<\d+>)?)", e.name)
        if m:
            names.add(m.group(1))
    return names


@pytest.mark.gpu
def test_routes_launch_the_expected_kernels(jb, cuda_dev):
    """Every case of the matrix takes the route it is listed under: if a dispatch threshold moves, this says so instead
    of a route silently losing its tests.  none+smem / none+scratch launch the same kernel and differ in the workspace
    they reserve."""
    from torch.profiler import ProfilerActivity, profile
    ctx = jb.get_context(cuda_dev)
    wrong = []
    for V, C, D, route in CASES:
        feats, text = (t.to(cuda_dev) for t in _inputs(jb, "unit035", V, C, D))
        ctx.trim()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            jb.blocks.mta_debug(feats, text)
            torch.cuda.synchronize()
        probs, solver = route.split("+")
        want = set({"tc": TC, "simt": ("mta_probs_kernel",), "none": ()}[probs])
        m = re.fullmatch(r"fast<(\d+)>", solver)
        want |= {f"mta_fast_kernel<{m.group(1)}>"} if m else set(BIG) if solver == "big" else {"mta_kernel<256>"}
        got = _kernels(prof)
        if got != want:
            wrong.append(((V, C, D), route, sorted(got)))
        if probs == "none" and (ctx.info()["workspace_bytes"] > 0) != (solver == "scratch"):
            wrong.append(((V, C, D), route, f"workspace {ctx.info()['workspace_bytes']} B"))
    assert not wrong, wrong


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [
    {"lambda_y": 0.0}, {"lambda_y": -0.2}, {"lambda_y": float("nan")}, {"lambda_q": float("inf")},
    {"temperature": 0.0}, {"temperature": -1.0}, {"temperature": float("inf")}, {"th": -1e-6}, {"th": float("nan")},
    {"max_iter": 0}, {"max_iter": -3}, {"k_frac": -0.1}, {"k_frac": 1.5}, {"k_frac": float("nan")},
], ids=lambda p: "-".join(f"{k}={v}" for k, v in p.items()))
def test_rejected_parameters(jb, cuda_dev, bad):
    feats, text = (t.to(cuda_dev) for t in _inputs(jb, "unit035", 9, 403, 512))
    for call in (lambda: jb.solve_mta_batched(feats, text, params=bad), lambda: jb.blocks.mta_debug(feats, text, bad)):
        with pytest.raises(jb.JcbError) as e:
            call()
        assert e.value.code == jb._capi.JCB_E_INVALID, str(e.value)


@pytest.mark.gpu
@pytest.mark.parametrize("I,V,C,D", [(-1, 9, 403, 512), (1, -1, 403, 512), (1, 0, 403, 512), (1, 2049, 403, 512),
                                     (1, 9, 0, 512), (1, 9, -403, 512), (1, 9, 403, 16), (1, 9, 403, 48),
                                     (1, 9, 403, 1056), (1, -(2 ** 31), 403, 512)])
def test_rejected_sizes(jb, cuda_dev, I, V, C, D):
    """Sizes are checked before the workspace is sized from them: a negative n_views is JCB_E_INVALID, not an
    allocation failure."""
    from ctypes import c_void_p
    ctx = jb.get_context(cuda_dev)
    buf = torch.zeros(1 << 20, device=cuda_dev)
    p = c_void_p(buf.data_ptr())
    for fn, extra in ((ctx.lib.jcb_mta, (None,)), (ctx.lib.jcb_mta_debug, (None, None, None, None))):
        rc = fn(ctx.handle, p, p, I, V, C, D, None, p, *extra)
        assert rc == jb._capi.JCB_E_INVALID, (fn.__name__, rc, ctx.lib.jcb_last_error(ctx.handle))
    ctx.sync()


def test_tolerances_have_power(jb):
    """CPU, float64 oracle: on the well-conditioned families each tolerance is at least 3x below what one deliberate
    mistake moves its quantity by, and at least 3x above the fp32 oracle's own rounding.  Keeps the tolerances from
    drifting loose (or so tight that rounding fails them).  max_iter 2 -> 1 rather than 5 -> 4: by the fifth
    iteration the solver can sit at its fixed point, where one iteration fewer moves nothing.  lambda_y x 1.0001 moves
    y by >= 8.6e-4 here while the kernels' y reaches 2.9e-4 (simt+big, none+smem): y is held to 2.5x, not 3x."""
    worst = {}

    def note(name, v, bound, power):
        ok = v >= bound if power else v <= bound
        cur = worst.get(name)
        if cur is None or (v < cur[0] if power else v > cur[0]):
            worst[name] = (v, bound, ok)

    for family in ("unit035", "unit1", "clusters"):
        for V in (33, 65, 513):
            feats, text = _inputs(jb, family, V, 403, 512, seed=5)
            k = max(int(0.3 * (V - 1)), 1)
            for x in feats:
                def run(dtype=torch.float64, **kw):
                    m, s = o_mta(x, text, True, dtype=dtype, **kw)
                    return {"mode": m[0].double(), "bw2": s["bandwidth"].double() ** 2,
                            "A": s["affinity"].double(), "y": s["y"].double()}
                ref, f32 = run(), run(torch.float32)
                ab = lambda a, b, q: float((a[q] - b[q]).abs().max())
                for q, tol in (("mode", MODE_TOL), ("bw2", BW2_TOL), ("A", A_TOL)):
                    note(f"fp32 {q}", ab(f32, ref, q), tol / 3, False)
                note("fp32 y", _y_err(f32["y"], ref["y"]), Y_RTOL / 3, False)
                note("k+1: bw2", ab(run(k_frac=(k + 1) / (V - 1) + 1e-9), ref, "bw2"), 3 * BW2_TOL, True)
                note("temperature x 1.0001: A", ab(run(temperature=1.0001), ref, "A"), 3 * A_TOL, True)
                note("lambda_y x 1.0001: y", _y_err(run(lambda_y=0.2 * 1.0001)["y"], ref["y"]), 2.5 * Y_RTOL, True)
                it2, it1 = run(th=0.0, max_iter=2), run(th=0.0, max_iter=1)
                note("max_iter 2 -> 1: mode", ab(it1, it2, "mode"), 3 * MODE_TOL, True)
                note("max_iter 2 -> 1: y", _y_err(it1["y"], it2["y"]), 3 * Y_RTOL, True)
    bad = {k: v for k, v in worst.items() if not v[2]}
    assert not bad, bad
