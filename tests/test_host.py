"""Host-side logic that needs no GPU: API surface parity with the reference, error behaviour,
the non-OT matchers (pure elementwise torch) against the golden vectors, NumPy-contract sampling,
shard arithmetic and the world_size-2 gloo path of the index all-gather."""
import inspect
import json
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import cfm_b200
from cfm_b200 import dist as cdist
from cfm_b200.optimal_transport import OTPlanSampler, wasserstein
from conftest import ROOT


def test_ctor_contract():
    s = OTPlanSampler("sinkhorn", reg=0.3, reg_m=2.0, normalize_cost=True, num_threads="max", warn=False)
    assert (s.reg, s.reg_m, s.normalize_cost, s.warn) == (0.3, 2.0, True, False)
    assert callable(s.ot_fn)
    with pytest.raises(ValueError, match="Unknown method: nope"):
        OTPlanSampler("nope")
    for m in ("unbalanced", "partial"):  # accepted like the reference; solving is out of scope
        with pytest.raises(NotImplementedError):
            OTPlanSampler(m).ot_fn(None, None, None)
    with pytest.raises(ValueError):
        wasserstein(torch.zeros(2, 2), torch.zeros(2, 2), "noname")
    with pytest.raises(ValueError):
        cfm_b200.SchrodingerBridgeConditionalFlowMatcher(sigma=0.0)
    with pytest.warns(UserWarning):
        cfm_b200.SchrodingerBridgeConditionalFlowMatcher(sigma=1e-4)
    fm = cfm_b200.SchrodingerBridgeConditionalFlowMatcher(sigma=0.5, ot_method="sinkhorn")
    assert fm.ot_method == "sinkhorn" and fm.ot_sampler.reg == 2 * 0.5**2
    assert cfm_b200.ExactOptimalTransportConditionalFlowMatcher().ot_sampler.method == "exact"


def test_signatures_match_reference_source():
    """Compare public signatures with the reference *source*, as parsed by tests/golden/make_golden_reference_checks.py
    into tests/golden/reference_signatures.json ("Class.method" or "function" -> positional parameters)."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_signatures.json")) as f:
        ref = {tuple(k.split(".")) if "." in k else ("", k): v for k, v in json.load(f).items()}
    assert len(ref) >= 20 and ("OTPlanSampler", "sample_plan") in ref and ("", "pad_t_like_x") in ref
    import cfm_b200.conditional_flow_matching as m_cfm
    import cfm_b200.models as m_models
    import cfm_b200.optimal_transport as m_ot
    for (cls, fn), args in ref.items():
        if cls == "":
            mod = m_ot if hasattr(m_ot, fn) else m_cfm
            obj = getattr(mod, fn)
        else:
            owner = next(getattr(m, cls) for m in (m_ot, m_cfm, m_models) if hasattr(m, cls))
            obj = getattr(owner, fn)
        mine = [p for p, v in inspect.signature(obj).parameters.items()
                if v.kind in (v.POSITIONAL_ONLY, v.POSITIONAL_OR_KEYWORD)]
        if cls and "self" not in mine:
            mine = ["self"] + mine
        assert mine == args, (cls, fn, mine, args)


@pytest.mark.parametrize("kind,cls", [("i_cfm", "ConditionalFlowMatcher"),
                                      ("t_cfm", "TargetConditionalFlowMatcher"),
                                      ("vp_cfm", "VariancePreservingConditionalFlowMatcher")])
def test_non_ot_matchers_bit_exact_vs_reference_vectors(golden, kind, cls):
    fm = getattr(cfm_b200, cls)(0.5)
    x0, x1 = torch.from_numpy(golden["fm_x0"]), torch.from_numpy(golden["fm_x1"])
    torch.manual_seed(1994)
    t, xt, ut, eps = fm.sample_location_and_conditional_flow(x0, x1, return_noise=True)
    for name, val in (("t", t), ("xt", xt), ("ut", ut), ("eps", eps)):
        assert torch.equal(val, torch.from_numpy(golden[f"fm_{kind}_{name}"])), name
    np.testing.assert_array_equal(np.asarray(fm.compute_lambda(t)), golden[f"fm_{kind}_lambda"])
    t2, *_ = fm.sample_location_and_conditional_flow(x0, x1, t=t)
    assert t2 is t
    with pytest.raises(AssertionError):
        fm.sample_location_and_conditional_flow(x0, x1, t=t[:5])


def test_pad_t_like_x():
    x = torch.zeros(7, 2, 3, 4)
    assert cfm_b200.pad_t_like_x(torch.arange(7.0), x).shape == (7, 1, 1, 1)
    assert cfm_b200.pad_t_like_x(0.3, x) == 0.3 and cfm_b200.pad_t_like_x(2, x) == 2


def test_sample_map_numpy_contract():
    """reference tests/test_optimal_transport.py:15-29: a permutation plan drawn without
    replacement returns every entry exactly once; with replacement it follows np.random.choice."""
    s = OTPlanSampler("exact")
    n = 128
    perm = np.random.default_rng(0).permutation(np.eye(n), axis=1)
    i, j = s.sample_map(perm, batch_size=n, replace=False)
    rec = np.zeros((n, n))
    rec[i, j] = 1
    assert np.array_equal(rec, perm)
    pi = np.random.default_rng(1).random((16, 24))
    np.random.seed(4)
    i, j = s.sample_map(pi, 50)
    np.random.seed(4)
    k = np.random.choice(pi.size, p=pi.flatten() / pi.sum(), size=50)
    assert np.array_equal(i, k // 24) and np.array_equal(j, k % 24)


def test_mlp_state_dict_and_cpu_autograd_path():
    m = cfm_b200.MLP(dim=2, time_varying=True, w=64)
    assert list(m.state_dict()) == [f"net.{i}.{p}" for i in (0, 2, 4, 6) for p in ("weight", "bias")]
    assert m.net[0].in_features == 3 and isinstance(m.net[1], torch.nn.SELU)
    y = m(torch.randn(5, 3))
    y.sum().backward()  # training path stays a plain nn.Sequential
    assert m.net[0].weight.grad is not None
    w = cfm_b200.torch_wrapper(m)
    assert w.model is m and w(torch.tensor(0.3), torch.randn(5, 2)).shape == (5, 2)
    with pytest.raises(TypeError):
        cfm_b200.NeuralODE(torch.nn.Linear(2, 2)).trajectory(torch.zeros(1, 2), torch.linspace(0, 1, 2))


def test_hot_path_refuses_to_run_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from cfm_b200._ffi import CfmLibraryError
    with pytest.raises(CfmLibraryError):
        OTPlanSampler("exact").sample_plan(torch.randn(8, 2), torch.randn(8, 2))
    m = cfm_b200.MLP(dim=2, time_varying=True)
    with pytest.raises(CfmLibraryError):
        cfm_b200.NeuralODE(cfm_b200.torch_wrapper(m)).trajectory(torch.zeros(4, 2), torch.linspace(0, 1, 2))
    with pytest.raises(CfmLibraryError), torch.no_grad():  # sampling regime on CPU tensors: no silent PyTorch fallback
        m(torch.zeros(4, 3))
    with pytest.raises(CfmLibraryError), torch.no_grad():
        cfm_b200.torch_wrapper(m)(torch.tensor(0.5), torch.zeros(4, 2))
    assert m(torch.zeros(4, 3)).requires_grad  # training path (autograd on): plain PyTorch, any device
    with pytest.raises(CfmLibraryError):
        cfm_b200.CouplingStream(OTPlanSampler("sinkhorn"))
    with pytest.raises(CfmLibraryError):
        OTPlanSampler("exact").sample_trajectory(torch.randn(8, 3, 2))


def test_coupling_stream_argument_contract():
    with pytest.raises(ValueError):
        cfm_b200.CouplingStream(OTPlanSampler("exact"), depth=0)


def test_compat_alias():
    import cfm_b200.compat as compat
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("torchcfm", "torchdyn")}
    try:
        compat.install_as_torchcfm()
        from torchcfm.conditional_flow_matching import ExactOptimalTransportConditionalFlowMatcher as E
        from torchcfm.models import MLP
        from torchcfm.optimal_transport import OTPlanSampler as O
        from torchcfm.utils import torch_wrapper  # noqa: F401
        from torchdyn.core import NeuralODE
        assert E is cfm_b200.ExactOptimalTransportConditionalFlowMatcher and O is OTPlanSampler
        assert MLP is cfm_b200.MLP and NeuralODE is cfm_b200.NeuralODE
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] in ("torchcfm", "torchdyn")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_shard_bounds_partition():
    for n, ws in ((16384, 4), (8192, 8), (10, 3), (5, 8)):
        cuts = [cdist.shard_bounds(n, ws, r) for r in range(ws)]
        assert cuts[0][0] == 0 and cuts[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
        assert max(h - l for l, h in cuts) - min(h - l for l, h in cuts) <= 1


def _gloo_worker(rank, world, port, n_local, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sizes = n_local if isinstance(n_local, (list, tuple)) else [n_local] * world
        n = sizes[rank]
        x0, x1 = torch.zeros(n, 3), torch.zeros(n, 3)

        def fake_pairs(a, b):  # deterministic stand-in for the device coupling
            idx = torch.arange(a.shape[0])
            return idx, (idx * 7 + rank) % a.shape[0]

        i, j, ig, jg = cdist.sharded_sample_pairs(None, x0, x1, pair_fn=fake_pairs,
                                                  equal_shards=len(set(sizes)) == 1)
        q.put((rank, i.tolist(), j.tolist(), ig.tolist(), jg.tolist()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("sizes", [[6, 6], [5, 3]])
def test_sharded_pairs_gloo_world2(sizes):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + len(sizes) + sizes[1]
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, sizes, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    want_i, want_j, off = [], [], 0
    for r, n in enumerate(sizes):
        want_i += [off + k for k in range(n)]
        want_j += [off + (k * 7 + r) % n for k in range(n)]
        off += n
    for rank, i, j, ig, jg in res:
        assert i == list(range(sizes[rank]))
        assert ig == want_i and jg == want_j


# ---- property tests (hypothesis) of the pure-host pieces -----------------------------------------------
from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=200, deadline=None)
@given(st.integers(0, 100000), st.integers(1, 64))
def test_shard_bounds_properties(n, ws):
    cuts = [cdist.shard_bounds(n, ws, r) for r in range(ws)]
    assert cuts[0][0] == 0 and cuts[-1][1] == n
    assert all(lo <= hi for lo, hi in cuts)
    assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
    sizes = [hi - lo for lo, hi in cuts]
    assert max(sizes) - min(sizes) <= 1 and sum(sizes) == n


@settings(max_examples=60, deadline=None)
@given(st.integers(1, 9), st.lists(st.integers(1, 4), min_size=0, max_size=3), st.floats(0.0, 2.0),
       st.sampled_from(["i_cfm", "t_cfm", "vp_cfm"]), st.integers(0, 2**31 - 1))
def test_non_ot_matchers_equal_the_oracle_formulas_on_any_shape(bs, dims, sigma, kind, seed):
    """The CPU (autograd / non-fused) branch of the non-OT matchers against the oracle's restatement of the
    reference formulas, bit for bit, for arbitrary trailing shapes (the fused CUDA branch is tested on the GPU)."""
    from oracle import coupling as oc
    cls = {"i_cfm": cfm_b200.ConditionalFlowMatcher, "t_cfm": cfm_b200.TargetConditionalFlowMatcher,
           "vp_cfm": cfm_b200.VariancePreservingConditionalFlowMatcher}[kind]
    g = torch.Generator().manual_seed(seed)
    shape = (bs, *dims) if dims else (bs, 1)
    x0, x1 = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    t = torch.rand(bs, generator=g)
    fm = cls(sigma=sigma)
    torch.manual_seed(seed % 1000)
    tt, xt, ut, eps = fm.sample_location_and_conditional_flow(x0, x1, t=t, return_noise=True)
    want_xt, want_ut = oc.matcher_xt_ut(kind, x0, x1, t, eps, sigma)
    assert torch.equal(tt, t) and torch.equal(xt, want_xt) and torch.equal(ut, want_ut)
    lam = fm.compute_lambda(t)
    assert torch.is_tensor(lam) or isinstance(lam, float)


@settings(max_examples=50, deadline=None)
@given(st.integers(1, 6), st.lists(st.integers(1, 5), min_size=0, max_size=4))
def test_pad_t_like_x_broadcasts(bs, dims):
    x = torch.zeros((bs, *dims))
    t = torch.arange(bs, dtype=torch.float32)
    p = cfm_b200.pad_t_like_x(t, x)
    assert p.shape == (bs,) + (1,) * len(dims)
    assert (p * torch.ones_like(x) if dims else p).shape == x.shape
    assert cfm_b200.pad_t_like_x(0.5, x) == 0.5


def _gloo_traj_worker(rank, world, port, n, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = torch.arange(n * 2, dtype=torch.float32).reshape(n, 2)
        span = torch.linspace(0, 1, 3)

        def fake_integrate(xs, ts):  # row-wise, shard-independent stand-in for NeuralODE.trajectory
            return torch.stack([xs * (1.0 + float(t)) for t in ts])

        full = cdist.sharded_trajectory(None, x, span, integrate_fn=fake_integrate)
        local = cdist.sharded_trajectory(None, x, span, gather=False, integrate_fn=fake_integrate)
        q.put((rank, full.tolist(), list(local.shape)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n", [8, 7])
def test_sharded_trajectory_gloo_world2(n):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000) + n
    procs = [ctx.Process(target=_gloo_traj_worker, args=(r, 2, port, n, q)) for r in range(2)]
    [p.start() for p in procs]
    res = sorted(q.get(timeout=120) for _ in range(2))
    [p.join(60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    x = torch.arange(n * 2, dtype=torch.float32).reshape(n, 2)
    want = torch.stack([x * (1.0 + float(t)) for t in torch.linspace(0, 1, 3)]).tolist()
    for rank, full, lshape in res:
        assert full == want
        lo, hi = cdist.shard_bounds(n, 2, rank)
        assert lshape == [3, hi - lo, 2]


# ------------------------------------------------------------------ facts the kernels rely on (CPU, no library calls)
def _eval_c_fraction_table(text):
    """A brace initialiser of rk_tableau.h ('{1.f / 5, 0, ...}', '(float)(35.0 / 384 - ...)') -> nested lists of
    floats rounded to fp32 the way the C compiler rounds them."""
    import re
    t = text.replace("\\\n", " ")
    t = re.sub(r"\(float\)", "", t)
    t = re.sub(r"(\d+(?:\.\d*)?)f\b", r"\1", t)
    t = t.replace("{", "[").replace("}", "]")
    return eval(t, {"__builtins__": {}})


def test_rk_tableau_header_is_the_oracles_dormand_prince_tableau():
    """csrc/rk_tableau.h feeds both rk.cu's device constants and the stage row cfm_mlp_forward_rkstage_f32 hands to the
    fused MLP kernel: every coefficient equals the oracle's (SciPy-pinned) Dormand-Prince tableau rounded to fp32."""
    import re
    from oracle import vector_field as vf
    src = open(os.path.join(ROOT, "cfm_b200", "csrc", "rk_tableau.h")).read()

    def macro(name):
        m = re.search(r"#define\s+" + name + r"\s+(.*?)(?=\n#define|\n/\*|\Z)", src, re.S)
        assert m, name
        return _eval_c_fraction_table(m.group(1).strip())

    c, a, e = macro("CFM_RK_C_INIT"), macro("CFM_RK_A_INIT"), macro("CFM_RK_E_INIT")
    f32 = lambda v: float(np.float32(v))  # noqa: E731
    assert [f32(v) for v in c] == [f32(v) for v in vf._C]
    for s in range(7):
        row = list(vf._A[s]) + [0.0] * (6 - len(vf._A[s]))
        # the header writes e.g. 44.f / 45: an fp32 quotient of exactly representable integers == fp32(44 / 45)
        assert [f32(v) for v in a[s]] == [f32(v) for v in row], s
    assert [f32(v) for v in e] == [f32(v) for v in vf._BERR]


def test_seeded_screening_bound_holds_on_sinkhorn_iterates():
    """The float64-potential Sinkhorn solver skips terms below  previous LSE + min(change of the other potential) - 34:
    that is safe because the new log-sum-exp of every row (column) is bounded below by the previous one plus that
    minimum.  Checked on real iterates of the oracle's log-domain solver, together with the size of the support the
    threshold leaves (the reason the screening pays)."""
    from scipy.special import logsumexp
    rng = np.random.default_rng(0)
    n, d = 300, 64
    x0, x1 = rng.standard_normal((n, d)), rng.standard_normal((n, d))
    M = ((x0[:, None, :] - x1[None, :, :]) ** 2).sum(-1).astype(np.float32)
    Mr = (-M / np.float32(0.1)).astype(np.float32).astype(np.float64)
    u, v = np.zeros(n), -np.log(n) - logsumexp(Mr, axis=0)
    lse_r_prev = None
    for it in range(12):
        lse_r = logsumexp(Mr + v[None, :], axis=1)
        if lse_r_prev is not None:
            assert (lse_r >= lse_r_prev + dv.min() - 1e-9).all()            # rows: bound with the v change
            thr = lse_r_prev + dv.min() - 34.0
            kept = (Mr + v[None, :] > thr[:, None])
            dropped = np.where(kept, -np.inf, Mr + v[None, :])
            assert (logsumexp(dropped, axis=1) - lse_r).max() < -25.0         # what is skipped is < e^-25 of the result
            assert kept.sum() < 0.05 * n * n                                  # ... and almost everything is skipped
        u_new = -np.log(n) - lse_r
        du = u_new - u
        lse_c_prev = -np.log(n) - v                                           # LSE_j(Mr + u_old) that produced v
        lse_c = logsumexp(Mr + u_new[:, None], axis=0)
        assert (lse_c >= lse_c_prev + du.min() - 1e-9).all()                  # columns: bound with the u change
        v_new = -np.log(n) - lse_c
        dv, u, v, lse_r_prev = v_new - v, u_new, v_new, lse_r


def test_fp16x3_operand_split_emulation():
    """The fp16x3 scheme of csrc/gemm_h3.cuh in NumPy: hi = fp16(x), lo = fp16((x - hi) 2^11), and
    acc0 = sum hi.hi, acc1 = sum (hi.lo + lo.hi), result acc0 + acc1 2^-11 (products of fp16 numbers are exact in the
    fp32 the tensor core accumulates in; only lo.lo, 2^-22 relative, is dropped).  Pins the accuracy DESIGN.md 3.0
    quotes for the representation itself -- 2.7e-8 of sum|a||b| at d = 784 -- against the 3xTF32 split of round 1, and
    the power-of-two row scaling that keeps unbounded inputs inside fp16's range exactly."""
    rng = np.random.default_rng(3)
    n, d = 64, 784
    a = rng.standard_normal((n, d)).astype(np.float32)
    b = (rng.standard_normal((n, d)) + 0.3).astype(np.float32)

    def split_h3(x):
        hi = x.astype(np.float16)
        lo = ((x - hi.astype(np.float32)) * np.float32(2048.0)).astype(np.float16)
        return hi.astype(np.float64), lo.astype(np.float64)

    def tf32_trunc(x):
        return (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)

    exact = a.astype(np.float64) @ b.astype(np.float64).T
    scale = np.abs(a).astype(np.float64) @ np.abs(b).astype(np.float64).T
    ah, al = split_h3(a)
    bh, bl = split_h3(b)
    h3 = ah @ bh.T + (ah @ bl.T + al @ bh.T) / 2048.0
    err_h3 = (np.abs(h3 - exact) / scale).max()
    a_hi = tf32_trunc(a); a_lo = tf32_trunc(a - a_hi)
    b_hi = tf32_trunc(b); b_lo = tf32_trunc(b - b_hi)
    t3 = (a_hi.astype(np.float64) @ b_hi.astype(np.float64).T + a_hi.astype(np.float64) @ b_lo.astype(np.float64).T
          + a_lo.astype(np.float64) @ b_hi.astype(np.float64).T)
    err_t3 = (np.abs(t3 - exact) / scale).max()
    assert err_h3 < 6e-8 and err_h3 < err_t3, (err_h3, err_t3)
    # rows scaled by exact powers of two (what the cost path does for unbounded data): same result, no overflow
    big = a * np.float32(3.0e5)
    s = np.exp2(np.floor(np.log2(32768.0 / np.abs(big).max(1)))).astype(np.float32)  # row max -> [16384, 32768)
    assert np.isfinite((big * s[:, None]).astype(np.float16)).all()
    gh, gl = split_h3(big * s[:, None])
    h3s = (gh @ bh.T + (gh @ bl.T + gl @ bh.T) / 2048.0) / s[:, None].astype(np.float64)
    exact_big = big.astype(np.float64) @ b.astype(np.float64).T
    assert (np.abs(h3s - exact_big) / (np.abs(big).astype(np.float64) @ np.abs(b).astype(np.float64).T)).max() < 6e-8
