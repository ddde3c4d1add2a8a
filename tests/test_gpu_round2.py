"""Round-2 parity tests (GPU, through the C ABI): the fp16x3 tensor-core paths (cost matrix, fused MLP), the
row-normalised pair draw at large |M/reg|, status words under warn=False, rectangular exact OT, full-size C2 against
the kernel-space oracle, and the B = 10 000 MLP against reference-generated vectors."""
import os

import numpy as np
import pytest
import torch

import cfm_b200
from cfm_b200 import _ffi
from cfm_b200.optimal_transport import OTPlanSampler, wasserstein
from oracle import coupling as oc
from oracle import ot as oot
from oracle import vector_field as vf

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gpu_cost(x0, x1, squared=True, algo=1):
    s = OTPlanSampler("exact", cost_algo=algo)
    M, cmax, n0, n1 = s._cost(x0.to(DEV), x1.to(DEV), torch.device(DEV), squared=squared)
    return M[:, :n1].cpu(), float(cmax.item())


# ------------------------------------------------------------------------- cost matrix, fp16x3 scheme
@pytest.mark.parametrize("n0,n1,d", [(256, 256, 32), (128, 512, 64), (300, 200, 36), (1024, 1024, 784),
                                     (130, 257, 100), (2048, 4096, 128), (8192, 256, 784)])
def test_cost_matrix_fp16x3_vs_simt_and_cdist(n0, n1, d):
    """kind::f16 tensor-core path (x = hi + lo 2^-11, two accumulators): fp32-grade agreement with the SIMT
    fp32-FMA path and with torch.cdist, same gate as the 3xTF32 path it replaces."""
    g = torch.Generator().manual_seed(n0 + n1 + d)
    x0, x1 = torch.randn(n0, d, generator=g), torch.randn(n1, d, generator=g) + 0.25
    simt, _ = gpu_cost(x0, x1, algo=1)
    h3, cmax = gpu_cost(x0, x1, algo=3)
    ref = oc.cost_matrix(x0, x1)
    scale = (x0.pow(2).sum(1).max() + x1.pow(2).sum(1).max()).item()
    assert (h3 - simt).abs().max().item() <= 2.5e-6 * scale
    assert (h3 - ref).abs().max().item() <= 2.5e-6 * scale
    assert cmax == h3.max().item() and (h3 >= 0).all()
    if n0 * n1 >= 256 * 256:  # auto mode (cost_algo=0) of a Sinkhorn sampler = the fp16x3 path from this size on
        sk = OTPlanSampler("sinkhorn")
        Ma, _, _, _ = sk._cost(x0.to(DEV), x1.to(DEV), torch.device(DEV))
        assert torch.equal(Ma[:, :n1].cpu(), h3)
    un, _ = gpu_cost(x0, x1, squared=False, algo=3)
    assert (un - torch.cdist(x0, x1)).abs().max().item() <= 1e-5 * max(1.0, ref.max().sqrt().item())


@pytest.mark.parametrize("kind", ["huge", "tiny", "mixed_rows", "images"])
def test_cost_matrix_fp16x3_dynamic_range(kind):
    """fp16 overflows at 65504: the pre-pass scales every row by a power of two (exact), so the data range is
    the caller's business exactly as in fp32."""
    g = torch.Generator().manual_seed(11)
    x0, x1 = torch.randn(384, 64, generator=g), torch.randn(256, 64, generator=g)
    if kind == "huge":
        x0, x1 = x0 * 3.0e6, x1 * 3.0e6
    elif kind == "tiny":
        x0, x1 = x0 * 1.0e-9, x1 * 1.0e-9
    elif kind == "mixed_rows":
        x0 = x0 * torch.logspace(-6, 6, 384)[:, None]
        x1 = x1 * torch.logspace(5, -5, 256)[:, None]
    else:
        x0, x1 = (x0.abs() * 80).clamp(0, 255).round(), (x1.abs() * 80).clamp(0, 255).round()
    h3, _ = gpu_cost(x0, x1, algo=3)
    ref = (x0.double()[:, None, :] - x1.double()[None, :, :]).pow(2).sum(-1)
    scale = x0.double().pow(2).sum(1)[:, None] + x1.double().pow(2).sum(1)[None, :]
    assert torch.isfinite(h3).all()
    assert ((h3.double() - ref).abs() / scale).max().item() <= 2.5e-6


# ------------------------------------------------------------------------- pair draw at large |M/reg|
@pytest.mark.parametrize("n,d,reg,normalize", [(512, 512, 0.1, False), (256, 2, 0.5, False), (256, 2, 0.02, False),
                                                (384, 64, 0.05, True)])
def test_fast_draw_large_cost_over_reg(n, d, reg, normalize):
    """ADVICE r1 (high): the uniform-rows draw used to normalise a row's weights by lv_0 only; its exponent is
    O(M/reg) and under/overflowed fp32 for whole rows (512 of 512 rows at d=512, reg=0.1), silently drawing uniform
    partners.  Now the weights are the plan entries themselves (exponent <= 0): flags stay 0 and the draws are
    those of the float64 row cdf."""
    g = torch.Generator().manual_seed(n + d)
    x0, x1 = torch.randn(n, d, generator=g), torch.randn(n, d, generator=g)
    s = OTPlanSampler("sinkhorn", reg=reg, normalize_cost=normalize, num_iter_max=200, stop_thr=0.0, warn=False)
    dev = torch.device(DEV)
    cp = s._couple(x0.to(DEV), x1.to(DEV), dev)
    u = np.random.RandomState(3).random_sample(n)
    i, j = s._draw(cp, n, torch.from_numpy(u).to(DEV))
    st = cp.status.cpu().tolist()
    assert st[0] & _ffi.FLAG_NONFINITE == 0, st
    # float64 reference of the same inversion from the device's own M and potentials
    M = cp.M[:, :n].double().cpu().numpy()
    if normalize:
        M = (cp.M[:, :n] / cp.cost_max).double().cpu().numpy()
    Mr = -(M.astype(np.float32) / np.float32(reg)).astype(np.float64)
    logp = Mr + cp.log_u.cpu().numpy()[:, None] + cp.log_v.cpu().numpy()[None, :]
    rows = np.minimum((u * n).astype(np.int64), n - 1)
    frac = u * n - rows
    same = 0
    jg = j.cpu().numpy()
    assert np.array_equal(i.cpu().numpy(), rows)
    for k in range(n):
        w = np.exp(logp[rows[k]] - logp[rows[k]].max())
        cdf = np.cumsum(w)
        want = min(int(np.searchsorted(cdf, frac[k] * cdf[-1], side="right")), n - 1)
        same += int(want == jg[k])
    assert same >= int(0.995 * n), (same, n)  # fp32 weights: a draw may differ only on a cdf boundary
    if reg <= 0.1 and not normalize:
        # a peaked plan: the drawn partner carries a visible share of its row's mass (an independent, uniform
        # partner -- what the underflowed rows used to get -- would carry ~1/n)
        from scipy.special import logsumexp
        share = np.exp(logp[rows, jg] - logsumexp(logp[rows], axis=1))
        assert np.median(share) > 5.0 / n


def test_row_conditional_draw_without_log_u():
    """cfm_plan_sample_rows with log_u == NULL centres the exponents with a row-maximum pass."""
    n = 256
    g = torch.Generator().manual_seed(9)
    x0, x1 = torch.randn(n, 128, generator=g), torch.randn(n, 128, generator=g)
    s = OTPlanSampler("sinkhorn", reg=0.1, num_iter_max=100, stop_thr=0.0, warn=False)
    cp = s._couple(x0.to(DEV), x1.to(DEV), torch.device(DEV))
    rows = torch.arange(n, dtype=torch.int64, device=DEV)
    u = torch.from_numpy(np.random.RandomState(1).random_sample(n)).to(DEV)
    with_u = s._draw_rows(cp, rows, u)
    nxt = torch.empty(n, dtype=torch.int64, device=DEV)
    _ffi.check(_ffi.lib().cfm_plan_sample_rows(
        _ffi.ptr(cp.M), cp.n0, cp.n1, cp.M.stride(0), cp.reg, _ffi.ptr(cp.cost_max), 0, None, _ffi.ptr(cp.log_v),
        _ffi.ptr(rows), _ffi.ptr(u), n, _ffi.ptr(nxt), _ffi.ptr(cp.status), _ffi.stream_ptr(torch.device(DEV))),
        "cfm_plan_sample_rows")
    assert cp.status.cpu()[0].item() & _ffi.FLAG_NONFINITE == 0
    assert (with_u == nxt).float().mean().item() >= 0.99


# ------------------------------------------------------------------------- status words with warn=False
def test_status_is_evaluated_with_warn_false(capsys):
    """ADVICE r1 (medium): ``warn`` gates only warnings.warn; infeasible exact OT still raises and a non-finite
    Sinkhorn plan still prints, and no index leaves its range."""
    x0 = torch.randn(64, 4)
    x1 = torch.randn(64, 4)
    x1[3, 2] = float("nan")
    s = OTPlanSampler("exact", warn=False)
    with pytest.raises(RuntimeError):
        s.sample_plan(x0.to(DEV), x1.to(DEV))
    with pytest.raises(RuntimeError):
        s.sample_pairs(x0.to(DEV), x1.to(DEV))
    torch.cuda.synchronize()  # no sticky error: the device is still usable
    sk = OTPlanSampler("sinkhorn", reg=0.05, warn=False, num_iter_max=20, stop_thr=0.0)
    a, b = sk.sample_plan(x0.to(DEV), x1.to(DEV))
    assert a.shape == (64, 4)
    info = sk.last_info  # resolves the deferred status word
    assert info["flags"] & _ffi.FLAG_NONFINITE
    assert "ERROR: p is not finite" in capsys.readouterr().out
    # a healthy warn=False call leaves a clean status and needs no synchronisation inside the call
    ok = OTPlanSampler("sinkhorn", reg=0.05, normalize_cost=True, warn=False, num_iter_max=30, stop_thr=0.0)
    ok.sample_plan(torch.randn(128, 8).to(DEV), torch.randn(128, 8).to(DEV))
    assert len(ok._pending) == 1
    assert ok.last_info["flags"] & (_ffi.FLAG_NONFINITE | _ffi.FLAG_ZERO_MASS) == 0 and len(ok._pending) == 0


# ------------------------------------------------------------------------- rectangular exact OT
@pytest.mark.parametrize("n0,n1,d", [(6, 9, 2), (12, 8, 3), (64, 96, 2), (100, 40, 5), (128, 256, 16)])
def test_exact_ot_unequal_batch_sizes_vs_lp_oracle(n0, n1, d):
    """pot.emd takes marginals of any two sizes (reference :79,87).  The device solves the lcm(n0, n1)-replicated
    assignment problem; the oracle solves the transport LP itself (SciPy HiGHS): same plan, same cost."""
    g = torch.Generator().manual_seed(n0 * 1000 + n1)
    x0, x1 = torch.randn(n0, d, generator=g), torch.randn(n1, d, generator=g)
    s = OTPlanSampler("exact")
    P = s.get_map(x0.to(DEV), x1.to(DEV))
    M = oc.cost_matrix(x0, x1).numpy()
    G = oot.emd(oot.unif(n0), oot.unif(n1), M)
    assert P.shape == (n0, n1) and P.dtype == np.float64
    np.testing.assert_allclose(P.sum(1), 1.0 / n0, rtol=1e-12)
    np.testing.assert_allclose(P.sum(0), 1.0 / n1, rtol=1e-12)
    np.testing.assert_allclose(P, G, atol=1e-12)
    w2 = wasserstein(x0.to(DEV), x1.to(DEV), method="exact", power=2)
    assert abs(w2 - float(np.sqrt((G * M.astype(np.float64)).sum()))) <= 1e-6 * max(1.0, w2)
    # sample_plan draws x0.shape[0] pairs from that plan with the reference's own host draw
    np.random.seed(5)
    a, b = s.sample_plan(x0.to(DEV), x1.to(DEV))
    np.random.seed(5)
    i, j = s.sample_map(P, n0)
    assert torch.equal(a.cpu(), x0[i]) and torch.equal(b.cpu(), x1[j])
    assert (P[i, j] > 0).all()


def test_exact_ot_unequal_sizes_too_large_is_refused():
    s = OTPlanSampler("exact")
    with pytest.raises(NotImplementedError):
        s.get_map(torch.randn(255, 2).to(DEV), torch.randn(256, 2).to(DEV))


# ------------------------------------------------------------------------- C2 at full size vs the oracle
def test_c2_full_size_against_kernel_space_oracle():
    """BASELINE config 2 at full size (N = 8192, d = 784, reg = 0.05, normalised cost, 100 iterations): the
    device potentials against the float64 kernel-space Sinkhorn-Knopp oracle (what OTPlanSampler('sinkhorn')
    calls in the reference) run on the device's own cost matrix.  Gate: marginals of the implied plans within
    1e-5 relative (north_star), plan entries within 1e-4 of the largest entry."""
    N, D, REG, ITERS = 8192, 784, 0.05, 100
    g = torch.Generator().manual_seed(0)
    x0, x1 = torch.randn(N, D, generator=g), torch.randn(N, D, generator=g)
    s = OTPlanSampler("sinkhorn", reg=REG, normalize_cost=True, num_iter_max=ITERS, stop_thr=0.0, warn=False)
    cp = s._couple(x0.to(DEV), x1.to(DEV), torch.device(DEV))
    Mn = (cp.M[:, :N] / cp.cost_max).cpu().numpy()  # fp32, the oracle's input (cost parity is gated separately)
    lu, lv = cp.log_u.cpu().numpy(), cp.log_v.cpu().numpy()
    # oracle: POT sinkhorn_knopp dtype pattern, exactly ITERS iterations (stopThr = 0)
    a = b = np.ones(N) / N
    K = np.exp(Mn / (-REG))
    Kp = (1 / a).reshape(-1, 1) * K
    u = np.ones(N, dtype=Mn.dtype) / N
    for _ in range(ITERS):
        v = b / np.dot(K.T, u)
        u = 1.0 / np.dot(Kp, v)
    P_ref_rows = u * (K @ v)
    P_ref_cols = v * (K.T @ u)
    Mr = -(Mn / np.float32(REG)).astype(np.float64)
    P = np.exp(Mr + lu[:, None] + lv[None, :])
    assert np.abs(P.sum(1) / P_ref_rows - 1).max() <= 1e-5
    assert np.abs(P.sum(0) / P_ref_cols - 1).max() <= 1e-5
    sel = np.random.RandomState(0).randint(0, N, size=64)
    P_ref = u[sel, None] * K[sel] * v[None, :]
    assert np.abs(P[sel] - P_ref).max() <= 1e-4 * P_ref.max()
    assert int(cp.status[1].item()) == ITERS


# ------------------------------------------------------------------------- MLP, tensor-core paths
def _mlp784():
    torch.manual_seed(0)
    m = cfm_b200.MLP(dim=784, w=256, time_varying=True)  # same init stream as the reference MLP
    return m


def _x10k():
    g = torch.Generator().manual_seed(2024)
    return torch.randn(10000, 784, generator=g)


@pytest.mark.parametrize("fused", [1, 0])
def test_mlp_b10000_tensor_core_vs_reference_vectors(fused, tmp_path):
    """BASELINE config 3's forward at the full batch through the tcgen05 paths -- the fused persistent kernel
    and the per-layer launches -- against vectors generated by the unmodified reference MLP
    (tests/golden/make_golden_mlp10k.py): 96 whole rows, all row sums, all column sums.  Gate: 1e-5 of max|y|."""
    gold = dict(np.load(os.path.join(GOLD, "mlp10k_vectors.npz")))
    m = _mlp784()
    np.testing.assert_array_equal(m.net[0].weight[:2, :4].detach().numpy(), gold["w0_probe"])  # same weights
    m = m.to(DEV)
    x = _x10k().to(DEV)
    if not fused:
        # the switch is read once per process by the library: run the per-layer variant in a fresh interpreter
        import subprocess, sys, textwrap
        code = textwrap.dedent("""
            import os, sys, numpy as np, torch
            sys.path.insert(0, %r)
            import cfm_b200
            torch.manual_seed(0)
            m = cfm_b200.MLP(dim=784, w=256, time_varying=True).to("cuda:0")
            g = torch.Generator().manual_seed(2024)
            x = torch.randn(10000, 784, generator=g).to("cuda:0")
            with torch.no_grad():
                y = m.vector_field(0.37, x)
            np.save(sys.argv[1], y.cpu().numpy())
        """ % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        out = str(tmp_path / "mlp10k_perlayer.npy")
        env = dict(os.environ, CFM_MLP_FUSED="0")
        subprocess.run([sys.executable, "-c", code, out], check=True, env=env, timeout=300)
        y = np.load(out).astype(np.float64)
    else:
        assert m.tc_path(10000)
        with torch.no_grad():
            y = m.vector_field(float(gold["t"]), x).double().cpu().numpy()
    amax = float(gold["abs_max"])
    assert np.abs(y[gold["rows"]] - gold["y64_rows"]).max() / amax <= 1e-5
    assert np.abs(y.sum(1) - gold["row_sums"]).max() / (amax * 784 ** 0.5) <= 1e-5
    assert np.abs(y.sum(0) - gold["col_sums"]).max() / (amax * 100.0) <= 1e-5


@pytest.mark.parametrize("B,dim,out_dim", [(128, 784, 784), (1000, 64, 64), (4097, 128, 200), (300, 256, 16)])
def test_mlp_fused_kernel_shapes_vs_float64_oracle(B, dim, out_dim):
    """Fused kernel on ragged slabs, several slabs per CTA (B > 148 * 128 is covered by the 10k x 2 case below),
    narrow / wide outputs and a ragged last output tile."""
    torch.manual_seed(B + dim)
    m = cfm_b200.MLP(dim=dim, out_dim=out_dim, w=256, time_varying=True)
    state = {k: v.clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    x = torch.randn(B, dim)
    with torch.no_grad():
        y = m.vector_field(0.21, x.to(DEV)).cpu().numpy()
    ref = vf.mlp_forward_from_state(state, torch.cat([x, torch.full((B, 1), 0.21)], 1)).numpy()
    assert y.shape == (B, out_dim)
    assert np.abs(y - ref).max() / np.abs(ref).max() <= 1e-5


def test_mlp_fused_kernel_many_slabs_and_silu():
    torch.manual_seed(3)
    m = cfm_b200.MLP(dim=64, w=256, time_varying=True)
    m.act = _ffi.ACT_SILU
    state = {k: v.clone() for k, v in m.state_dict().items()}
    m = m.to(DEV)
    B = 148 * 128 * 2 + 77  # three slabs on some CTAs: exercises the slab loop and its barrier phases
    x = torch.randn(B, 64)
    with torch.no_grad():
        y = m.vector_field(0.5, x.to(DEV)).cpu()
    h = torch.cat([x, torch.full((B, 1), 0.5)], 1).double()
    for li, key in enumerate(("net.0", "net.2", "net.4", "net.6")):
        h = h @ state[key + ".weight"].double().T + state[key + ".bias"].double()
        if li < 3:
            h = torch.nn.functional.silu(h)
    assert (y.double() - h).abs().max() / h.abs().max() <= 1e-5


def test_dopri5_config3_full_batch_one_launch_per_nfe():
    """C3 through the device-resident controller with the fused forward: same step sequence as the oracle driver,
    one MLP launch per function evaluation."""
    m = _mlp784()
    mc = vf.make_mlp(784, w=256, time_varying=True)
    mc.load_state_dict(m.state_dict())
    m = m.to(DEV)
    x = _x10k()[:4096]
    node = cfm_b200.NeuralODE(cfm_b200.torch_wrapper(m), solver="dopri5", atol=1e-4, rtol=1e-4)
    node.use_cuda_graph = False
    L = _ffi.lib()
    node.trajectory(x.to(DEV), torch.linspace(0, 1, 2))  # warm-up (prepare, first-touch)
    n0 = L.cfm_launch_count()
    traj = node.trajectory(x.to(DEV), torch.linspace(0, 1, 2))
    launches = L.cfm_launch_count() - n0
    ref, st = vf.dopri5_trajectory(lambda t, z: vf.wrapped_forward(mc, t, z), x, torch.linspace(0, 1, 2))
    assert node.stats["nfe"] == st["nfe"] == 20 and node.stats["accepted"] == st["accepted"]
    assert (traj[-1].cpu() - ref[-1]).abs().max() <= 1e-4 * ref.abs().max()
    # initial step: 2 x (fp32 -> fp16x3 split + fused MLP) + 2 reductions + probe + finish = 8 launches;
    # per step: stage-1 input + 5 x (partial on the side stream + finish) + 6 x ONE fused MLP launch + error norm +
    # control + commit = 20 (15 with the one-piece stage inputs).  Four launches per forward would need 38.
    steps = node.stats["accepted"] + node.stats["rejected"]
    assert launches <= 8 + (steps + 1) * 20, (launches, steps)


# ------------------------------------------------------------------------- dopri5 driver, split stage inputs
def _rk_state(dt=0.0625, t=0.25):
    st = _ffi.RkState()
    st.t, st.dt, st.t_end, st.atol, st.rtol = t, dt, 1.0, 1e-4, 1e-4
    st.n_span, st.ckpt, st.save_slot = 2, 1, -1
    return torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(DEV)


@pytest.mark.parametrize("stage", [2, 3, 4, 5, 6])
def test_rk_stage_partial_plus_finish_is_bit_identical_to_the_one_piece_kernel(stage):
    """cfm_rk_stage_partial (everything but the newest derivative; runs on a side stream during the MLP) followed by
    cfm_rk_stage_finish performs the same fp32 operations in the same order as cfm_rk_stage_input."""
    L = _ffi.lib()
    B, D = 513, 64
    numel = B * D
    g = torch.Generator().manual_seed(stage)
    x = torch.randn(B, D, generator=g).to(DEV)
    k = torch.randn(7, B, D, generator=g).to(DEV)
    st = _rk_state()
    sp = _ffi.stream_ptr(torch.device(DEV))
    f32 = lambda: torch.zeros(B, D, dtype=torch.float32, device=DEV)  # noqa: E731
    f16 = lambda: torch.zeros(B, D, dtype=torch.float16, device=DEV)  # noqa: E731
    out_a, hi_a, lo_a, e_a, t_a = f32(), f16(), f16(), f32(), torch.zeros(1, device=DEV)
    _ffi.check(L.cfm_rk_stage_input(_ffi.ptr(st), _ffi.ptr(x), _ffi.ptr(k), _ffi.ptr(out_a), _ffi.ptr(hi_a), _ffi.ptr(lo_a),
                                    _ffi.ptr(t_a), _ffi.ptr(e_a) if stage == 6 else None, numel, stage, sp), "stage_input")
    part, out_b, hi_b, lo_b, e_b, t_b = f32(), f32(), f16(), f16(), f32(), torch.zeros(1, device=DEV)
    _ffi.check(L.cfm_rk_stage_partial(_ffi.ptr(st), _ffi.ptr(x), _ffi.ptr(k), _ffi.ptr(part),
                                      _ffi.ptr(e_b) if stage == 6 else None, _ffi.ptr(t_b), numel, stage, sp), "partial")
    _ffi.check(L.cfm_rk_stage_finish(_ffi.ptr(st), _ffi.ptr(part), _ffi.ptr(k), _ffi.ptr(out_b), _ffi.ptr(hi_b), _ffi.ptr(lo_b),
                                     _ffi.ptr(e_b) if stage == 6 else None, numel, stage, sp), "finish")
    assert torch.equal(out_a, out_b) and torch.equal(t_a, t_b)
    assert torch.equal(hi_a.view(torch.int16), hi_b.view(torch.int16)) and torch.equal(lo_a.view(torch.int16), lo_b.view(torch.int16))
    if stage == 6:
        assert torch.equal(e_a, e_b)
    # and the operand pair is the fp16x3 split of the fp32 stage input
    rec = hi_b.float() + lo_b.float() / 2048.0
    assert (rec - out_b).abs().max().item() <= 2.0 ** -21 * out_b.abs().max().item()


def test_dopri5_overlapped_stage_inputs_equal_the_serial_driver():
    """Trajectories with the stage inputs split across two streams (graph and eager) are bit-identical to the serial
    one-stream driver: same kernels' arithmetic, only the schedule differs."""
    torch.manual_seed(0)
    m = cfm_b200.MLP(dim=64, w=256, time_varying=True).to(DEV)
    x = torch.randn(1500, 64, generator=torch.Generator().manual_seed(1)).to(DEV)
    span = torch.linspace(0, 1, 4)
    outs = []
    for overlap, graph in ((False, True), (True, True), (True, False)):
        node = cfm_b200.NeuralODE(cfm_b200.torch_wrapper(m), solver="dopri5", atol=1e-5, rtol=1e-5)
        node.overlap_stages, node.use_cuda_graph = overlap, graph
        node.trajectory(x, span)
        outs.append((node.trajectory(x, span).clone(), dict(node.stats)))
    for o, s in outs[1:]:
        assert torch.equal(o, outs[0][0])
        assert (s["nfe"], s["accepted"], s["rejected"]) == (outs[0][1]["nfe"], outs[0][1]["accepted"], outs[0][1]["rejected"])


@pytest.mark.parametrize("B,dim,act", [(1500, 64, "selu"), (1000, 784, "selu"), (300, 200, "silu")])
def test_dopri5_stage_input_formed_inside_the_fused_mlp_equals_the_separate_kernel(B, dim, act):
    """cfm_mlp_forward_rkstage_f32 (stage input formed by the fused MLP kernel's layer-1 operand producer, one launch per
    NFE) against the two-launch form (cfm_rk_stage_input + cfm_mlp_forward_split_gated_f32): the same fp32 operations
    in the same order, so trajectories, step counts and the controller's error ratios are bit-identical -- on ragged
    slabs (B % 128 != 0), a ragged last K chunk (784 = 12 x 64 + 16; 200 = 3 x 64 + 8) and both activations."""
    torch.manual_seed(3)
    m = cfm_b200.MLP(dim=dim, w=256, time_varying=True).to(DEV)
    if act == "silu":
        m.act = _ffi.ACT_SILU
    x = torch.randn(B, dim, generator=torch.Generator().manual_seed(4)).to(DEV)
    span = torch.linspace(0, 1, 3)
    outs = []
    for fuse, graph in ((False, True), (True, True), (True, False)):
        node = cfm_b200.NeuralODE(cfm_b200.torch_wrapper(m), solver="dopri5", atol=1e-5, rtol=1e-5)
        node.fuse_stage_input, node.use_cuda_graph = fuse, graph
        node.trajectory(x, span)
        outs.append((node.trajectory(x, span).clone(), dict(node.stats)))
        P = next(iter(node._plans.values()))
        assert P["rkfused"] == fuse
    for o, s in outs[1:]:
        assert torch.equal(o, outs[0][0])
        assert (s["nfe"], s["accepted"], s["rejected"], s["last_ratio"]) == \
            (outs[0][1]["nfe"], outs[0][1]["accepted"], outs[0][1]["rejected"], outs[0][1]["last_ratio"])


def test_rkstage_single_evaluation_against_the_float64_oracle():
    """One stage evaluation through the one-launch form, checked directly: k_{s+1}, xnew and the error partial against
    float64 arithmetic on the same inputs (1e-5 of max|y| for the field, fp32 rounding for the combinations)."""
    from oracle import vector_field as vf
    torch.manual_seed(5)
    B, D = 777, 784
    m = cfm_b200.MLP(dim=D, w=256, time_varying=True)
    sd = {k_: v_.clone() for k_, v_ in m.state_dict().items()}

    def f64(t, z):  # utils.py:51-52 + models.py:20-21 in float64
        return vf.mlp_forward_from_state(sd, torch.cat([z.double(), torch.full((z.shape[0], 1), t, dtype=torch.float64)], 1))
    m = m.to(DEV)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(B, D, generator=g)
    k = torch.randn(7, B, D, generator=g)
    st = _ffi.RkState()
    st.t, st.dt, st.t_end, st.atol, st.rtol = 0.25, 0.125, 1.0, 1e-4, 1e-4
    std = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(DEV)
    A6 = [35 / 384, 0.0, 500 / 1113, 125 / 192, -2187 / 6784, 11 / 84]
    E = [35 / 384 - 1951 / 21600, 0.0, 500 / 1113 - 22642 / 50085, 125 / 192 - 451 / 720,
         -2187 / 6784 + 12231 / 42400, 11 / 84 - 649 / 6300]
    xd, kd = x.to(DEV), k.to(DEV).contiguous()
    xnew, errp = torch.zeros(B, D, device=DEV), torch.zeros(B, D, device=DEV)
    m.vector_field_rkstage(std, xd, kd, 6, xnew, errp)
    xs = x.double() + 0.125 * sum(a * k[j].double() for j, a in enumerate(A6))
    ep = sum(e * k[j].double() for j, e in enumerate(E))
    assert (xnew.cpu().double() - xs).abs().max() <= 4e-6 * xs.abs().max()
    assert (errp.cpu().double() - ep).abs().max() <= 4e-6 * max(1.0, ep.abs().max().item())
    ref = f64(0.25 + 1.0 * 0.125, xnew.cpu())
    got = kd[6].cpu().double()
    assert (got - ref).abs().max() <= 1e-5 * ref.abs().max()
    # stage 2 (two derivative arrays, c = 3/10), no side outputs
    m.vector_field_rkstage(std, xd, kd, 2)
    xs2 = (x.double() + 0.125 * (3 / 40 * k[0].double() + 9 / 40 * k[1].double())).float()
    ref2 = f64(float(np.float32(0.25) + np.float32(0.3) * np.float32(0.125)), xs2)
    assert (kd[2].cpu().double() - ref2).abs().max() <= 1e-5 * ref2.abs().max()


# ------------------------------------------------- float64-potential Sinkhorn with fp32 screening (BASELINE config 4)
def _sk(M, reg, precision, iters, normalize=False):
    """Solve on a given cost matrix (the oracle's own M) through OTPlanSampler's solver stage."""
    s = OTPlanSampler("sinkhorn", reg=reg, precision=precision, stall_tol=0.0, num_iter_max=iters, stop_thr=0.0, warn=False)
    n0, n1 = M.shape
    ld = (n1 + 3) // 4 * 4
    buf = torch.zeros((n0, ld), dtype=torch.float32, device=DEV)
    buf[:, :n1] = M.to(DEV)
    cmax = M.max().reshape(1).float().to(DEV)
    cp = s._solve_sinkhorn(buf, cmax, n0, n1, reg, normalize)
    st = cp.status.cpu().tolist()
    return cp, cp.log_u.cpu().numpy(), cp.log_v.cpu().numpy(), st, float(cp.err.item())


@pytest.mark.parametrize("n0,n1,d,reg,normalize", [(2048, 2048, 512, 0.1, False), (1000, 1500, 64, 0.01, False),
                                                   (777, 515, 32, 0.002, True), (4096, 4096, 512, 0.1, False)])
def test_screened_mixed_sinkhorn_equals_the_unscreened_and_float64_solvers(n0, n1, d, reg, normalize):
    """The fp32 screening of negligible log-sum-exp terms (mode 3 / auto in the |M/reg| >> 64 regime) changes which
    terms take the float64 path, not the result: potentials within 1e-6 of the unscreened mixed solver (4e-6 of the
    all-float64 solver) after 1, 7 and 60 iterations -- aligned and ragged shapes, rectangular, normalised cost."""
    g = torch.Generator().manual_seed(n0 + n1)
    x0, x1 = torch.randn(n0, d, generator=g), torch.randn(n1, d, generator=g) + 0.1
    M = oc.cost_matrix(x0, x1)
    scale = float(M.max()) if normalize else 1.0
    assert float(M.max()) / scale / reg > 200
    for iters in (1, 7, 60):
        _, lu, lv, st, _ = _sk(M, reg, "fp64-mixed", iters, normalize)
        _, lu0, lv0, st0, _ = _sk(M, reg, "fp64-mixed-unscreened", iters, normalize)
        _, lu1, lv1, st1, _ = _sk(M, reg, "fp64", iters, normalize)
        assert st[2] == 2 and st0[2] == 2 and st1[2] == 1
        assert np.abs(lu - lu0).max() < 1e-6 and np.abs(lv - lv0).max() < 1e-6, iters
        # against all-float64 arithmetic: the fp32 exponentials of mixed mode (1e-7 per term) accumulate over iterations
        assert np.abs(lu - lu1).max() < 4e-6 and np.abs(lv - lv1).max() < 4e-6, iters
    _, lua, lva, sta, _ = _sk(M, reg, "auto", 60, normalize)
    assert sta[2] == 2 and np.array_equal(lua, lu) and np.array_equal(lva, lv)  # auto resolves to the screened path


def test_screened_mixed_sinkhorn_wide_row_offsets_and_nan():
    """Row norms spread over three decades put large offsets into u as well as v (both potentials ~1e4, their
    cancellation with -M/reg is what the float64 path is for): the screening margin must still hold.  A NaN cost is
    never screened out: it reaches the potentials as in the unscreened solver."""
    g = torch.Generator().manual_seed(5)
    n, d = 512, 16
    x0 = torch.randn(n, d, generator=g) * torch.logspace(-1, 1.3, n)[:, None]
    x1 = torch.randn(n, d, generator=g) * torch.logspace(1.3, -1, n)[:, None]
    M = oc.cost_matrix(x0, x1)
    assert float(M.max()) / 0.5 > 5e3
    for iters in (1, 25):
        _, lu, lv, st, _ = _sk(M, 0.5, "fp64-mixed", iters)
        _, lu1, lv1, _, _ = _sk(M, 0.5, "fp64", iters)
        assert st[2] == 2
        tol = 1e-9 * float(M.max()) / 0.5 + 1e-6  # float64 cancellation floor of potentials this large
        assert np.abs(lu - lu1).max() < tol and np.abs(lv - lv1).max() < tol, iters
    Mn = M.clone()
    Mn[3, 7] = float("nan")
    _, lu, lv, st, err = _sk(Mn, 0.5, "fp64-mixed", 5)
    assert np.isnan(lu[3]) and np.isnan(lv[7])


@pytest.mark.parametrize("n0,n1", [(64, 9000), (40, 12288)])
def test_screened_mixed_sinkhorn_wide_matrices(n0, n1):
    """n1 > 8192 leaves the seeded solver (one column panel) for the generic sweep, whose mixed mode screens with
    thresholds from row / block maxima: same potentials as the unscreened and the all-float64 solvers."""
    g = torch.Generator().manual_seed(n1)
    M = torch.rand(n0, n1, generator=g) * 40.0 + 5.0
    for iters in (1, 12):
        _, lu, lv, st, _ = _sk(M, 0.05, "fp64-mixed", iters)
        _, lu0, lv0, st0, _ = _sk(M, 0.05, "fp64-mixed-unscreened", iters)
        _, lu1, lv1, st1, _ = _sk(M, 0.05, "fp64", iters)
        assert st[2] == 2 and st[3] == 0 and st0[2] == 2 and st1[2] == 1
        assert np.abs(lu - lu0).max() < 1e-6 and np.abs(lv - lv0).max() < 1e-6, iters
        assert np.abs(lu - lu1).max() < 2e-6 and np.abs(lv - lv1).max() < 2e-6, iters
