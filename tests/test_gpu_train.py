"""Training step (SURVEY 8a a19-a23) on the GPU against the fixtures generated from the LIVE reference
(tests/golden/train_c5small.npz: DiffusionLoss.__call__ + loss.backward() of the unmodified reference, fp64) and
against the oracle (oracle/training.py) on seeded inputs.  Everything goes through the C ABI.

Tolerances: noising / targets are fp64 kernels -> 1e-12 (types bit exact); the network runs in fp32 -> loss and
outputs 1e-4 of max|ref| (north_star), parameter gradients 2e-3 of max|ref| per tensor (fp32 accumulation over up to
E*O rows against an fp64 reference; measured ~1e-5)."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import f64_default, rel_err

pytestmark = pytest.mark.gpu
T, Z = 1000, 90


def _case(z, case):
    p = f"{case}/"
    return {k[len(p):]: z[k] for k in z.files if k.startswith(p)}


def _engine(device, weights_npz, num_atoms, sd=None, backward_precision="fp32"):
    from arreau_b200.tables import build_tables
    from arreau_b200.training import FlatParams, TrainEngine
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")} if sd is None else sd
    p = FlatParams(164, 4, Z, device)
    p.load_state_dict(sd)
    return TrainEngine(p, build_tables(T, Z), weights_npz["fourier_w"], weights_npz["ori_grid"], num_atoms, 5.0, 8,
                       device=device, backward_precision=backward_precision)


@pytest.mark.parametrize("tf32", [0, 1])
@pytest.mark.parametrize("M,N,K,ak,bk,acc", [(300, 128, 96, 1, 1, 0), (128, 256, 20000, 0, 0, 0), (1000, 512, 128, 1, 0, 1),
                                             (128, 16, 256, 0, 0, 0), (77, 128, 94, 1, 0, 1), (512, 128, 5000, 0, 0, 1),
                                             (640, 256, 50000, 0, 0, 0), (4000, 640, 256, 1, 1, 0), (2100, 256, 640, 1, 0, 0),
                                             (96, 64, 1000, 0, 1, 0)])
def test_sgemm_against_torch(device, M, N, K, ak, bk, acc, tf32):
    """The generic GEMM of the backward pass (fp32 FFMA, and its TF32 tensor-core variant: operands rounded to 10
    mantissa bits -> 2e-3 of max|ref|) against a torch fp64 matmul of the same operands."""
    from arreau_b200 import _lib
    g = torch.Generator(device="cpu").manual_seed(M + N + K)
    Kp = (K + 3) // 4 * 4
    A = torch.randn((M, Kp) if ak else (K, M), generator=g).to(device)
    B = torch.randn((N, Kp) if bk else (K, N), generator=g).to(device)
    if ak:
        A[:, K:] = 0
    if bk:
        B[:, K:] = 0
    Cm = torch.randn(M, N, generator=g).to(device)
    bias = torch.randn(N, generator=g).to(device)
    ref = (A.double()[:, :K] if ak else A.double().T) @ (B.double()[:, :K].T if bk else B.double())
    ref = 0.5 * ref + (Cm.double() if acc else 0)
    use_bias = K <= 4096
    if use_bias:
        ref = ref + bias.double()
    partial = torch.empty(4 << 20, device=device)
    _lib.call("arreau_sgemm", ak | (2 * tf32), bk, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(), N, M,
              N, K, C.c_float(0.5), bias.data_ptr() if use_bias else None, acc, partial.data_ptr(), partial.numel(),
              torch.cuda.current_stream().cuda_stream)
    tol = 2e-3 if tf32 else 2e-6 * max(1.0, np.sqrt(K) / 16)
    assert rel_err(Cm.cpu().numpy(), ref.cpu().numpy()) < tol


def test_sgemm_tma_operands_round_to_nearest(device):
    """The TMA-fed TF32 GEMM reads its operands through TFLOAT32 tensor maps: the TMA engine must ROUND fp32 to TF32
    (1 + 0.75 * 2^-10 -> 1 + 2^-10), not truncate (-> 1), in all four operand orders -- truncation would bias every
    product of the chain by ~1e-3 in the same direction."""
    from arreau_b200 import _lib
    M, N, K = 128, 128, 64
    partial = torch.empty(1 << 20, device=device)
    for ak in (1, 0):
        for bk in (1, 0):
            A = torch.full((M, K) if ak else (K, M), 1.0 + 0.75 * 2.0 ** -10, device=device)
            B = torch.ones((N, K) if bk else (K, N), device=device)
            Cm = torch.zeros(M, N, device=device)
            _lib.call("arreau_sgemm", ak | 2, bk, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(), N, M, N, K,
                      C.c_float(1.0), None, 0, partial.data_ptr(), partial.numel(), torch.cuda.current_stream().cuda_stream)
            assert torch.all(Cm == K * (1.0 + 2.0 ** -10)), (ak, bk, float(Cm[0, 0]) / K)


@pytest.mark.parametrize("M,N,K,ak,bk", [(77, 132, 96, 1, 0), (300, 128, 200, 1, 1), (640, 256, 9000, 0, 0), (132, 96, 5000, 0, 1)])
def test_sgemm_tf32_stays_in_bounds_and_is_deterministic(device, M, N, K, ak, bk):
    """Ragged tiles of the TF32 GEMM (TMA zero fill of the operands, predicated epilogue, split second stage): nothing is
    written outside C[M, N] inside a larger allocation (compute-sanitizer is closed on this pool), and two runs agree bit
    for bit."""
    from arreau_b200 import _lib
    g = torch.Generator(device="cpu").manual_seed(7 * M + N + K)
    A = torch.randn((M, K) if ak else (K, M), generator=g).to(device)
    B = torch.randn((N, K) if bk else (K, N), generator=g).to(device)
    ldc, pad = N + 4, 5
    partial = torch.empty(4 << 20, device=device)
    outs = []
    for _ in range(2):
        Cm = torch.full((M + pad, ldc), -7.25, device=device)
        _lib.call("arreau_sgemm", ak | 2, bk, A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), Cm.data_ptr(), ldc, M, N, K,
                  C.c_float(1.0), None, 0, partial.data_ptr(), partial.numel(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert torch.all(Cm[M:] == -7.25) and torch.all(Cm[:, N:] == -7.25)
        outs.append(Cm[:M, :N].clone())
    assert torch.equal(outs[0], outs[1])
    ref = (A.double() if ak else A.double().T) @ (B.double().T if bk else B.double())
    assert rel_err(outs[0].cpu().numpy(), ref.cpu().numpy()) < 2e-3


def test_flat_weight_layouts_match_state_dict_layouts(device, weights_npz):
    """The training engine's kernel layouts (PonitaWeights.from_flat) against the sampling engine's (PonitaWeights of the
    state_dict) for the same weights: bit-identical, except the folded first basis layer w1m_t, which the host folds in
    fp64 and from_flat in fp32 on the device.  A monomial gathers at most 6 columns of basis_fn.1.weight, so the fp32
    sum is within 5 * 2^-24 of the sum of the folded terms' magnitudes."""
    from arreau_b200.training import FlatParams
    from arreau_b200.weights import HIDDEN, MONO_PAD, NUM_MONO, PonitaWeights, monomial_fold_table
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    p = FlatParams(164, 4, Z, device)
    p.load_state_dict(sd)
    host = PonitaWeights(sd, weights_npz["ori_grid"], device=device)
    flat = PonitaWeights.from_flat(p, torch.as_tensor(weights_npz["ori_grid"]).to(device))
    assert set(flat.t) <= set(host.t) and len(flat.t) == 17
    assert (flat.num_scalar, flat.num_vec, flat.num_states) == (host.num_scalar, host.num_vec, host.num_states)
    for k in flat.t:
        if k != "w1m_t":
            assert flat.t[k].dtype == host.t[k].dtype and torch.equal(flat.t[k], host.t[k]), k
    mag = np.zeros((HIDDEN, NUM_MONO))
    np.add.at(mag, (slice(None), monomial_fold_table()), np.abs(sd["basis_fn.1.weight"].astype(np.float64)))
    bound = np.zeros((MONO_PAD, HIDDEN))
    bound[:NUM_MONO] = 5 * 2.0 ** -24 * mag.T           # the bias row and the padding must be equal
    err = np.abs(flat.t["w1m_t"].double().cpu().numpy() - host.t["w1m_t"].double().cpu().numpy())
    assert np.all(err <= bound), float((err - bound).max())


@pytest.mark.parametrize("case", [0, 1])
def test_noising_matches_reference(device, gold, weights_npz, case):
    c = _case(gold("train_c5small.npz"), case)
    te = _engine(device, weights_npz, c["num_atoms"])
    te.set_batch(c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    te.noise_batch()
    e = te.eng
    assert np.array_equal(e.types.cpu().numpy(), c["noisy_types"])
    d = np.abs(e.frac.cpu().numpy() - c["noisy_frac"])
    assert np.minimum(d, 1 - d).max() < 1e-12
    d = np.abs(te.target_eps.cpu().numpy() - c["target_eps"])
    assert np.minimum(d, 1 - d).max() < 1e-10
    assert rel_err(te.lengths0.cpu().numpy(), c["lengths"]) < 1e-14
    assert rel_err(te.angles0.cpu().numpy(), c["angles"]) < 1e-13
    assert rel_err(e.lengths.cpu().numpy(), c["noisy_lengths"]) < 1e-14


@pytest.mark.parametrize("case", [0, 1])
def test_loss_and_gradients_match_reference(device, gold, weights_npz, case):
    c = _case(gold("train_c5small.npz"), case)
    te = _engine(device, weights_npz, c["num_atoms"])
    loss, _ = te.loss_and_grads(c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    torch.cuda.synchronize()
    e = te.eng
    assert rel_err(e.score.cpu().numpy(), c["pred_eps"]) < 1e-4
    assert rel_err(e.logits.cpu().numpy(), c["pred_logits"]) < 1e-4
    assert rel_err(e.len0.cpu().numpy(), c["pred_len"]) < 1e-4
    got = loss.cpu().numpy()
    assert abs(got[0] - float(c["loss"])) <= 1e-4 * abs(float(c["loss"]))
    for i, k in enumerate(("e_frac", "vb", "ce", "e_lat"), start=1):
        assert abs(got[i] - float(c[k])) <= 1e-4 * max(abs(float(c[k])), 1e-3), (k, got[i], float(c[k]))
    gv = te.p.grad_views()
    worst = {}
    for k, g in gv.items():
        g = g.cpu().numpy()
        if case == 0:
            err = rel_err(g, c["grad/" + k])
        else:
            ref_norm = float(c["gradnorm/" + k])
            err = max(abs(float(np.linalg.norm(g.astype(np.float64))) - ref_norm) / max(ref_norm, 1e-30),
                      rel_err(g.reshape(-1)[:64], c["gradhead/" + k]) if np.abs(c["gradhead/" + k]).max() > 1e-3 * ref_norm else 0.0)
        worst[k] = err
    bad = {k: v for k, v in worst.items() if not v < 2e-3}
    assert not bad, bad


def test_loss_gradients_wrt_outputs_against_oracle(device, gold, weights_npz):
    """dloss/d(score, logits, len0) of arreau_training_loss against autograd on the oracle's loss (fp64)."""
    from oracle import restatement as R, training as TR
    c = _case(gold("train_c5small.npz"), 0)
    te = _engine(device, weights_npz, c["num_atoms"])
    te.set_batch(c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    te.noise_batch()
    e = te.eng
    N, G = e.N, e.G
    g = torch.Generator().manual_seed(3)
    score = torch.randn(N, 3, generator=g, dtype=torch.float64) * 0.7
    logits = torch.randn(N, Z, generator=g, dtype=torch.float64) * 2.0
    len0 = torch.randn(G, 3, generator=g, dtype=torch.float64) + 2.0
    e.score.copy_(score)
    e.logits.copy_(logits)
    e.len0.copy_(len0)
    te.compute_loss()
    with f64_default():
        tabs = R.DiffusionTables.build(T, Z)
        s, l, n = [x.float().double().requires_grad_(True) for x in (score, logits, len0)]
        t_atom = torch.as_tensor(c["timestep"]).reshape(-1).repeat_interleave(torch.as_tensor(c["num_atoms"]))
        ef = TR.frac_x_error(s, torch.as_tensor(c["target_eps"]))
        et, vb, ce = TR.d3pm_calculate_loss(tabs, torch.as_tensor(c["types0"]), l, torch.as_tensor(c["noisy_types"]), t_atom)
        el = torch.nn.functional.mse_loss(n, torch.as_tensor(c["lengths"]) / torch.as_tensor(c["num_atoms"]).unsqueeze(-1))
        total = ef + et + el
        gs, gl, gn = torch.autograd.grad(total, [s, l, n])
    got = te.loss.cpu().numpy()
    for a, b in zip(got, (total, ef, vb, ce, el)):
        assert abs(a - b.item()) <= 1e-10 * max(1.0, abs(b.item()))
    assert rel_err(te.dscore.cpu().numpy(), gs.numpy()) < 1e-6
    assert rel_err(te.dlogits.cpu().numpy(), gl.numpy()) < 1e-6
    assert rel_err(te.dlen0.cpu().numpy(), gn.numpy()) < 1e-6


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_backward_is_deterministic(device, gold, weights_npz, precision):
    """Two runs of the whole step give bit-identical losses and gradients on both precision paths: fixed-order split
    reductions, per-CTA column sums in a static item order, no atomics."""
    c = _case(gold("train_c5small.npz"), 1)
    te = _engine(device, weights_npz, c["num_atoms"], backward_precision=precision)
    args = (c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    te.loss_and_grads(*args)
    g0, l0 = te.p.grad.clone(), te.loss.clone()
    te.loss_and_grads(*args)
    assert torch.equal(g0, te.p.grad) and torch.equal(l0, te.loss)


def test_calibrate_matches_reference(device, gold, weights_npz):
    """FiberBundleConv.callibrate (conv.py:122-123,140-146): the rescaled kernel / fiber_kernel weights."""
    c = _case(gold("train_c5small.npz"), "cal")
    te = _engine(device, weights_npz, c["num_atoms"])
    te.calibrate(c["frac"], c["types"], c["lengths"], c["angles"], int(c["timestep"]))
    v = te.p.views()
    for k in c:
        if k.startswith("after/"):
            assert rel_err(v[k[6:]].cpu().numpy(), c[k]) < 1e-4, k


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_larger_batch_against_oracle(device, weights_npz, precision):
    """A C5-shaped batch (48 crystals, 1..40 atoms): loss and gradients against the oracle's autograd -- the fp32 parity
    path (loss 1e-4, gradients 2e-3 of max|ref| per tensor) and the TF32 path of `train.fit` / `bench.py --workload train`
    (TMA-fed tcgen05 GEMMs in forward and backward; stated tolerance: loss 1e-3, gradients 4e-3; measured 1.4e-4 / 8.8e-4)."""
    from arreau_b200.synthetic import make_crystals
    from oracle import restatement as R, training as TR
    cr = make_crystals(48, 1, 40, seed=77)
    G, N = cr.num_crystals, cr.total_atoms
    with f64_default():
        torch.manual_seed(9)
        timestep, eps_x, u, eps_l = TR.draw_training_noise(G, N, Z, T)
        sd = {k: torch.as_tensor(weights_npz[k], dtype=torch.float64) for k in weights_npz.files
              if k not in ("ori_grid", "fourier_w")}
        W = R.PonitaWeights(sd, torch.as_tensor(weights_npz["ori_grid"], dtype=torch.float64), 5.0)
        tabs = R.DiffusionTables.build(T, Z)
        L0 = R.lattice_from_params(torch.as_tensor(cr.lengths), torch.as_tensor(cr.angles))
        loss, grads, parts = TR.training_grads(W, tabs, torch.as_tensor(weights_npz["fourier_w"], dtype=torch.float64),
                                               torch.as_tensor(cr.frac), torch.as_tensor(cr.types), L0,
                                               torch.as_tensor(cr.num_atoms), timestep, eps_x, u, eps_l, 5.0, 8)
    te = _engine(device, weights_npz, cr.num_atoms, backward_precision=precision)
    got, _ = te.loss_and_grads(cr.frac, cr.types, L0.numpy(), timestep.numpy(), eps_x.numpy(), u.numpy(), eps_l.numpy())
    loss_tol, grad_tol = (1e-4, 2e-3) if precision == "fp32" else (1e-3, 4e-3)
    assert abs(got[0].item() - loss.item()) <= loss_tol * abs(loss.item())
    gv = te.p.grad_views()
    errs = {k: rel_err(gv[k].cpu().numpy(), grads[k].numpy()) for k in grads}
    print(f"{precision}: loss rel err {abs(got[0].item() - loss.item()) / abs(loss.item()):.2e}, worst gradient error "
          f"{max(errs.values()):.2e} ({max(errs, key=errs.get)})")
    bad = {k: v for k, v in errs.items() if not v < grad_tol}
    assert not bad, bad


def _mirror_model(device, weights_npz):
    import argparse
    from arreau_b200.diffusion.diffusion_helpers import GaussianFourierProjection
    from arreau_b200.diffusion.diffusion_loss import DiffusionLoss
    from arreau_b200.ponita.models.ponita import PonitaFiberBundle
    net = PonitaFiberBundle(164 + 4, 128, Z, 3, 0, 0, 5, output_dim_vec=1, radius=5.0, num_ori=16, basis_dim=256,
                            degree=3, widening_factor=4, layer_scale=1e-6, multiple_readouts=True,
                            ori_grid=weights_npz["ori_grid"])
    net.load_state_dict({k: torch.as_tensor(weights_npz[k]) for k in weights_npz.files if k not in ("ori_grid", "fourier_w")})
    temb = GaussianFourierProjection(32, 16)
    with torch.no_grad():
        temb.gaussian_fourier_proj_w.copy_(torch.as_tensor(weights_npz["fourier_w"]))
    dl = DiffusionLoss(argparse.Namespace(radius=5.0, max_neighbors=8, num_timesteps=T), Z)
    return net.to(device), temb, dl


def _batch(c, device):
    import argparse
    return argparse.Namespace(X0=torch.as_tensor(c["frac0"]).to(device), A0=torch.as_tensor(c["types0"]).to(device),
                              L0=torch.as_tensor(c["lattice0"]).reshape(-1, 3).to(device),
                              num_atoms=torch.as_tensor(c["num_atoms"]).to(device))


def test_python_face_loss_backward(device, gold, weights_npz):
    """DiffusionLoss.__call__ of the mirror (reference signature) + loss.backward(): the parameters' .grad are the
    reference's gradients; the draws are injected (the mirror draws on the GPU stream otherwise)."""
    c = _case(gold("train_c5small.npz"), 0)
    net, temb, dl = _mirror_model(device, weights_npz)
    noise = tuple(torch.as_tensor(c[k]).to(device) for k in ("eps_x", "u", "eps_l"))
    t = torch.as_tensor(c["timestep"]).to(device)
    # per-crystal timesteps: drive the engine directly with the golden's timestep vector through `noise` + monkeypatch
    orig = torch.randint
    torch.randint = lambda *a, **k: t
    try:
        loss = dl(net, _batch(c, device), temb, noise=noise)
    finally:
        torch.randint = orig
    assert abs(loss.item() - float(c["loss"])) <= 1e-4 * abs(float(c["loss"]))
    loss.backward()
    for name, p in net.named_parameters():
        if p.numel():
            assert p.grad is not None and rel_err(p.grad.cpu().numpy(), c["grad/" + name]) < 2e-3, name
    # a second call without injected noise runs on the GPU generator and accumulates into .grad like autograd
    g0 = net.x_embedder.weight.grad.clone()
    dl(net, _batch(c, device), temb).backward()
    assert not torch.equal(g0, net.x_embedder.weight.grad)


def test_fused_adam_matches_torch(device, weights_npz):
    from arreau_b200.training import FlatParams, FusedAdam
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    p = FlatParams(164, 4, Z, device)
    p.load_state_dict(sd)
    ref = {k: v.clone().requires_grad_(True) for k, v in p.views().items()}
    decay = [v for k, v in ref.items() if k.endswith(".weight") and ".norm." not in k]
    no_decay = [v for k, v in ref.items() if not (k.endswith(".weight") and ".norm." not in k)]
    topt = torch.optim.Adam([{"params": decay, "weight_decay": 0.01}, {"params": no_decay, "weight_decay": 0.0}], lr=3e-4)
    opt = FusedAdam(p, lr=3e-4, weight_decay=0.01, max_grad_norm=0.5)
    g = torch.Generator(device="cpu").manual_seed(1)
    for step in range(3):
        grad = (torch.randn(p.total, generator=g) * (10.0 if step == 0 else 1e-4)).to(device)   # clipped, then not
        p.grad.copy_(grad)
        for k, v in p._views(grad).items():
            ref[k].grad = v.clone()
        torch.nn.utils.clip_grad_norm_(list(ref.values()), 0.5)
        topt.step()
        opt.step()
        assert abs(opt.grad_norm() - float(grad.double().norm())) < 1e-6 * float(grad.double().norm())
    for k, v in p.views().items():
        assert rel_err(v.cpu().numpy(), ref[k].detach().cpu().numpy()) < 2e-6, k


def test_training_reduces_loss_on_a_fixed_batch(device, gold, weights_npz):
    """Ten Adam steps on one fixed noised batch: the loss must fall (end-to-end sanity of sign and scale)."""
    from arreau_b200.training import FusedAdam
    c = _case(gold("train_c5small.npz"), 0)
    te = _engine(device, weights_npz, c["num_atoms"])
    opt = FusedAdam(te.p, lr=1e-3, max_grad_norm=0.5)
    args = (c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    losses = []
    for _ in range(10):
        loss, _ = te.loss_and_grads(*args)
        losses.append(loss[0].item())
        opt.step()
    assert losses[-1] < losses[0] - 0.05, losses


def test_tf32_backward_against_reference(device, gold, weights_npz):
    """ARREAU_PRECISION_TF32: every dense contraction of the training forward and backward on the TMA-fed tcgen05 TF32
    GEMM (operands rounded to 10 mantissa bits by the TMA engine, fp32 accumulation).  Stated tolerance of this path
    against the live reference's fp64 loss and gradients (golden fixture): loss 1e-3 (measured 1e-4), every parameter
    gradient 4e-3 of max|ref| per tensor (measured 1.1e-3).  Each of the four loss terms is held to the same 1e-3 of its
    own size, so that the total, which e_lat dominates, cannot hide an error in e_frac, the score's term."""
    c = _case(gold("train_c5small.npz"), 0)
    te = _engine(device, weights_npz, c["num_atoms"], backward_precision="tf32")
    loss, _ = te.loss_and_grads(c["frac0"], c["types0"], c["lattice0"], c["timestep"], c["eps_x"], c["u"], c["eps_l"])
    assert abs(loss[0].item() - float(c["loss"])) <= 1e-3 * abs(float(c["loss"]))
    got = loss.cpu().numpy()
    parts = {k: abs(got[i] - float(c[k])) / max(abs(float(c[k])), 1e-3)
             for i, k in enumerate(("e_frac", "vb", "ce", "e_lat"), start=1)}
    print("tf32 loss terms rel err", parts)
    assert all(v <= 1e-3 for v in parts.values()), parts
    gv = te.p.grad_views()
    errs = {k: rel_err(g.cpu().numpy(), c["grad/" + k]) for k, g in gv.items()}
    print("tf32 loss rel err", abs(loss[0].item() - float(c["loss"])) / abs(float(c["loss"])), "worst gradient error", max(errs.values()))
    bad = {k: v for k, v in errs.items() if not v < 4e-3}
    assert not bad, bad


def test_capacity_engine_reuses_buffers_across_topologies(device, weights_npz):
    """SURVEY 8f-4 / VERDICT r1 missing #2: shuffled variable-size batches run through ONE TrainEngine whose buffers are
    re-bound in place (no reallocation), and a step on a re-bound engine is bit-identical to the same step on an
    engine built for exactly that topology."""
    from arreau_b200.diffusion.lattice_helpers import lattice_from_params
    from arreau_b200.synthetic import make_training_batch
    from arreau_b200.tables import build_tables
    from arreau_b200.training import FlatParams, TrainEngine
    sd = {k: weights_npz[k] for k in weights_npz.files if k not in ("ori_grid", "fourier_w")}
    tabs = build_tables(1000, 90)
    batches = [make_training_batch(g, seed=s) for g, s in ((14, 1), (9, 2), (16, 3), (5, 4))]
    n_cap, g_cap = max(b.total_atoms for b in batches), max(b.num_crystals for b in batches)

    def draws(cr, seed):
        g = torch.Generator(device=device).manual_seed(seed)
        G, N = cr.num_crystals, cr.total_atoms
        lat0 = lattice_from_params(torch.as_tensor(cr.lengths).to(device), torch.as_tensor(cr.angles).to(device))
        return (torch.as_tensor(cr.frac).to(device), torch.as_tensor(cr.types).to(device), lat0,
                torch.randint(1, 1001, (G,), device=device, generator=g),
                torch.randn(N, 3, device=device, dtype=torch.float64, generator=g),
                torch.rand(N, 90, device=device, dtype=torch.float64, generator=g),
                torch.randn(G, 3, device=device, dtype=torch.float64, generator=g))

    p = FlatParams(164, 4, 90, device)
    p.load_state_dict(sd)
    shared = TrainEngine(p, tabs, weights_npz["fourier_w"], weights_npz["ori_grid"], batches[0].num_atoms, 5.0, 8,
                         device=device, node_capacity=n_cap, crystal_capacity=g_cap)
    ptrs = {k: v[1].data_ptr() for k, v in shared.eng._bufs.items()}
    kernels_ptr = shared.eng.kernels.data_ptr()
    for i, cr in enumerate(batches):
        shared.set_topology(cr.num_atoms)
        loss_s, grad_s = shared.loss_and_grads(*draws(cr, 10 + i))
        loss_s, grad_s = loss_s.clone(), grad_s.clone()
        exact = TrainEngine(p, tabs, weights_npz["fourier_w"], weights_npz["ori_grid"], cr.num_atoms, 5.0, 8, device=device)
        loss_e, grad_e = exact.loss_and_grads(*draws(cr, 10 + i))
        assert torch.equal(loss_s, loss_e) and torch.equal(grad_s, grad_e), i
        assert float(grad_s.abs().max()) > 0
    assert {k: v[1].data_ptr() for k, v in shared.eng._bufs.items()} == ptrs and shared.eng.kernels.data_ptr() == kernels_ptr
    with pytest.raises(ValueError, match="capacity"):
        shared.set_topology([n_cap + 1])


@pytest.mark.parametrize("unindexed", [False, True])
def test_shuffled_epoch_builds_one_engine(device, weights_npz, tmp_path, unindexed):
    """arreau_b200.train.fit over a shuffled dataset of ragged crystals: DiffusionLoss keeps ONE capacity-based
    TrainEngine (grown at most a couple of times while the first batches arrive), not one per batch topology -- also when
    the caller names the device torch.device("cuda") while the tensors report "cuda:0" (the flat parameter buffer used to
    be re-created, and `callibrate` read an engine that had never run)."""
    if unindexed:
        device = torch.device("cuda")
    from arreau_b200.diffusion.lattice_dataset import CrystalDataset, save_dataset_npz
    from arreau_b200.lightning_wrappers.diffusion import PONITA_DIFFUSION
    from arreau_b200.synthetic import make_crystals
    from arreau_b200.train import default_args, fit
    cr = make_crystals(40, 1, 12, seed=19)
    off = np.concatenate([[0], np.cumsum(cr.num_atoms)])
    zs = [cr.types[off[i]:off[i + 1]] % 7 + 1 for i in range(40)]
    frac = [cr.frac[off[i]:off[i + 1]] for i in range(40)]
    lat = np.stack([np.diag(cr.lengths[i]) for i in range(40)])
    ds = CrystalDataset([save_dataset_npz(str(tmp_path / "ragged"), zs, lat, frac)])
    torch.manual_seed(0)
    model = PONITA_DIFFUSION(default_args(lr=1e-3, epochs=3, warmup=0), ds.z_table)
    hist = fit(model, ds, epochs=3, batch_size=7, device=device, backward_precision="tf32", log=lambda *_: None)
    assert len(hist) == 3 and all(np.isfinite(hist))
    dl = model.diffusion_loss
    assert len(dl._train_engines) == 1 and dl.train_engine_builds <= 3, dl.train_engine_builds     # 18 steps, <= 3 builds
