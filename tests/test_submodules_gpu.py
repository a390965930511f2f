"""The six sub-modules called on their own (VERDICT r1 item 7, SURVEY section 8b): FactorEncoder (reference module.py:52-67),
AlphaLayer (:78-84), BetaLayer (:92-94), FactorDecoder (:107-123), AttentionLayer (:134-153), FactorPredictor (:169-188).
Each `forward` goes through the C ABI (`fvae_heads_parts`, one launch of the fp32 heads kernel on the caller's stock latents) and
is compared with (1) a float64 restatement of the reference lines written out below and (2) what the UNMODIFIED reference
classes, loaded with our state_dict, returned on the same inputs: tests/golden/submodules_reference.npz, written by
oracle/gen_submodule_golden.py (outputs with more than REF_ROWS rows are stored for a fixed sample of rows).
Tolerance: 2e-5 relative to the output's scale (fp32 kernel vs float64)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "submodules_reference.npz")
REF_ROWS = 48

SHAPES = [dict(N=300, H=20, K=8, M=16), dict(N=517, H=48, K=48, M=64), dict(N=3, H=32, K=5, M=7), dict(N=1000, H=64, K=60, M=128)]


def _close(a, b, tol=2e-5):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(1.0, float(b.abs().max()))
    err = float((a - b).abs().max())
    assert err <= tol * scale, (err, scale)


def _modules(H, K, M, seed=3):
    import factorvae_b200.module as m
    torch.manual_seed(seed)
    enc = m.FactorEncoder(K, M, H)
    dec = m.FactorDecoder(m.AlphaLayer(H), m.BetaLayer(H, K))
    pred = m.FactorPredictor(H, K)
    return m, enc, dec, pred


def _build(H, K, M):
    m, enc, dec, pred = _modules(H, K, M)
    return m, enc.cuda(), dec.cuda(), pred.cuda()


def _p64(mod):
    return {n: p.detach().double().cpu() for n, p in mod.named_parameters()}


def shape_key(shape):
    return "N{N}_H{H}_K{K}_M{M}".format(**shape)


def ref_rows(N):
    """The rows of an (N, ...) output that the golden file keeps: all of them, or a fixed sample of REF_ROWS."""
    if N <= REF_ROWS:
        return np.arange(N)
    return np.sort(np.random.default_rng(N).choice(N, REF_ROWS, replace=False))


def _close_ref(ours, shape, name):
    """`ours` against the reference classes' output stored for this shape (the same rows when a sample is stored)."""
    with np.load(REF_GOLDEN) as z:
        ref = torch.from_numpy(z[f"{shape_key(shape)}:{name}"])
    if ours.dim() == 2 and ours.shape[0] == shape["N"]:
        ours = ours[torch.from_numpy(ref_rows(shape["N"])).to(ours.device)]
    _close(ours, ref)


def _inputs(N, H, seed=11):
    g = torch.Generator().manual_seed(seed)
    e = torch.tanh(torch.randn(N, H, generator=g))          # GRU hidden states live in (-1, 1)
    y = 0.05 * torch.randn(N, 1, generator=g)
    return e, y


def _decoder_noise(N, K):
    g = torch.Generator().manual_seed(5)
    zmu, zsg, eps = torch.randn(K, generator=g), torch.rand(K, generator=g) + 0.1, torch.randn(N, generator=g)
    zsg[K // 2] = 0.0                                                                         # exercises the :117 replacement
    return zmu, zsg, eps


@pytest.mark.parametrize("shape", SHAPES)
def test_factor_encoder_alone(shape, cuda_device):
    N, H, K, M = (shape[k] for k in "NHKM")
    m, enc, _, _ = _build(H, K, M)
    e, y = _inputs(N, H)
    with torch.no_grad():
        mu, sg = enc(e.cuda(), y.cuda())
        mu1, _ = enc(e.cuda(), y.cuda().reshape(-1))                            # returns.dim() == 1 is accepted (:62-63)
    p = _p64(enc)
    w = torch.softmax(e.double() @ p["linear.weight"].T + p["linear.bias"], dim=0)            # :55-56, softmax over stocks
    yp = w.T @ y.double()                                                                     # :64
    mu_r = yp.squeeze(1) @ p["linear_mu.weight"].T + p["linear_mu.bias"]                      # :48
    sg_r = F.softplus(yp.squeeze(1) @ p["linear_sigma.weight"].T + p["linear_sigma.bias"])    # :49
    assert mu.shape == (K,) and sg.shape == (K,)
    _close(mu, mu_r), _close(sg, sg_r), _close(mu1, mu_r)
    _close_ref(mu, shape, "enc_mu"), _close_ref(sg, shape, "enc_sigma")


@pytest.mark.parametrize("shape", SHAPES)
def test_alpha_beta_decoder_alone(shape, cuda_device):
    N, H, K, M = (shape[k] for k in "NHKM")
    m, _, dec, _ = _build(H, K, M)
    e, _ = _inputs(N, H)
    zmu, zsg, eps = _decoder_noise(N, K)
    zsg_dev = zsg.cuda()
    with torch.no_grad():
        amu, asg = dec.alpha_layer(e.cuda())
        beta = dec.beta_layer(e.cuda())
        with m.inject_noise(eps.cuda()):
            ys = dec(e.cuda(), zmu.cuda(), zsg_dev)
    assert amu.shape == (N, 1) and asg.shape == (N, 1) and beta.shape == (N, K) and ys.shape == (N, 1)
    assert float(zsg_dev[K // 2]) == pytest.approx(1e-6)                                      # the caller's tensor, like :117
    p = _p64(dec)
    hid = F.leaky_relu(e.double() @ p["alpha_layer.linear1.weight"].T + p["alpha_layer.linear1.bias"])           # :80-81
    amu_r = hid @ p["alpha_layer.mu_layer.weight"].T + p["alpha_layer.mu_layer.bias"]                            # :82
    asg_r = F.softplus(hid @ p["alpha_layer.sigma_layer.weight"].T + p["alpha_layer.sigma_layer.bias"])          # :83-84
    beta_r = e.double() @ p["beta_layer.linear1.weight"].T + p["beta_layer.linear1.bias"]                        # :93
    zs = zsg.double().clone()
    zs[zs == 0] = 1e-6                                                                                           # :117
    mu_r = amu_r + beta_r @ zmu.double().view(-1, 1)                                                             # :120
    sg_r = torch.sqrt(asg_r ** 2 + (beta_r ** 2) @ (zs.view(-1, 1) ** 2) + 1e-6)                                 # :121
    _close(amu, amu_r), _close(asg, asg_r), _close(beta, beta_r)
    _close(ys, mu_r + eps.double().view(-1, 1) * sg_r)                                                           # :104-105, :123
    _close_ref(amu, shape, "alpha_mu"), _close_ref(asg, shape, "alpha_sigma"), _close_ref(beta, shape, "beta")
    _close_ref(ys, shape, "decoder_y")                                                        # the same eps on both sides
    # Philox draw when nothing is injected: finite, and a different draw on the next call
    with torch.no_grad():
        a = dec(e.cuda(), zmu.cuda(), zsg_dev)
        b = dec(e.cuda(), zmu.cuda(), zsg_dev)
    assert torch.isfinite(a).all() and (N < 2 or not torch.equal(a, b))


def _attention64(p, pre, e, keep=None):
    key = e @ p[pre + "key_layer.weight"].T + p[pre + "key_layer.bias"]                       # :137
    val = e @ p[pre + "value_layer.weight"].T + p[pre + "value_layer.bias"]                   # :138
    a = (p[pre + "query"] @ key.T) / torch.sqrt(torch.tensor(key.shape[1]) + 1e-6).double()   # :140-142
    if keep is not None:
        a = a * keep.double() / 0.9                                                           # :144 (train)
    a = torch.softmax(F.relu(a), dim=0)                                                       # :145-146
    if torch.isnan(a).any() or torch.isinf(a).any():                                          # :149-150
        return torch.zeros_like(val[0])
    return a @ val                                                                            # :152


@pytest.mark.parametrize("shape", SHAPES)
def test_attention_and_predictor_alone(shape, cuda_device):
    N, H, K, M = (shape[k] for k in "NHKM")
    m, _, _, pred = _build(H, K, M)
    e, _ = _inputs(N, H)
    pred.eval()
    with torch.no_grad():
        ctx0 = pred.attention_layers[0](e.cuda())
        ctx_last = pred.attention_layers[K - 1](e.cuda())
        pmu, psg = pred(e.cuda())
    p = _p64(pred)
    ctx = torch.stack([_attention64(p, f"attention_layers.{k}.", e.double()) for k in range(K)])
    assert ctx0.shape == (H,) and pmu.shape == (K,) and psg.shape == (K,)
    _close(ctx0, ctx[0]), _close(ctx_last, ctx[K - 1])
    hm = F.leaky_relu(ctx @ p["linear.weight"].T + p["linear.bias"])                          # :180-181
    _close(pmu, (hm @ p["mu_layer.weight"].T + p["mu_layer.bias"]).view(-1))                  # :182, :185
    _close(psg, F.softplus(hm @ p["sigma_layer.weight"].T + p["sigma_layer.bias"]).view(-1))  # :183-184, :186
    _close_ref(ctx0, shape, "context0"), _close_ref(pmu, shape, "predictor_mu"), _close_ref(psg, shape, "predictor_sigma")
    # train mode: dropout on the scores with an injected keep mask (one column per head)
    pred.train()
    g = torch.Generator().manual_seed(9)
    keep = (torch.rand(N, K, generator=g) > 0.1).to(torch.uint8)
    with torch.no_grad(), m.inject_noise(None, keep.cuda()):
        tmu, tsg = pred(e.cuda())
    with torch.no_grad(), m.inject_noise(None, keep[:, :1].contiguous().cuda()):
        tctx0 = pred.attention_layers[0](e.cuda())
    ctx_t = torch.stack([_attention64(p, f"attention_layers.{k}.", e.double(), keep[:, k]) for k in range(K)])
    _close(tctx0, ctx_t[0])
    hm = F.leaky_relu(ctx_t @ p["linear.weight"].T + p["linear.bias"])
    _close(tmu, (hm @ p["mu_layer.weight"].T + p["mu_layer.bias"]).view(-1))
    _close(tsg, F.softplus(hm @ p["sigma_layer.weight"].T + p["sigma_layer.bias"]).view(-1))
    # the NaN guard: one NaN latent row (a stock whose features hold NaN) poisons the softmax -> the head returns zeros and the
    # prior is the bias path of the shared MLP (:149-150)
    bad = e.clone()
    bad[N // 2, 0] = float("nan")
    pred.eval()
    with torch.no_grad():
        z = pred.attention_layers[0](bad.cuda())
        gmu, gsg = pred(bad.cuda())
    assert torch.count_nonzero(_attention64(p, "attention_layers.0.", bad.double())) == 0
    assert torch.count_nonzero(z) == 0 and z.shape == (H,)
    hm0 = F.leaky_relu(p["linear.bias"]).expand(K, H)
    _close(gmu, (hm0 @ p["mu_layer.weight"].T + p["mu_layer.bias"]).view(-1))
    _close(gsg, F.softplus(hm0 @ p["sigma_layer.weight"].T + p["sigma_layer.bias"]).view(-1))


def test_sub_modules_refuse_cpu_inputs_and_warn_about_autograd(cuda_device):
    m, enc, dec, pred = _build(20, 4, 8)
    e, y = _inputs(50, 20)
    for call in (lambda: enc(e, y), lambda: dec.alpha_layer(e), lambda: dec.beta_layer(e), lambda: pred(e),
                 lambda: pred.attention_layers[0](e), lambda: dec(e, torch.zeros(4), torch.ones(4))):
        with pytest.raises(RuntimeError, match="no CPU"):
            call()
    m._WARNED.discard("BetaLayer")
    with pytest.warns(UserWarning, match="forward-only"):
        out = dec.beta_layer(e.cuda())
    assert not out.requires_grad
