"""Pin the oracle (oracle/bbb_oracle.py) against fixtures produced by the
UNMODIFIED reference (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import bbb_oracle as O

CFG_PRIORS = {"prior_mu": 0, "prior_sigma": 0.1,
              "posterior_mu_initial": (0, 0.1), "posterior_rho_initial": (-5, 0.1)}


def layer_names(g):
    return sorted({k.split("/")[0] for k in g})


def load_case(g, name):
    d = {k.split("/", 1)[1]: g[k] for k in g if k.startswith(name + "/")}
    t = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) and v.dtype == np.float32 and v.ndim > 0 else v)
         for k, v in d.items()}
    return t


def run_oracle_layer(name, c, dtype=torch.float32):
    conv = None
    if "conv" in c:
        s = [int(v) for v in c["conv"]]
        conv = ((s[0], s[1]), (s[2], s[3]), (s[4], s[5]))
    f = lambda k: c[k].to(dtype) if k in c else None
    pm, ps = float(c["prior"][0]), float(c["prior"][1])
    if "_bbb_" in name:
        y = O.bbb_forward(f("x"), f("W_mu"), f("W_rho"), f("bias_mu"), f("bias_rho"),
                          f("eps_w"), f("eps_b"), conv)
        ym = O.bbb_forward(f("x"), f("W_mu"), f("W_rho"), f("bias_mu"), f("bias_rho"),
                           None, None, conv, sample=False)
    else:
        y = O.lrt_forward(f("x"), f("W_mu"), f("W_rho"), f("bias_mu"), f("bias_rho"), f("eps_y"), conv)
        ym = O.lrt_forward(f("x"), f("W_mu"), f("W_rho"), f("bias_mu"), f("bias_rho"), None, conv,
                           sample=False)
    kl = O.kl_loss(f("W_mu"), f("W_rho"), f("bias_mu"), f("bias_rho"), pm, ps)
    return y, ym, kl


def test_layer_cases_bitwise(golden_layers):
    torch.set_num_threads(1)
    names = layer_names(golden_layers)
    assert len(names) >= 19
    for name in names:
        c = load_case(golden_layers, name)
        y, ym, kl = run_oracle_layer(name, c)
        assert torch.equal(y, c["y"]), name
        assert torch.equal(ym, c["y_mean"]), name
        assert float(kl) == pytest.approx(float(c["kl"]), rel=1e-6), name


def test_layer_cases_float64_budget(golden_layers):
    """fp64 restatement vs the reference's fp32: the fp32 rounding budget that the
    1e-3 parity bar has to absorb is ~1e-6 of the output scale."""
    for name in layer_names(golden_layers):
        c = load_case(golden_layers, name)
        y, _, kl = run_oracle_layer(name, c, torch.float64)
        ref = c["y"].double()
        assert (y - ref).abs().max() <= 2e-5 * ref.abs().max(), name
        assert float(kl) == pytest.approx(float(c["kl"]), rel=1e-5), name


def test_model_cases(golden_models):
    torch.set_num_threads(1)
    names = layer_names(golden_models)
    assert len(names) == 7
    for name in names:
        c = load_case(golden_models, name)
        key, inputs, outputs, variant, act, batch = [str(v) for v in c["meta"]]
        inputs, outputs, batch = int(inputs), int(outputs), int(batch)
        params = O.init_params(key, outputs, inputs, CFG_PRIORS, seed=123)
        sums = [float(p[k].double().sum()) for p in params for k in ("W_mu", "W_rho", "bias_mu", "bias_rho")]
        np.testing.assert_allclose(sums, c["param_sums"], rtol=0, atol=0)
        eps = O.draw_eps_like_reference(O.eps_shapes(key, outputs, inputs, variant, batch), seed=7)
        logits, kl = O.net_forward(key, params, c["x"], eps, variant, act, 0.0, 0.1, outputs)
        assert torch.equal(logits, c["logits"]), name
        assert float(kl) == pytest.approx(float(c["kl"]), rel=1e-6), name


def test_kl_is_prior_to_posterior():
    """SURVEY D1: the executed formula is KL(prior || posterior)."""
    mu = torch.tensor([0.3]); rho = torch.tensor([-1.0])
    s = float(O.softplus_sigma(rho)); sp, mp = 0.1, 0.0
    want = 0.5 * (2 * np.log(s / sp) - 1 + (sp / s) ** 2 + ((0.3 - mp) / s) ** 2)
    got = float(O.kl_loss(mu, rho, None, None, mp, sp))
    assert got == pytest.approx(want, rel=1e-6)
    tb = float(O.kl_textbook(mu, rho, None, None, mp, sp))
    assert tb == pytest.approx(np.log(sp / s) + (s * s + 0.09) / (2 * sp * sp) - 0.5, rel=1e-6)
    assert abs(tb - got) > 1.0


def test_mc_combine_and_uncertainty_match_reference_loops():
    g = torch.Generator().manual_seed(3)
    logits = [torch.randn(5, 10, generator=g) for _ in range(7)]
    # main_bayesian.py:43-53 restated literally
    outputs = torch.zeros(5, 10, 7)
    for j, l in enumerate(logits):
        outputs[:, :, j] = torch.nn.functional.log_softmax(l, dim=1)
    assert torch.allclose(O.mc_combine(logits), O.logmeanexp(outputs, 2))
    # uncertainty_estimation.py:80-96 per-image numpy loop
    pred, epi, ale, ent = O.uncertainty(logits)
    T = 7
    for i in range(5):
        p_hat = np.stack([torch.softmax(l, 1)[i].numpy() for l in logits]).astype(np.float64)
        p_bar = p_hat.mean(0)
        tmp = p_hat - p_bar[None]
        e = np.diag(tmp.T @ tmp / T)
        a = np.diag(np.diag(p_bar) - p_hat.T @ p_hat / T)
        np.testing.assert_allclose(epi[i].numpy(), e, rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(ale[i].numpy(), a, rtol=1e-5, atol=1e-9)


def test_philox_known_answer():
    """Random123 kat_vectors: philox4x32-10, ctr=0 key=0 and the all-ones vector."""
    r = O.philox4x32_10(np.zeros((1, 4), np.uint32), np.zeros(2, np.uint32))[0]
    assert [hex(int(v)) for v in r] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    r = O.philox4x32_10(np.full((1, 4), 0xFFFFFFFF, np.uint32), np.full(2, 0xFFFFFFFF, np.uint32))[0]
    assert [hex(int(v)) for v in r] == ["0x408f276d", "0x41c83b0e", "0xa20bc7c6", "0x6d5451fd"]


def test_philox_normal_moments():
    z = O.philox_normal(1 << 18, seed=1234, stream=5)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    assert abs((z ** 3).mean()) < 0.03 and abs((z ** 4).mean() - 3) < 0.08
    z2 = O.philox_normal(100, seed=1234, stream=5, offset=1000)
    assert np.array_equal(z2, z[1000:1100])
