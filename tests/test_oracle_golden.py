"""Pins oracle/vitvq_oracle.py against outputs of the unmodified reference
(tests/golden/*.npz, written by oracle/gen_golden.py in the build container)."""
import os

import numpy as np
import pytest
import torch

from oracle import vitvq_oracle as O


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _t(a):
    return torch.from_numpy(np.asarray(a))


def test_pos_embed_matches_reference(golden_dir):
    g = _load(golden_dir, "pos_embed.npz")
    np.testing.assert_array_equal(O.sincos_pos_embed(64, (4, 4)), g["pos_64_4x4"])
    np.testing.assert_array_equal(O.sincos_pos_embed(96, (4, 6)), g["pos_96_4x6"])
    big = O.sincos_pos_embed(768, (32, 32))
    np.testing.assert_array_equal(big[::37, ::29], g["pos_768_32x32_sample"])
    assert abs(big.astype(np.float64).sum() - float(g["pos_768_32x32_sum"])) < 1e-9
    assert abs(np.abs(big.astype(np.float64)).sum() - float(g["pos_768_32x32_abs"])) < 1e-9


def test_attention_block_fwd_bwd(golden_dir):
    g = _load(golden_dir, "blocks.npz")
    x = _t(g["attn.x"]).requires_grad_(True)
    w_qkv, w_out, b_out = (_t(g[k]).requires_grad_(True) for k in ("attn.w_qkv", "attn.w_out", "attn.b_out"))
    y = O.attention(x, w_qkv, w_out, b_out, heads=2)
    torch.testing.assert_close(y.detach(), _t(g["attn.y"]), rtol=1e-5, atol=1e-6)
    (y * _t(g["attn.g"])).sum().backward()
    for got, key in ((x.grad, "attn.gx"), (w_qkv.grad, "attn.gw_qkv"), (w_out.grad, "attn.gw_out"), (b_out.grad, "attn.gb_out")):
        torch.testing.assert_close(got, _t(g[key]), rtol=1e-4, atol=1e-5)


def test_prenorm_feedforward_fwd_bwd(golden_dir):
    g = _load(golden_dir, "blocks.npz")
    sd = {k[len("ff.sd."):]: _t(g[k]).requires_grad_(True) for k in g.files if k.startswith("ff.sd.")}
    x = _t(g["ff.x"]).requires_grad_(True)
    y = O.feed_forward(O.layer_norm(x, sd["norm.weight"], sd["norm.bias"]), sd["fn.net.0.weight"], sd["fn.net.0.bias"],
                       sd["fn.net.2.weight"], sd["fn.net.2.bias"])
    torch.testing.assert_close(y.detach(), _t(g["ff.y"]), rtol=1e-5, atol=1e-6)
    (y * _t(g["ff.g"])).sum().backward()
    torch.testing.assert_close(x.grad, _t(g["ff.gx"]), rtol=1e-4, atol=1e-5)
    for k, p in sd.items():
        torch.testing.assert_close(p.grad, _t(g["ff.grad." + k]), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("tag,kw", [("plain", {}), ("res4", dict(use_residual=True, num_quantizers=4)),
                                    ("res2", dict(use_residual=True, num_quantizers=2)), ("clustered", {})])
def test_quantizer_matches_reference(golden_dir, tag, kw):
    g = _load(golden_dir, "vq_cases.npz")
    z = _t(g[f"{tag}.z"]).requires_grad_(True)
    E = _t(g[f"{tag}.E"]).requires_grad_(True)
    out, loss, idx = O.vq_forward(z, E, 0.25, **kw)
    np.testing.assert_array_equal(idx.numpy(), g[f"{tag}.idx"])            # indices bit-exact
    assert idx.dtype == torch.int64
    np.testing.assert_array_equal(out.detach().numpy(), g[f"{tag}.zq"])     # same fp32 op sequence
    torch.testing.assert_close(loss.detach(), _t(g[f"{tag}.loss"]), rtol=1e-6, atol=0)
    g_out = _t(g[f"{tag}.g_out"]) if f"{tag}.g_out" in g.files else torch.zeros_like(out)
    g_loss = float(g[f"{tag}.g_loss"]) if f"{tag}.g_loss" in g.files else 1.0
    ((out * g_out).sum() + loss * g_loss).backward()
    torch.testing.assert_close(z.grad, _t(g[f"{tag}.gz"]), rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(E.grad, _t(g[f"{tag}.gE"]), rtol=1e-4, atol=1e-7)
    # the hand-written closed-form backward must agree with the reference's autograd too
    gz, gE = O.vq_backward_np(g[f"{tag}.z"], g[f"{tag}.E"], g[f"{tag}.idx"], g_out.numpy(), g_loss, 0.25,
                              use_residual=bool(kw.get("use_residual")))
    np.testing.assert_allclose(gz, g[f"{tag}.gz"], rtol=2e-4, atol=1e-7)
    np.testing.assert_allclose(gE, g[f"{tag}.gE"], rtol=2e-3, atol=2e-7)
    # and the numpy lookup restatement
    if not kw:
        np.testing.assert_array_equal(O.vq_lookup_np(g[f"{tag}.z"].reshape(-1, 32), g[f"{tag}.E"]).reshape(idx.shape),
                                      g[f"{tag}.idx"])


def test_vitvq_end_to_end_matches_reference(golden_dir):
    g = _load(golden_dir, "vit_tiny.npz")
    sd = {k[3:]: _t(g[k]).clone().requires_grad_(True) for k in g.files if k.startswith("sd.")}
    cfg = dict(image_size=int(g["cfg_image"]), patch_size=int(g["cfg_patch"]),
               encoder=dict(dim=64, depth=2, heads=2, mlp_dim=128), decoder=dict(dim=96, depth=2, heads=3, mlp_dim=160),
               quantizer=dict(embed_dim=32, n_embed=256))
    img = _t(g["img"])
    h = O.vit_encoder(sd, img, patch=8, depth=2, heads=2, prefix="encoder.")
    torch.testing.assert_close(h.detach(), _t(g["enc_out"]), rtol=1e-4, atol=1e-5)
    loss, rec, idx = O.vitvq_loss(sd, img, cfg)
    np.testing.assert_array_equal(idx.numpy(), g["idx"])
    torch.testing.assert_close(rec.detach(), _t(g["rec"]), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(loss.detach(), _t(g["loss"]), rtol=1e-5, atol=1e-6)
    loss.backward()
    n = 0
    for k in g.files:
        if k.startswith("grad."):
            torch.testing.assert_close(sd[k[5:]].grad, _t(g[k]), rtol=2e-3, atol=1e-6, msg=lambda m, k=k: f"{k}: {m}")
            n += 1
    assert n > 10
    # decode_codes path
    with torch.no_grad():
        q = O.decode_codes_embed(idx, sd["quantizer.embedding.weight"], False)
        t = q @ sd["post_quant.weight"].t() + sd["post_quant.bias"]
        d = O.vit_decoder(sd, t, patch=8, depth=2, heads=3, grid_hw=(4, 4), prefix="decoder.")
    torch.testing.assert_close(d, _t(g["decode_codes"]), rtol=1e-4, atol=1e-5)


def test_init_sd_has_reference_keys(golden_dir):
    g = _load(golden_dir, "vit_tiny.npz")
    cfg = dict(image_size=32, patch_size=8, encoder=dict(dim=64, depth=2, heads=2, mlp_dim=128),
               decoder=dict(dim=96, depth=2, heads=3, mlp_dim=160, dim_head=32), quantizer=dict(embed_dim=32, n_embed=256))
    sd = O.init_vitvq_sd(cfg)
    ref = {k[3:]: g[k].shape for k in g.files if k.startswith("sd.")}
    assert set(sd) == set(ref)
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(ref[k]), k
    np.testing.assert_array_equal(sd["encoder.en_pos_embedding"].numpy(), g["sd.encoder.en_pos_embedding"])
    np.testing.assert_array_equal(sd["decoder.de_pos_embedding"].numpy(), g["sd.decoder.de_pos_embedding"])


def test_flops_match_baseline_md():
    assert abs(O.flops_per_image(O.CONFIGS["small"]) / 1e9 - 138.4) < 0.1
    assert abs(O.flops_per_image(O.CONFIGS["base"]) / 1e9 - 426.4) < 0.1
    assert abs(O.flops_per_image(O.CONFIGS["large"]) / 1e9 - 1410.1) < 0.2


def test_oracle_matches_the_vendored_reference_modules(golden_dir):
    """the oracle port against the reference's own layers.py / quantizers.py modules, fwd + bwd, on a config no other
    fixture covers (tests/golden/ref_modules.npz, oracle/gen_golden_live.py: reconstruction and gradients as strided
    samples, gradient norms in full)"""
    from oracle.gen_golden_live import ORACLE_CFG as cfg
    from oracle.seeded import strided_sample
    g = _load(golden_dir, "ref_modules.npz")
    sd = O.init_vitvq_sd(cfg, seed=7)
    img = torch.rand(2, 3, 48, 48, generator=torch.Generator().manual_seed(3))
    sdg = {k: v.clone().requires_grad_(v.is_floating_point() and "pos_embedding" not in k) for k, v in sd.items()}
    loss_o, rec_o, idx_o = O.vitvq_loss(sdg, img, cfg)
    loss_o.backward()
    np.testing.assert_array_equal(idx_o.numpy(), g["oracle.idx"])
    torch.testing.assert_close(strided_sample(rec_o.detach(), 2048), _t(g["oracle.rec"]), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(loss_o.detach(), _t(g["oracle.loss"]), rtol=1e-6, atol=1e-8)
    nograd = set(g["oracle.nograd"].tolist())
    n = 0
    for k, v in sdg.items():
        if k in nograd:
            assert v.grad is None or v.grad.abs().max() == 0
            continue
        torch.testing.assert_close(strided_sample(v.grad), _t(g["oracle.grad." + k]), rtol=1e-4, atol=1e-8, msg=lambda m, k=k: f"{k}: {m}")
        assert abs(v.grad.double().norm().item() - float(g["oracle.gradnorm." + k])) <= 1e-4 * float(g["oracle.gradnorm." + k]) + 1e-8, k
        n += 1
    assert n == sum(1 for k in g.files if k.startswith("oracle.grad."))
