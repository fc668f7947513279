"""GPU parity of the nn.Module boundary: the replacement ViTEncoder / ViTDecoder / VectorQuantizer (+ QuantLinear
pre/post_quant), wired as ViTVQ.forward wires them (vitvqgan.py:44-72), against the reference's own outputs
(golden fixtures) and against the oracle sharing one state_dict -- at the miniature configs on the CPU oracle and
at the BASELINE configs (base, base + residual depth 4, large) on the oracle evaluated in fp64 on the GPU.

Tolerances (north_star: codes bit-exact on identical z; reconstructions within 1e-3 relative, fp32), written at
each assert as max|err| / max|ref|:
  precision "parity" (3xTF32)   every stage < 5e-5 (measured ~1e-6): the margin against the 1e-3 tolerance
  precision "fp16" / "tf32"     tf32-level rounding: < 1e-3 at tiny/small; at the 24- and 40-layer BASELINE configs
                                the measured decoder error is ~1.0e-3 (DESIGN.md section 2), asserted < 1.5e-3 and
                                reported, not hidden.
The decoder is always checked on the *oracle's own codes* (no skip when a near-tie flips a code end to end)."""
import os

import numpy as np
import pytest
import torch

import enhancing_transformers_b200 as etb
from oracle import vitvq_oracle as O

pytestmark = pytest.mark.gpu
MODES = ("fp16", "tf32", "parity")


def relmax(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


@pytest.fixture(autouse=True)
def _restore_precision():
    prev = etb.get_precision()
    yield
    etb.set_precision(prev)


def build(cfg, sd):
    e, d, q = cfg["encoder"], cfg["decoder"], cfg["quantizer"]
    mods = dict(encoder=etb.ViTEncoder(cfg["image_size"], cfg["patch_size"], **e),
                decoder=etb.ViTDecoder(cfg["image_size"], cfg["patch_size"], **d),
                quantizer=etb.VectorQuantizer(**q),
                pre_quant=etb.QuantLinear(e["dim"], q["embed_dim"]), post_quant=etb.QuantLinear(q["embed_dim"], d["dim"]))
    for name, m in mods.items():
        m.load_state_dict({k[len(name) + 1:]: v for k, v in sd.items() if k.startswith(name + ".")}, strict=True)
        m.cuda()
    return mods


def run(mods, img):
    h = mods["encoder"](img)
    z = mods["pre_quant"](h)
    zq, qloss, idx = mods["quantizer"](z)
    rec = mods["decoder"](mods["post_quant"](zq))
    return ((rec - img) ** 2).mean() + qloss, rec, idx, h, z


def decode(mods, codes):
    """ViTVQ.decode_codes (vitvqgan.py:81-90)"""
    with torch.no_grad():
        return mods["decoder"](mods["post_quant"](mods["quantizer"].embed_codes(codes)))


def audit_flipped_codes(idx, idx_ref, z, z_ref, E):
    """codes may differ end to end only where the reference's own distance gap is within what the measured
    perturbation of the (normalised) z can bridge: d = 2 - 2 zn.en moves by <= 2|dzn| per candidate"""
    idx, idx_ref = idx.reshape(-1, idx.shape[-1]) if idx.dim() == 3 else idx.reshape(-1, 1), \
        idx_ref.reshape(-1, idx_ref.shape[-1]) if idx_ref.dim() == 3 else idx_ref.reshape(-1, 1)
    bad = (idx[:, 0] != idx_ref[:, 0]).nonzero().view(-1).cpu().numpy()      # depth 0 sees z itself
    if bad.size == 0:
        return 0.0
    zn = torch.nn.functional.normalize(z.reshape(-1, 32).double(), dim=-1)
    zr = torch.nn.functional.normalize(z_ref.reshape(-1, 32).double(), dim=-1)
    dz = (zn - zr).norm(dim=-1).max().item()
    gaps = O.vq_top2_gap_f64(z_ref.reshape(-1, 32).double().cpu().numpy()[bad], E.double().cpu().numpy())
    assert (gaps <= 4 * dz + 1e-6).all(), (gaps.max(), dz)
    return float(gaps.max())


GOLD_CFG = dict(image_size=32, patch_size=8, encoder=dict(dim=64, depth=2, heads=2, mlp_dim=128),
                decoder=dict(dim=96, depth=2, heads=3, mlp_dim=160, dim_head=32), quantizer=dict(embed_dim=32, n_embed=256))
FWD_TOL = {"fp16": 1e-3, "tf32": 1e-3, "parity": 5e-5}
GRAD_TOL = {"fp16": 5e-3, "tf32": 5e-3, "parity": 1e-4}


@pytest.mark.parametrize("mode", MODES)
def test_against_reference_golden_fwd_bwd(golden_dir, mode):
    """the reference's own outputs (tests/golden/vit_tiny.npz, written by oracle/gen_golden.py from /root/reference)"""
    etb.set_precision(mode)
    g = np.load(os.path.join(golden_dir, "vit_tiny.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    mods = build(GOLD_CFG, sd)
    loss, rec, idx, h, z = run(mods, torch.from_numpy(g["img"]).cuda())
    tol = FWD_TOL[mode]
    assert relmax(h.cpu(), torch.from_numpy(g["enc_out"])) < tol
    assert relmax(z.cpu(), torch.from_numpy(g["z"])) < tol
    # codes: bit-exact on identical z ...
    assert torch.equal(idx.cpu(), O.vq_forward(z.detach().cpu(), sd["quantizer.embedding.weight"])[2])
    # ... and end to end up to near-ties bridged by the encoder's rounding (none at all in parity mode)
    gidx = torch.from_numpy(g["idx"])
    audit_flipped_codes(idx.cpu(), gidx, z.detach().cpu(), torch.from_numpy(g["z"]), sd["quantizer.embedding.weight"])
    if mode == "parity":
        assert torch.equal(idx.cpu(), gidx)
    # decoder on the reference's codes: always checked
    assert relmax(decode(mods, gidx.cuda()).cpu(), torch.from_numpy(g["decode_codes"])) < tol
    if torch.equal(idx.cpu(), gidx):
        assert relmax(rec.cpu(), torch.from_numpy(g["rec"])) < tol
        assert abs(loss.item() - float(g["loss"])) < tol * float(g["loss"])
    loss.backward()
    for k in g.files:
        if k.startswith("grad."):
            mod, _, pname = k[5:].partition(".")
            p = dict(mods[mod].named_parameters())[pname]
            ref = torch.from_numpy(g[k])
            rel = ((p.grad.cpu() - ref).norm() / ref.norm().clamp_min(1e-30)).item()
            assert rel < GRAD_TOL[mode], (k, rel)
    with torch.no_grad():
        q = mods["quantizer"].embed_codes(gidx.cuda())
        q2 = mods["quantizer"].norm(mods["quantizer"].embedding(gidx.cuda()))
        assert torch.allclose(q, q2, atol=1e-6)


@pytest.mark.parametrize("mode", ["fp16", "parity"])
def test_post_quant_with_positional_table_in_the_epilogue(golden_dir, mode):
    """SURVEY.md section 8f-1 (opt-in `etb.fuse_post_quant_pos`): post_quant's GEMM adds de_pos_embedding in its epilogue and
    the decoder skips its own add.  Same fp32 operations in the same order as the separate path: identical reconstruction,
    identical decode_codes (vs the reference golden too), identical gradients; state-dict keys unchanged."""
    etb.set_precision(mode)
    g = np.load(os.path.join(golden_dir, "vit_tiny.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    img = torch.from_numpy(g["img"]).cuda()
    gidx = torch.from_numpy(g["idx"]).cuda()

    class Holder(torch.nn.Module):      # the attribute names ViTVQ uses (vitvqgan.py:35-39)
        def __init__(self, mods):
            super().__init__()
            for k, v in mods.items():
                setattr(self, k, v)

    def grads(mods):
        loss, rec, idx, _, _ = run(mods, img)
        loss.backward()
        return rec.detach(), idx, {f"{m}.{n}": p.grad.clone() for m, mod in mods.items() for n, p in mod.named_parameters() if p.grad is not None}

    plain = build(GOLD_CFG, sd)
    rec0, idx0, g0 = grads(plain)
    fused = build(GOLD_CFG, sd)
    holder = Holder(fused)
    keys = set(holder.state_dict())
    etb.fuse_post_quant_pos(holder)
    assert set(holder.state_dict()) == keys and isinstance(holder.post_quant, etb.PosQuantLinear)
    fused["post_quant"] = holder.post_quant
    rec1, idx1, g1 = grads(fused)
    assert torch.equal(idx0, idx1)
    assert relmax(rec1, rec0) < 1e-6
    assert relmax(decode(fused, gidx).cpu(), torch.from_numpy(g["decode_codes"])) < FWD_TOL[mode]
    assert set(g0) == set(g1)
    for k in g0:
        assert ((g1[k] - g0[k]).norm() / g0[k].norm().clamp_min(1e-30)).item() < 1e-5, k
    etb.fuse_post_quant_pos(holder, False)
    assert not holder.decoder.pos_added_upstream and type(holder.post_quant) is etb.QuantLinear


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,B", [("tiny", 3), ("small", 1)])
def test_against_oracle_shared_state_dict(name, B, mode):
    etb.set_precision(mode)
    cfg = O.CONFIGS[name]
    sd = O.init_vitvq_sd(cfg, seed=1)
    img = torch.rand(B, 3, cfg["image_size"], cfg["image_size"], generator=torch.Generator().manual_seed(2))
    sdg = {k: v.clone().requires_grad_(v.is_floating_point() and "pos_embedding" not in k) for k, v in sd.items()}
    loss_ref, rec_ref, idx_ref = O.vitvq_loss(sdg, img, cfg)
    loss_ref.backward()
    mods = build(cfg, sd)
    loss, rec, idx, h, z = run(mods, img.cuda())
    loss.backward()
    assert torch.equal(idx.cpu(), O.vq_forward(z.detach().cpu(), sd["quantizer.embedding.weight"])[2])
    agree = (idx.cpu() == idx_ref).float().mean().item()
    assert agree > (0.9999 if mode == "parity" else 0.985), agree      # tiny: 192 tokens, one near-tie flip = 0.5 %
    tol = FWD_TOL[mode]
    assert relmax(decode(mods, idx_ref.cuda()).cpu(), rec_ref.detach()) < tol          # decoder on the oracle's codes
    if agree == 1.0:
        assert relmax(rec.cpu(), rec_ref.detach()) < tol
        assert abs(loss.item() - loss_ref.item()) < tol * abs(loss_ref.item())
    else:
        assert abs(loss.item() - loss_ref.item()) < 5e-3 * abs(loss_ref.item())
    for k, v in sdg.items():
        if v.grad is None or v.grad.norm() == 0:
            continue
        mod, _, pname = k.partition(".")
        p = dict(mods[mod].named_parameters())[pname]
        rel = ((p.grad.cpu() - v.grad).norm() / v.grad.norm()).item()
        assert rel < (5e-2 if agree < 1.0 else GRAD_TOL[mode]), (k, rel)      # a flipped code is a different decoder input


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs 2 / 3 / 4 (reference configs/imagenet_vitvq_base.yaml:7-19, imagenet_vitvq_large.yaml:7-19)
# against the oracle evaluated in float64 on the GPU
# ------------------------------------------------------------------------------------------------
BASELINE_CASES = [("base", 2, "fp16"), ("base", 2, "tf32"), ("base", 2, "parity"), ("base_rq4", 2, "fp16"),
                  ("base_rq4", 2, "parity"), ("large", 1, "fp16"), ("large", 1, "parity")]


@pytest.mark.parametrize("name,B,mode", BASELINE_CASES)
def test_baseline_config_parity_vs_fp64_oracle(name, B, mode):
    torch.backends.cuda.matmul.allow_tf32 = False
    etb.set_precision(mode)
    cfg = O.CONFIGS[name]
    sd = O.init_vitvq_sd(cfg, seed=0)
    img = torch.rand(B, 3, 256, 256, generator=torch.Generator().manual_seed(0)).cuda()
    qc = cfg["quantizer"]
    E = sd["quantizer.embedding.weight"].cuda()
    p, g = cfg["patch_size"], cfg["image_size"] // cfg["patch_size"]
    e, d = cfg["encoder"], cfg["decoder"]
    # ---- oracle in float64 (the quantiser lookup itself in fp32 on the fp64 z, as the reference computes it)
    sd64 = {k: v.double().cuda().requires_grad_(v.is_floating_point() and "pos_embedding" not in k) for k, v in sd.items()}
    h64 = O.vit_encoder(sd64, img.double(), patch=p, depth=e["depth"], heads=e["heads"], prefix="encoder.")
    z64 = h64 @ sd64["pre_quant.weight"].t() + sd64["pre_quant.bias"]
    with torch.no_grad():
        _, _, idx64 = O.vq_forward(z64.float(), E, qc.get("beta", 0.25), qc.get("use_residual", False), qc.get("num_quantizers"))
    zq64, qloss64, _ = _vq_with_codes_f64(z64, sd64["quantizer.embedding.weight"], idx64, qc)
    t64 = zq64 @ sd64["post_quant.weight"].t() + sd64["post_quant.bias"]
    rec64 = O.vit_decoder(sd64, t64, patch=p, depth=d["depth"], heads=d["heads"], grid_hw=(g, g), prefix="decoder.")
    loss64 = ((rec64 - img.double()) ** 2).mean() + qloss64
    loss64.backward()
    # ---- replacement modules
    mods = build(cfg, sd)
    loss, rec, idx, h, z = run(mods, img)
    loss.backward()
    fast = mode != "parity"
    tol = 1.5e-3 if fast else 5e-5
    errs = dict(enc=relmax(h, h64.detach()), z=relmax(z, z64.detach()))
    assert errs["enc"] < (1e-3 if fast else 5e-5), errs
    assert errs["z"] < (1e-3 if fast else 5e-5), errs
    # codes bit-exact on identical z (same fp32 lookup), end-to-end agreement, audited flips
    with torch.no_grad():
        _, _, idx_same = O.vq_forward(z.detach(), E, qc.get("beta", 0.25), qc.get("use_residual", False), qc.get("num_quantizers"))
    ntok = idx.numel() // (idx.shape[-1] if idx.dim() == 3 else 1)
    tok_same = (idx == idx_same).reshape(ntok, -1).all(dim=1)
    n_mism = int((~tok_same).sum())     # torch's fp32 GEMM order vs the kernel's sequential FMA: exact fp32 near-ties only
    assert n_mism <= max(2, ntok // 5000), n_mism
    if n_mism:
        bad = (~tok_same).nonzero().view(-1).cpu().numpy()
        assert (O.vq_top2_gap_f64(z.detach().reshape(-1, 32).double().cpu().numpy()[bad], E.double().cpu().numpy()) < 2e-6).all()
    tok_agree = (idx == idx64).reshape(ntok, -1).all(dim=1)
    agree = tok_agree.float().mean().item()
    errs["code_agreement"] = agree
    errs["tokens_differing"] = int((~tok_agree).sum())
    # parity mode: only exact fp32 near-ties may differ (a few tokens in thousands); fast modes: tf32-level z rounding
    depth = idx.shape[-1] if idx.dim() == 3 else 1      # every depth is one more lookup that a near-tie can flip
    assert (errs["tokens_differing"] <= max(2, ntok // 5000)) if not fast else (agree >= 1.0 - 0.008 * depth), errs
    audit_flipped_codes(idx, idx64, z.detach(), z64.detach(), E)
    # decoder fed the ORACLE'S codes: the reconstruction tolerance proper
    dec = decode(mods, idx64)
    errs["dec_on_oracle_codes"] = relmax(dec, rec64.detach())
    assert errs["dec_on_oracle_codes"] < tol, errs
    # the same comparison under two stricter readings of "relative", reported next to it (DESIGN.md section 2):
    # relative l2 over the image, and the 99.9th percentile of the per-pixel error relative to the per-image RMS
    diff = (dec.double() - rec64.detach())
    errs["dec_rel_l2"] = (diff.norm() / rec64.detach().norm()).item()
    rms = rec64.detach().pow(2).mean(dim=(1, 2, 3), keepdim=True).sqrt()
    errs["dec_p999_over_rms"] = torch.quantile((diff.abs() / rms).flatten()[:4_000_000].float(), 0.999).item()
    assert errs["dec_rel_l2"] < tol, errs
    if agree == 1.0:
        assert relmax(rec, rec64.detach()) < tol and abs(loss.item() - loss64.item()) < tol * abs(loss64.item()), errs
    else:
        assert abs(loss.item() - loss64.item()) < 5e-3 * abs(loss64.item()), errs
    # parameter gradients (rel-l2); with flipped codes the decoder input differs slightly -> looser bound
    gtol = (2e-2 if agree < 1.0 else 5e-3) if fast else (5e-3 if agree < 1.0 else 2e-4)
    worst = ("", 0.0)
    for k, v in sd64.items():
        if v.grad is None or v.grad.norm() == 0:
            continue
        mod, _, pname = k.partition(".")
        pp = dict(mods[mod].named_parameters())[pname]
        rel = ((pp.grad.double() - v.grad).norm() / v.grad.norm()).item()
        worst = max(worst, (k, rel), key=lambda t: t[1])
        assert rel < gtol, (k, rel, errs)
    print(f"\n[parity] {name} B={B} {mode}: " + " ".join(f"{k}={v:.3e}" for k, v in errs.items()) + f" worst-grad {worst[0]} {worst[1]:.2e}")


def _vq_with_codes_f64(z, E, idx, qc):
    """quantizers.py:38-63,85-92 in float64 with the code indices given (so that the fp64 graph follows the fp32 lookup)"""
    beta = qc.get("beta", 0.25)

    def one(r, i):
        zq_n, z_n = O.l2norm(E[i]), O.l2norm(r)
        return zq_n, beta * ((zq_n.detach() - z_n) ** 2).mean() + ((zq_n - z_n.detach()) ** 2).mean()
    if not qc.get("use_residual", False):
        zq, loss = one(z, idx)
    else:
        zq, r, losses = torch.zeros_like(z), z.detach().clone(), []
        for t in range(int(qc["num_quantizers"])):
            q, l = one(r, idx[..., t])
            r, zq = r - q, zq + q
            losses.append(l)
        loss = torch.stack(losses, dim=-1).mean()
    return z + (zq - z).detach(), loss, idx


def test_residual_quantizer_module_and_modes():
    """use_residual=True, num_quantizers=4 (BASELINE config 3) + eval/no_grad + double forward"""
    torch.manual_seed(0)
    vq = etb.VectorQuantizer(embed_dim=32, n_embed=512, use_residual=True, num_quantizers=4).cuda()
    z = torch.randn(2, 64, 32, device="cuda", requires_grad=True)
    zq, loss, idx = vq(z)
    assert idx.shape == (2, 64, 4) and idx.dtype == torch.int64
    ref = O.vq_forward(z.detach().cpu().requires_grad_(True), vq.embedding.weight.detach().cpu().requires_grad_(True), 0.25, True, 4)
    assert torch.equal(idx.cpu(), ref[2])
    assert torch.allclose(zq.detach().cpu(), ref[0].detach(), atol=1e-6)
    (zq.sum() + loss).backward()
    assert torch.allclose(z.grad, torch.ones_like(z))          # residual mode: z only gets the straight-through gradient
    vq.eval()
    with torch.no_grad():
        zq2, loss2, idx2 = vq(z)
        assert torch.equal(idx2, idx)
        q = vq.embed_codes(idx)
        assert torch.allclose(q, zq2, atol=1e-5)


def test_unnormalised_quantizer_module():
    """use_norm=False (quantizers.py:24) through the module surface, against plain torch autograd"""
    torch.manual_seed(0)
    vq = etb.VectorQuantizer(embed_dim=32, n_embed=128, use_norm=False).cuda()
    z = torch.randn(2, 40, 32, device="cuda", requires_grad=True)
    zq, loss, idx = vq(z)
    E = vq.embedding.weight
    d = (z.detach().reshape(-1, 32) ** 2).sum(1, keepdim=True) + (E.detach() ** 2).sum(1) - 2 * z.detach().reshape(-1, 32) @ E.detach().t()
    assert (idx.view(-1) == d.argmin(1)).float().mean() > 0.99
    q = E[idx]
    lref = 0.25 * ((q.detach() - z) ** 2).mean() + ((q - z.detach()) ** 2).mean()
    assert abs(loss.item() - lref.item()) < 1e-5 * lref.item()
    assert torch.allclose(vq.embed_codes(idx), vq.norm(vq.embedding(idx)), atol=1e-6)


@pytest.mark.parametrize("mode", MODES)
def test_sub_modules_run_standalone(mode):
    etb.set_precision(mode)
    torch.manual_seed(0)
    attn = etb.Attention(64, heads=2, dim_head=32).cuda()
    ff = etb.PreNorm(64, etb.FeedForward(64, 96)).cuda()
    x = torch.randn(2, 24, 64, device="cuda", requires_grad=True)
    y = ff(attn(x))
    xr = x.detach().cpu().requires_grad_(True)
    sd = {k: v.detach().cpu() for k, v in list(attn.state_dict().items()) + list(ff.state_dict().items())}
    a = O.attention(xr, sd["to_qkv.weight"], sd["to_out.weight"], sd["to_out.bias"], 2)
    yr = O.feed_forward(O.layer_norm(a, sd["norm.weight"], sd["norm.bias"]), sd["fn.net.0.weight"], sd["fn.net.0.bias"],
                        sd["fn.net.2.weight"], sd["fn.net.2.bias"])
    assert relmax(y.detach().cpu(), yr.detach()) < (1e-4 if mode == "parity" else 2e-3)
    y.sum().backward(); yr.sum().backward()
    assert relmax(x.grad.cpu(), xr.grad) < (1e-4 if mode == "parity" else 5e-3)


def test_single_head_identity_projection_transformer():
    """heads == 1 and dim_head == dim: to_out is nn.Identity (reference layers.py:112,120)"""
    torch.manual_seed(0)
    tr = etb.Transformer(64, 2, 1, 64, 128).cuda()
    assert isinstance(tr.layers[0][0].fn.to_out, torch.nn.Identity)
    x = torch.randn(2, 24, 64, device="cuda", requires_grad=True)
    y = tr(x)
    sd = {k: v.detach().cpu() for k, v in tr.state_dict().items()}
    xr = x.detach().cpu().requires_grad_(True)
    h = xr
    for i in range(2):
        hn = O.layer_norm(h, sd[f"layers.{i}.0.norm.weight"], sd[f"layers.{i}.0.norm.bias"])
        qkv = hn @ sd[f"layers.{i}.0.fn.to_qkv.weight"].t()
        q, k, v = qkv.chunk(3, dim=-1)
        h = torch.softmax(q @ k.transpose(-1, -2) * 64 ** -0.5, -1) @ v + h
        hn = O.layer_norm(h, sd[f"layers.{i}.1.norm.weight"], sd[f"layers.{i}.1.norm.bias"])
        h = O.feed_forward(hn, sd[f"layers.{i}.1.fn.net.0.weight"], sd[f"layers.{i}.1.fn.net.0.bias"],
                           sd[f"layers.{i}.1.fn.net.2.weight"], sd[f"layers.{i}.1.fn.net.2.bias"]) + h
    yr = O.layer_norm(h, sd["norm.weight"], sd["norm.bias"])
    assert relmax(y.detach().cpu(), yr.detach()) < 2e-3
    wsum = torch.randn(2, 24, 64)                 # (a plain .sum() of LayerNorm outputs has zero gradient)
    (y * wsum.cuda()).sum().backward(); (yr * wsum).sum().backward()
    assert relmax(x.grad.cpu(), xr.grad) < 5e-3


def test_weight_shadows_track_every_kind_of_update():
    """the tensor-core copy of a weight must follow in-place updates, must not leak between parameters that happen
    to be allocated at the same device address, must see `.data` writes outside autograd recording, and a refresh
    must not clobber the copy a still-pending backward holds (ADVICE round 1)"""
    from enhancing_transformers_b200 import functional as Fn
    torch.manual_seed(0)
    x = torch.randn(64, 64, device="cuda")

    def ref_of(ff):
        sd = {k: v.detach().cpu() for k, v in ff.state_dict().items()}
        return O.feed_forward(x.cpu(), sd["net.0.weight"], sd["net.0.bias"], sd["net.2.weight"], sd["net.2.bias"])
    outs = []
    for seed in (1, 2, 3):                       # fresh modules of identical shape: the allocator recycles addresses
        torch.manual_seed(seed)
        ff = etb.FeedForward(64, 96).cuda()
        y = ff(x)
        assert relmax(y.detach().cpu(), ref_of(ff)) < 2e-3
        outs.append(y.detach().clone())
        del ff, y
    assert not torch.allclose(outs[0], outs[1])
    ff = etb.FeedForward(64, 96).cuda()
    y0 = ff(x).detach().clone()
    with torch.no_grad():
        ff.net[0].weight.mul_(0.5)               # what an optimizer step does: bumps the version counter
    y1 = ff(x).detach()
    assert relmax(y1.cpu(), ref_of(ff)) < 2e-3 and not torch.allclose(y0, y1)
    # .data write (EMA swap) outside autograd recording: picked up without any explicit call
    ff.net[0].weight.data.mul_(2.0)
    with torch.no_grad():
        y2 = ff(x)
    assert relmax(y2.cpu(), ref_of(ff)) < 2e-3 and torch.allclose(y2, y0, rtol=1e-3, atol=1e-4)
    # .data write between two grad-enabled forwards: needs invalidate_shadows
    ff(x)
    ff.net[0].weight.data.mul_(0.5)
    etb.invalidate_shadows(ff)
    assert relmax(ff(x).detach().cpu(), ref_of(ff)) < 2e-3
    # forward -> in-place weight update -> forward -> backward(first graph): like stock torch this must RAISE (the
    # Functions save the parameter itself, so autograd's version check sees the update), never return gradients
    # computed from a half-refreshed copy; and a refresh never overwrites the buffer an older graph holds
    xg = x.clone().requires_grad_(True)
    w0 = ff.net[0].weight.detach().clone()
    ya = ff(xg)
    sh_old = Fn.weight_shadow(ff.net[0].weight, "tf32")
    with torch.no_grad():
        ff.net[0].weight.add_(1.0)
    ff(xg)
    assert torch.equal(sh_old, Fn.ops.round_tf32(w0)) and Fn.weight_shadow(ff.net[0].weight, "tf32") is not sh_old
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        ya.sum().backward()


def test_autocast_inputs_are_cast_to_fp32():
    """reference main.py --use_amp: under torch.autocast the unchanged nn.Linear pre/post_quant produce fp16;
    the replacement modules must accept that (ADVICE round 1)"""
    cfg = O.CONFIGS["tiny"]
    sd = O.init_vitvq_sd(cfg, seed=4)
    mods = build(cfg, sd)
    mods["pre_quant"] = torch.nn.Linear(cfg["encoder"]["dim"], 32).cuda()          # stock nn.Linear -> fp16 under autocast
    mods["post_quant"] = torch.nn.Linear(32, cfg["decoder"]["dim"]).cuda()
    for name in ("pre_quant", "post_quant"):
        mods[name].load_state_dict({k[len(name) + 1:]: v for k, v in sd.items() if k.startswith(name + ".")})
    img = torch.rand(2, 3, 64, 64, device="cuda")
    with torch.autocast("cuda", dtype=torch.float16):
        loss, rec, idx, h, z = run(mods, img)
    assert z.dtype == torch.float16 and rec.dtype == torch.float32 and torch.isfinite(loss)
    loss.backward()
    assert all(torch.isfinite(p.grad).all() for m in mods.values() for p in m.parameters() if p.grad is not None)
    loss32, rec32, *_ = run(mods, img)
    assert relmax(rec, rec32.detach()) < 2e-2          # fp16 z: a different quantiser input, same pipeline


def test_wrong_device_is_rejected(monkeypatch):
    if torch.cuda.device_count() < 2:
        x = torch.randn(64, 64, device="cuda")
        monkeypatch.setattr(torch.cuda, "current_device", lambda: 1)
        with pytest.raises(RuntimeError, match="current CUDA device"):
            etb.ops.round_tf32(x)
    else:
        with pytest.raises(RuntimeError, match="current CUDA device"):
            etb.ops.round_tf32(torch.randn(64, 64, device="cuda:1"))


def test_frozen_model_backward_skips_parameter_gradients():
    """reference stage2/transformer.py:44-46 freezes stage 1: only the input gradient is wanted"""
    enc = etb.ViTEncoder(32, 8, dim=64, depth=2, heads=2, mlp_dim=128, dim_head=32).cuda()
    img = torch.rand(2, 3, 32, 32, device="cuda", requires_grad=True)
    g_full = torch.autograd.grad(enc(img).square().mean(), img)[0]
    for p in enc.parameters():
        p.requires_grad_(False)
    n0 = etb.ops.launch_count()
    g_frozen = torch.autograd.grad(enc(img).square().mean(), img)[0]
    n_frozen = etb.ops.launch_count() - n0
    assert torch.allclose(g_full, g_frozen, rtol=1e-5, atol=1e-9)
    for p in enc.parameters():
        p.requires_grad_(True)
    n0 = etb.ops.launch_count()
    enc(img).square().mean().backward()
    assert n_frozen < etb.ops.launch_count() - n0


def test_non_square_patches_match_the_reference_modules(golden_dir):
    """reference layers.py:157-166 accepts (height, width) patches; checked against the reference's own modules
    (tests/golden/ref_modules.npz, oracle/gen_golden_live.py: outputs as strided samples, the reference's positional tables)"""
    from oracle.gen_golden_live import NONSQUARE_KW as kw
    from oracle.seeded import parse_shapes, seeded_state_dict, strided_sample
    g = np.load(os.path.join(golden_dir, "ref_modules.npz"))
    etb.set_precision("parity")
    enc, dec = etb.ViTEncoder(**kw), etb.ViTDecoder(**kw)
    for tag, m, pos in (("enc", enc, "en_pos_embedding"), ("dec", dec, "de_pos_embedding")):
        sd = seeded_state_dict(parse_shapes(g[f"nonsquare.{tag}.shapes"]), seed=11)
        sd[pos] = torch.from_numpy(g["nonsquare." + pos])
        m.load_state_dict(sd, strict=True)
    enc.cuda(); dec.cuda()
    img = torch.rand(2, 3, 32, 48, generator=torch.Generator().manual_seed(0))
    h = enc(img.cuda())
    assert h.shape == (2, 48, 64)

    def rel(a, key):
        return ((strided_sample(a.detach().cpu(), 2048).double() - torch.from_numpy(g[key]).double()).abs().max()
                / float(g[key + "_absmax"])).item()
    assert rel(h, "nonsquare.h") < 5e-5
    assert rel(dec(h), "nonsquare.rec") < 5e-5
    with pytest.raises(NotImplementedError, match="multiple of 4"):
        etb.ViTEncoder(image_size=30, patch_size=6, dim=64, depth=1, heads=2, mlp_dim=64)


@pytest.mark.parametrize("residual", [False, True])
def test_gumbel_quantizer_matches_reference(golden_dir, residual):
    """reference quantizers.py:95-126 (SURVEY.md section 8 f-4).  The quantiser is stochastic; with the generator seeded
    identically F.gumbel_softmax draws the same noise on the same device, so the soft sample, the KL loss and the
    gradients the reference class produced on a B200 with TF32 matmuls off (tests/golden/gumbel_cuda.npz,
    oracle/gen_golden_live.py --gumbel: strided samples) are reproduced up to the rounding of the logits; in eval mode (hard
    one-hot of a noisy arg-max) the indices agree except at near-ties."""
    from oracle.gen_golden_live import GUMBEL_KW
    from oracle.seeded import seeded_state_dict, strided_sample
    g = np.load(os.path.join(golden_dir, "gumbel_cuda.npz"))
    tag = "res3" if residual else "plain"
    torch.backends.cuda.matmul.allow_tf32 = False
    ours = etb.GumbelQuantizer(use_residual=residual, num_quantizers=3 if residual else None, **GUMBEL_KW)
    ours.load_state_dict(seeded_state_dict({k: tuple(p.shape) for k, p in ours.named_parameters()}, seed=5), strict=True)
    ours.cuda()
    z0 = torch.randn(2, 96, 32, generator=torch.Generator().manual_seed(6)).cuda()

    def rel(a, key):
        return ((strided_sample(a.detach().cpu(), 2048).double() - torch.from_numpy(g[key]).double()).abs().max()
                / float(g[key + "_absmax"])).item()
    # training mode: soft samples, gradients through the sample
    ours.train()
    z = z0.clone().requires_grad_(True)
    torch.manual_seed(123)
    zq_o, l_o, i_o = ours(z)
    (zq_o.square().mean() + l_o).backward()
    i_r, l_r = torch.from_numpy(g[f"{tag}.train.idx"]), float(g[f"{tag}.train.loss"])
    assert i_o.shape == i_r.shape and i_o.dtype == torch.int64
    assert rel(zq_o, f"{tag}.train.zq") < 2e-4 and abs(l_o.item() - l_r) < 1e-5 * max(1.0, abs(l_r))
    assert (i_o.cpu() == i_r).float().mean() > 0.99
    if f"{tag}.train.gz" not in g.files:      # residual mode quantises a detached copy of z (quantizers.py:43) and has no straight-through term
        assert z.grad is None
    else:
        assert rel(z.grad, f"{tag}.train.gz") < 2e-3
    assert rel(ours.embedding.weight.grad, f"{tag}.train.ge") < 2e-3
    # eval mode: hard samples (every third token stored)
    ours.eval()
    torch.manual_seed(7)
    with torch.no_grad():
        zq_o, _, i_o = ours(z0)
    i_r = torch.from_numpy(g[f"{tag}.eval.idx"])
    assert (i_o.cpu() == i_r).float().mean() > 0.99
    same = (i_o.cpu() == i_r)[:, ::3]
    same = same.all(-1) if residual else same
    assert relmax(zq_o[:, ::3].cpu()[same], torch.from_numpy(g[f"{tag}.eval.zq"])[same]) < 1e-4
