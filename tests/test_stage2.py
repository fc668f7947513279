"""Stage-2 transformer (SURVEY.md section 8f-3, BASELINE config 5; reference enhancing/modules/stage2/layers.py).

CPU part: oracle/gpt_oracle.py against the reference-generated golden (tests/golden/gpt_tiny.npz, oracle/gen_golden_gpt.py;
tests/golden/ref_modules.npz, oracle/gen_golden_live.py); the replacement's module tree / state-dict keys against the golden's.
GPU part (-m gpu): the new kernels against torch fp64, and `etb.GPT` (forward, backward, sampling steps) against the golden
and the fp64 oracle."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import gpt_oracle as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "gpt_tiny.npz"))
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    cfg = {k[4:]: int(g[k]) for k in g.files if k.startswith("cfg.")}
    return g, sd, cfg


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


# ------------------------------------------------------------------------------------------- CPU
def test_gpt_oracle_matches_reference_golden(golden_dir):
    g, sd, cfg = _golden(golden_dir)
    codes, conds = torch.from_numpy(g["codes"]), torch.from_numpy(g["conds"])
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss, logits = G.gpt_loss(sdg, codes, conds, cfg["n_heads"])
    torch.testing.assert_close(logits.detach(), torch.from_numpy(g["logits"]), rtol=1e-5, atol=1e-6)
    assert abs(loss.item() - float(g["loss"])) < 1e-6
    loss.backward()
    for k in g.files:
        if k.startswith("grad."):
            # key.bias: softmax is invariant to a per-row constant, so this gradient is exactly zero in exact arithmetic
            torch.testing.assert_close(sdg[k[5:]].grad, torch.from_numpy(g[k]), rtol=1e-4, atol=2e-7, msg=lambda m: f"{k}: {m}")


def test_gpt_oracle_sampling_steps_match_reference_golden(golden_dir):
    g, sd, cfg = _golden(golden_dir)
    sl = G.gpt_sample_logits(sd, torch.from_numpy(g["conds"]), torch.from_numpy(g["sample_codes"]), cfg["n_heads"])
    torch.testing.assert_close(sl, torch.from_numpy(g["sample_logits"]), rtol=1e-5, atol=1e-6)


def _seeded_gpt(golden_dir, prefix, cfg, seed, gain):
    """etb.GPT carrying the weights the reference class ran with (oracle/seeded.py), after checking that both have the same
    parameters"""
    import enhancing_transformers_b200 as etb
    from oracle.seeded import parse_shapes, seeded_state_dict
    g = np.load(os.path.join(golden_dir, "ref_modules.npz"))
    shapes = parse_shapes(g[prefix + "shapes"])
    model = etb.GPT(**cfg)
    assert {k: tuple(p.shape) for k, p in model.named_parameters()} == shapes
    model.load_state_dict(seeded_state_dict(shapes, seed=seed, gain=gain), strict=True)
    return g, model


def test_gpt_oracle_matches_the_vendored_reference_class(golden_dir):
    """the oracle's forward against the reference's own GPT on a config no other fixture covers: no biases, 3-token prefix
    (tests/golden/ref_modules.npz, oracle/gen_golden_live.py)"""
    from oracle.seeded import parse_shapes, seeded_state_dict
    g = np.load(os.path.join(golden_dir, "ref_modules.npz"))
    sd = seeded_state_dict(parse_shapes(g["gptfwd.shapes"]), seed=3, gain=1.2)
    codes, conds = torch.from_numpy(g["gptfwd.codes"]), torch.from_numpy(g["gptfwd.conds"])
    torch.testing.assert_close(G.gpt_forward(sd, codes, conds, 3), torch.from_numpy(g["gptfwd.logits"]), rtol=1e-5, atol=1e-6)


def test_gpt_module_tree_and_state_dict_match_reference(golden_dir):
    import enhancing_transformers_b200 as etb
    g, sd, cfg = _golden(golden_dir)
    model = etb.GPT(**cfg)
    own = model.state_dict()
    assert set(own) == set(sd), (set(own) ^ set(sd))
    for k, v in sd.items():
        assert tuple(own[k].shape) == tuple(v.shape), k
    model.load_state_dict(sd, strict=True)
    # what stage2/transformer.py:141-160 (configure_optimizers) sorts parameters by
    kinds = {type(m) for m in model.modules()}
    assert {torch.nn.Linear, torch.nn.LayerNorm, torch.nn.Embedding} <= kinds
    assert isinstance(model.blocks, torch.nn.Sequential) and "mask" not in own           # non-persistent buffer, as in the reference
    blk = model.blocks[0]
    assert torch.equal(blk.attn.mask[0, :3, :3], torch.tensor([[1., 1, 0], [1, 1, 0], [1, 1, 1]]))   # cond_len = 2 prefix block
    torch.testing.assert_close(blk.attn.time_mix.detach().view(-1), torch.arange(64.) / 63)
    # reference init (layers.py:184-192): N(0, 0.02) matrices, zero biases, zero positional tables
    fresh = etb.GPT(**cfg)
    assert abs(fresh.head.weight.std().item() - 0.02) < 0.004 and fresh.pos_emb_code.abs().max().item() == 0
    assert fresh.blocks[1].mlp.p0.bias.abs().max().item() == 0


def test_gpt_rejects_geometries_without_a_kernel():
    import enhancing_transformers_b200 as etb
    with pytest.raises(NotImplementedError, match="head size"):
        etb.GPT(vocab_cond_size=10, vocab_img_size=64, embed_dim=6144, cond_num_tokens=1, img_num_tokens=4, n_heads=16, n_layers=1)
    with pytest.raises(AssertionError):
        etb.GPT(vocab_cond_size=10, vocab_img_size=64, embed_dim=100, cond_num_tokens=1, img_num_tokens=4, n_heads=3, n_layers=1)
    model = etb.GPT(vocab_cond_size=10, vocab_img_size=64, embed_dim=64, cond_num_tokens=1, img_num_tokens=4, n_heads=2, n_layers=1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        model(torch.zeros(2, 4, dtype=torch.int64), torch.zeros(2, 1, dtype=torch.int64))


def test_patch_stage2_rebinds_the_reference_names():
    import enhancing_transformers_b200 as etb
    fake = types.ModuleType("fake_stage2_layers")
    fake.GPT = object
    etb.patch_stage2(fake)
    assert fake.GPT is etb.GPT and fake.Block is etb.stage2.Block and fake.MultiHeadSelfAttention is etb.stage2.MultiHeadSelfAttention


@pytest.mark.parametrize("mode", ["parity", "tf32", "fp16"])
def test_gpt_host_logic_with_emulated_kernels(golden_dir, monkeypatch, mode):
    """stage2.py's autograd wiring / packed-qkv layout / row windows / KV-cache bookkeeping, with every C-ABI call replaced
    by a torch stand-in that follows the contract in include/b200vq.h (tests/emulated_ops.py): the host side alone must
    reproduce the reference golden.  (The kernels themselves are checked on the GPU below.)"""
    import enhancing_transformers_b200 as etb
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emulated_ops
    emulated_ops.install(monkeypatch)
    g, sd, cfg = _golden(golden_dir)
    prev = etb.set_precision(mode)
    try:
        model = etb.GPT(**cfg)
        model.load_state_dict(sd, strict=True)
        codes, conds = torch.from_numpy(g["codes"]), torch.from_numpy(g["conds"])
        logits = model(codes, conds)
        loss = F.cross_entropy(logits.view(-1, logits.shape[-1]), codes.view(-1))
        loss.backward()
        half = mode == "fp16"       # the stand-ins really round operands to fp16 there (the scaling logic depends on the dtype)
        assert _rel(logits.detach(), torch.from_numpy(g["logits"])) < (3e-3 if half else 1e-5)
        for name, p in model.named_parameters():
            want = torch.from_numpy(g["grad." + name])
            if name.endswith("attn.key.bias"):
                assert p.grad.abs().max().item() < 1e-4
                continue
            e = ((p.grad - want).norm() / want.norm().clamp_min(1e-12)).item()
            assert e < (1e-2 if half else 1e-4), (name, e)
        model.eval()
        s_codes = torch.from_numpy(g["sample_codes"])
        past, got = None, []
        for i in range(cfg["img_num_tokens"]):
            lg, past = model.sample_step(None if i == 0 else s_codes[:, i - 1:i], conds,
                                         None if i == 0 else model.pos_emb_code[:, i - 1:i, :], False, past)
            got.append(lg)
        assert _rel(torch.stack(got, 1), torch.from_numpy(g["sample_logits"])) < (3e-3 if half else 1e-5)
        torch.manual_seed(99)                                   # the seed the golden's sampler ran under, same CPU RNG stream
        s_logits, drawn = model.sample(conds, use_fp16=False)
        if not half:
            assert torch.equal(drawn, s_codes)
    finally:
        etb.set_precision(prev)


def test_gpt_sampler_filters_match_the_vendored_reference(golden_dir, monkeypatch):
    """top-k / nucleus filtering and the multinomial draw of GPT.sample (reference stage2/layers.py:228-254): with the kernels
    emulated and the same torch RNG stream, the replacement draws the codes the reference class drew
    (tests/golden/ref_modules.npz, oracle/gen_golden_live.py)"""
    import enhancing_transformers_b200 as etb
    from oracle.gen_golden_live import GPT_SAMPLE_CFG, SAMPLE_KW
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emulated_ops
    emulated_ops.install(monkeypatch)
    prev = etb.set_precision("parity")
    try:
        g, mine = _seeded_gpt(golden_dir, "gptsample.", GPT_SAMPLE_CFG, seed=7, gain=1.6)
        mine.eval()
        conds = torch.from_numpy(g["gptsample.conds"])
        for i, kw in enumerate(SAMPLE_KW):
            l_ref, c_ref = torch.from_numpy(g[f"gptsample.{i}.logits"]), torch.from_numpy(g[f"gptsample.{i}.codes"])
            torch.manual_seed(123)
            l_mine, c_mine = mine.sample(conds, use_fp16=False, **kw)
            assert torch.equal(c_mine, c_ref), kw
            finite = torch.isfinite(l_ref)
            assert torch.equal(finite, torch.isfinite(l_mine))
            torch.testing.assert_close(l_mine[finite], l_ref[finite], rtol=1e-4, atol=1e-5)
    finally:
        etb.set_precision(prev)


# ------------------------------------------------------------------------------------------- GPU kernels
def _mask(T, cond, device):
    m = torch.tril(torch.ones(T, T, device=device, dtype=torch.bool))
    m[:cond, :cond] = True
    return m


def _ref_attention(qkv, B, T, heads, hs, cond):
    q, k, v = (t.view(B, T, heads, hs).transpose(1, 2) for t in qkv.view(B, T, 3, heads * hs).unbind(2))
    att = (q @ k.transpose(-2, -1)) / math.sqrt(hs)
    att = att.masked_fill(~_mask(T, cond, qkv.device), float("-inf")).softmax(-1)
    return (att @ v).transpose(1, 2).reshape(B * T, heads * hs)


@gpu
@pytest.mark.parametrize("exact", [True, False])
@pytest.mark.parametrize("B,T,heads,hs,cond", [(2, 16, 2, 32, 1), (1, 24, 3, 64, 0), (2, 200, 2, 64, 5), (1, 130, 1, 32, 130),
                                               (1, 1025, 2, 64, 1), (2, 257, 2, 64, 70), (1, 64, 1, 64, 3)])
def test_attention_causal_fwd_bwd(exact, B, T, heads, hs, cond):
    from enhancing_transformers_b200 import ops
    torch.manual_seed(T + cond)
    qkv = torch.randn(B * T, 3 * heads * hs, device="cuda")
    dout = torch.randn(B * T, heads * hs, device="cuda")
    if not exact:
        qkv, dout = ops.round_tf32(qkv), ops.round_tf32(dout)
    scale = 1.0 / math.sqrt(hs)
    out, lse = ops.attention_causal_fwd(qkv, B, T, heads, hs, scale, cond, exact)
    dqkv = ops.attention_causal_bwd(qkv, out, lse, dout, B, T, heads, hs, scale, cond, exact)
    q64 = qkv.double().requires_grad_(True)
    ref = _ref_attention(q64, B, T, heads, hs, cond)
    ref.backward(dout.double())
    tol_o, tol_g = (2e-5, 5e-5) if exact else (2e-3, 4e-3)
    assert torch.isfinite(out).all() and torch.isfinite(dqkv).all()
    assert _rel(out.double(), ref.detach()) < tol_o
    assert _rel(dqkv.double(), q64.grad) < tol_g
    # the log-sum-exp the backward recomputes the probabilities from
    q, k, _ = (t.view(B, T, heads, hs).transpose(1, 2) for t in q64.detach().view(B, T, 3, heads * hs).unbind(2))
    s = ((q @ k.transpose(-2, -1)) * scale).masked_fill(~_mask(T, cond, "cuda"), float("-inf"))
    assert (lse.double().view(B, heads, T) - torch.logsumexp(s, -1)).abs().max().item() < (1e-4 if exact else 2e-3)


@gpu
def test_attention_causal_full_prefix_equals_unmasked_core():
    """cond_len == T makes every key visible: the masked entry point must then agree with the stage-1 kernels bit for bit"""
    from enhancing_transformers_b200 import ops
    torch.manual_seed(1)
    B, T, heads, hs = 2, 200, 2, 64
    qkv = torch.randn(B * T, 3 * heads * hs, device="cuda")
    scale = hs ** -0.5
    o1, l1 = ops.attention_exact_fwd(qkv, B, T, heads, hs, scale)
    o2, l2 = ops.attention_causal_fwd(qkv, B, T, heads, hs, scale, T, True)
    assert torch.equal(o1, o2) and torch.equal(l1, l2)


@gpu
@pytest.mark.parametrize("B,T,C", [(2, 7, 64), (3, 130, 256), (1, 1025, 1024)])
def test_time_mix_is_bit_identical_to_the_reference_ops(B, T, C):
    from enhancing_transformers_b200 import ops
    torch.manual_seed(C)
    x = torch.randn(B, T, C, device="cuda")
    w = torch.rand(1, 1, C, device="cuda")
    shift = torch.nn.ZeroPad2d((0, 0, 1, -1))
    ref = x * w + shift(x) * (1 - w)                                    # reference stage2/layers.py:58, fp32 on the GPU
    got = ops.time_mix_fwd(x.view(B * T, C), w.view(-1), T)
    assert torch.equal(got.view(B, T, C), ref)
    g = torch.randn(B * T, C, device="cuda")
    x64, w64 = x.double().requires_grad_(True), w.double().requires_grad_(True)
    (x64 * w64 + shift(x64) * (1 - w64)).backward(g.view(B, T, C).double())
    gx, gw = ops.time_mix_bwd(g, x.view(B * T, C), w.view(-1), T)
    assert _rel(gx.double().view(B, T, C), x64.grad) < 1e-6
    assert _rel(gw.double(), w64.grad.view(-1)) < 1e-5


@gpu
def test_sqrelu_token_embed_copy_rows():
    from enhancing_transformers_b200 import ops
    torch.manual_seed(0)
    x = torch.randn(130, 256, device="cuda")
    g = torch.randn_like(x)
    assert torch.equal(ops.sqrelu(x), torch.square(torch.relu(x)))
    xr = x.clone().requires_grad_(True)
    torch.square(torch.relu(xr)).backward(g)
    torch.testing.assert_close(ops.sqrelu(x, g), xr.grad, rtol=1e-6, atol=0)
    # embeddings + positional tables, and their dense gradients
    B, Tc, Ti, C, Vc, Vi = 3, 2, 37, 64, 11, 50
    Wc, Wi = torch.randn(Vc, C, device="cuda"), torch.randn(Vi, C, device="cuda")
    pc, pi = torch.randn(1, Tc, C, device="cuda"), torch.randn(1, Ti, C, device="cuda")
    conds = torch.randint(0, Vc, (B, Tc), device="cuda")
    codes = torch.randint(0, 4, (B, Ti), device="cuda")                 # few distinct codes: contended scatter
    got = ops.token_embed_fwd(conds, codes, Wc, pc, Wi, pi).view(B, Tc + Ti, C)
    ref = torch.cat([F.embedding(conds, Wc) + pc, F.embedding(codes, Wi) + pi], dim=1)
    assert torch.equal(got, ref)
    gg = torch.randn(B * (Tc + Ti), C, device="cuda")
    leaves = [t.double().requires_grad_(True) for t in (Wc, pc, Wi, pi)]
    torch.cat([F.embedding(conds, leaves[0]) + leaves[1], F.embedding(codes, leaves[2]) + leaves[3]], dim=1).backward(
        gg.view(B, Tc + Ti, C).double())
    gWc, gpc, gWi, gpi = ops.token_embed_bwd(conds, codes, gg, Vc, Vi)
    for a, b in ((gWc, leaves[0].grad), (gpc, leaves[1].grad[0]), (gWi, leaves[2].grad), (gpi, leaves[3].grad[0])):
        assert _rel(a.double(), b) < 1e-5
    # row windows
    src = torch.randn(B * 9, C, device="cuda")
    win = ops.copy_rows(src, B, 9, 5, 2, 0, 5)
    assert torch.equal(win.view(B, 5, C), src.view(B, 9, C)[:, 2:7])
    back = ops.copy_rows(win, B, 5, 9, 0, 2, 5).view(B, 9, C)
    assert torch.equal(back[:, 2:7], win.view(B, 5, C)) and back[:, :2].abs().max().item() == 0 and back[:, 7:].abs().max().item() == 0


@gpu
@pytest.mark.parametrize("heads,hs,pos", [(2, 32, 0), (3, 64, 17), (2, 64, 1024)])
def test_decode_attention_against_torch(heads, hs, pos):
    from enhancing_transformers_b200 import ops
    torch.manual_seed(pos)
    B, C, Tmax = 3, heads * hs, 1025
    ck, cv = torch.randn(B, Tmax, C, device="cuda"), torch.randn(B, Tmax, C, device="cuda")
    qkv = torch.randn(B, 3 * C, device="cuda")
    k_ref, v_ref = ck.clone(), cv.clone()
    k_ref[:, pos], v_ref[:, pos] = qkv[:, C:2 * C], qkv[:, 2 * C:]
    out = ops.decode_attention(qkv, ck, cv, heads, hs, pos, hs ** -0.5)
    assert torch.equal(ck, k_ref) and torch.equal(cv, v_ref)           # the step's key / value rows were appended
    q = qkv[:, :C].double().view(B, heads, 1, hs)
    K = k_ref[:, :pos + 1].double().view(B, pos + 1, heads, hs).transpose(1, 2)
    V = v_ref[:, :pos + 1].double().view(B, pos + 1, heads, hs).transpose(1, 2)
    ref = (((q @ K.transpose(-2, -1)) * hs ** -0.5).softmax(-1) @ V).reshape(B, C)
    assert _rel(out.double(), ref) < 1e-5


# ------------------------------------------------------------------------------------------- GPU model
def _gpt_on_gpu(sd, cfg):
    import enhancing_transformers_b200 as etb
    model = etb.GPT(**cfg)
    model.load_state_dict(sd, strict=True)
    return model.cuda()


@gpu
@pytest.mark.parametrize("mode,tol_logit,tol_grad", [("parity", 1e-4, 1e-3), ("tf32", 1e-2, 3e-2), ("fp16", 1e-2, 3e-2)])
def test_gpt_matches_reference_golden(golden_dir, mode, tol_logit, tol_grad):
    """forward logits, cross-entropy loss and every parameter gradient of the reference's own GPT (tiny config);
    north_star tolerance for logits: 1e-3 relative -- the parity data path is asserted at 1e-4"""
    import enhancing_transformers_b200 as etb
    g, sd, cfg = _golden(golden_dir)
    prev = etb.set_precision(mode)
    try:
        model = _gpt_on_gpu(sd, cfg)
        codes, conds = torch.from_numpy(g["codes"]).cuda(), torch.from_numpy(g["conds"]).cuda()
        n0 = etb.ops.launch_count()
        logits = model(codes, conds)
        loss = F.cross_entropy(logits.view(-1, logits.shape[-1]), codes.view(-1))
        loss.backward()
        torch.cuda.synchronize()
        assert etb.ops.launch_count() - n0 > 60                      # the CUDA path ran
    finally:
        etb.set_precision(prev)
    ref = torch.from_numpy(g["logits"])
    r = _rel(logits.detach().cpu(), ref)
    print(f"gpt_tiny [{mode}] logits rel err {r:.2e}, loss {loss.item():.6f} vs {float(g['loss']):.6f}")
    assert r < tol_logit
    assert abs(loss.item() - float(g["loss"])) < tol_logit * abs(float(g["loss"])) * 10
    worst = 0.0
    for name, p in model.named_parameters():
        want = torch.from_numpy(g["grad." + name])
        assert p.grad is not None, name
        if name.endswith("attn.key.bias"):                             # exactly zero in exact arithmetic (softmax shift invariance)
            assert p.grad.abs().max().item() < 1e-5
            continue
        e = ((p.grad.cpu() - want).norm() / want.norm().clamp_min(1e-12)).item()
        worst = max(worst, e)
        assert e < tol_grad, (name, e)
    print(f"gpt_tiny [{mode}] worst parameter-gradient rel-l2 {worst:.2e}")


@gpu
@pytest.mark.parametrize("mode,tol", [("parity", 1e-4), ("fp16", 1e-2)])
def test_gpt_sampling_steps_match_reference_golden(golden_dir, mode, tol):
    """GPT.sample_step fed the codes the reference drew reproduces the logits the reference drew them from
    (KV cache, one-token time mixing, unmasked cached attention: reference layers.py:264-303)"""
    import enhancing_transformers_b200 as etb
    g, sd, cfg = _golden(golden_dir)
    prev = etb.set_precision(mode)
    try:
        model = _gpt_on_gpu(sd, cfg).eval()
        conds = torch.from_numpy(g["conds"]).cuda()
        codes = torch.from_numpy(g["sample_codes"]).cuda()
        past, got = None, []
        for i in range(cfg["img_num_tokens"]):
            c = None if i == 0 else codes[:, i - 1:i]
            pos = None if i == 0 else model.pos_emb_code[:, i - 1:i, :]
            lg, past = model.sample_step(c, conds, pos, False, past)
            got.append(lg)
        got = torch.stack(got, dim=1).cpu()
        # and the public sampler runs end to end on the device
        torch.manual_seed(0)
        s_logits, s_codes = model.sample(conds, top_k=5, top_p=0.9, use_fp16=False)
    finally:
        etb.set_precision(prev)
    r = _rel(got, torch.from_numpy(g["sample_logits"]))
    print(f"gpt_tiny [{mode}] sampling-step logits rel err {r:.2e}")
    assert r < tol
    assert s_codes.shape == (3, cfg["img_num_tokens"]) and s_codes.min().item() >= 0 and s_codes.max().item() < cfg["vocab_img_size"]
    assert s_logits.shape == (3, cfg["img_num_tokens"] * cfg["vocab_img_size"])      # the reference concatenates the [B, vocab] steps along dim 1


@gpu
@pytest.mark.parametrize("mode,tol", [("parity", 1e-4), ("tf32", 1e-2), ("fp16", 1e-2)])
def test_gpt_base_shaped_sequence_vs_fp64_oracle(mode, tol):
    """config 5's sequence geometry (1 class token + 32 x 32 codes = 1025 positions, 8192-entry vocabulary) at a width the
    kernels cover (embed_dim 256, 64-wide heads), against the oracle evaluated in fp64 on the GPU"""
    import enhancing_transformers_b200 as etb
    cfg = dict(vocab_cond_size=1000, vocab_img_size=8192, embed_dim=256, cond_num_tokens=1, img_num_tokens=1024, n_heads=4, n_layers=2)
    torch.manual_seed(11)
    model = etb.GPT(**cfg)
    with torch.no_grad():
        model.pos_emb_code.normal_(0, 0.1)
        model.pos_emb_cond.normal_(0, 0.1)
        for p in model.parameters():
            if p.dim() == 2:
                p.mul_(4.0)
    model = model.cuda()
    codes = torch.randint(0, 8192, (2, 1024), device="cuda")
    conds = torch.randint(0, 1000, (2, 1), device="cuda")
    prev = etb.set_precision(mode)
    try:
        logits = model(codes, conds)
        loss = F.cross_entropy(logits.view(-1, 8192), codes.view(-1))
        loss.backward()
    finally:
        etb.set_precision(prev)
    sd64 = {k: v.detach().double().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}
    loss64, logits64 = G.gpt_loss(sd64, codes, conds, 4)
    loss64.backward()
    r = _rel(logits.detach().double(), logits64.detach())
    worst = max(((p.grad.double() - sd64[n].grad).norm() / sd64[n].grad.norm().clamp_min(1e-12)).item()
                for n, p in model.named_parameters() if not n.endswith("attn.key.bias"))
    print(f"gpt 1025-token [{mode}] logits rel err {r:.2e}, worst grad rel-l2 {worst:.2e}, loss {loss.item():.5f} vs {loss64.item():.5f}")
    assert r < tol and worst < 30 * tol
