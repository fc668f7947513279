"""Generate the fixtures that pin this package against the reference's own classes, which are not part of this
repository: tests/golden/ref_modules.npz (CPU) and tests/golden/gumbel_cuda.npz (needs a CUDA device: the Gumbel noise
is drawn by the device's generator).

The reference files are imported by path from $B200VQ_REFERENCE (default /root/reference), or from the byte-for-byte
copies oracle/build_ref.py leaves in oracle/_ref/ when the reference tree is absent.  Weights come from
oracle/seeded.py, so the fixtures hold the reference's outputs and strided samples of the larger ones, not its weights.
No reference source is copied; only outputs are stored.

    python oracle/gen_golden_live.py                 # tests/golden/ref_modules.npz
    python oracle/gen_golden_live.py --gumbel [DIR]  # DIR/gumbel_cuda.npz (default tests/golden), on a CUDA device
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import vitvq_oracle as O  # noqa: E402
from oracle.seeded import seeded_state_dict, strided_sample  # noqa: E402

REF = os.environ.get("B200VQ_REFERENCE", "/root/reference")
VENDORED = os.path.join(HERE, "_ref", "enhancing_ref")
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

# the configurations the tests run (tests/test_oracle_golden.py, test_stage2.py, test_gpu_model.py, test_abi_and_boundary.py)
ORACLE_CFG = dict(image_size=48, patch_size=8, encoder=dict(dim=64, depth=2, heads=2, mlp_dim=96, dim_head=32),
                  decoder=dict(dim=64, depth=1, heads=2, mlp_dim=64, dim_head=32),
                  quantizer=dict(embed_dim=32, n_embed=128, use_residual=True, num_quantizers=2))
GPT_FWD_CFG = dict(vocab_cond_size=7, vocab_img_size=33, embed_dim=96, cond_num_tokens=3, img_num_tokens=21, n_heads=3, n_layers=2,
                   mlp_bias=False, attn_bias=False)
GPT_SAMPLE_CFG = dict(vocab_cond_size=6, vocab_img_size=64, embed_dim=64, cond_num_tokens=2, img_num_tokens=9, n_heads=2, n_layers=1)
SAMPLE_KW = (dict(top_k=7), dict(top_p=0.8), dict(top_k=12, top_p=0.6, softmax_temperature=0.7))
NONSQUARE_KW = dict(image_size=(32, 48), patch_size=(8, 4), dim=64, depth=1, heads=2, mlp_dim=128, dim_head=32)
VITVQ_KW = dict(image_size=32, patch_size=8, encoder=dict(dim=64, depth=1, heads=2, mlp_dim=64), quantizer=dict(embed_dim=32, n_embed=128))
GPT_ABI_CFG = dict(vocab_cond_size=10, vocab_img_size=64, embed_dim=64, cond_num_tokens=1, img_num_tokens=16, n_heads=2, n_layers=2)
GUMBEL_KW = dict(embed_dim=32, n_embed=512, temp_init=0.7)


def _load(relpath, vendored_name, modname):
    path = os.path.join(REF, relpath)
    if not os.path.exists(path):
        path = os.path.join(VENDORED, vendored_name)
    if "omegaconf" not in sys.modules:               # stage2/layers.py imports it for a type annotation only
        stub = types.ModuleType("omegaconf")
        stub.OmegaConf = type("OmegaConf", (), {})
        sys.modules["omegaconf"] = stub
    if not hasattr(np, "float"):
        np.float = float                             # stage1/layers.py uses the alias numpy removed in 1.24
    spec = importlib.util.spec_from_file_location(modname, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def stage1():
    return (_load("enhancing/modules/stage1/layers.py", "layers.py", "ref_live.layers"),
            _load("enhancing/modules/stage1/quantizers.py", "quantizers.py", "ref_live.quantizers"))


def param_shapes(module):
    return {k: tuple(p.shape) for k, p in module.named_parameters()}


def _shapes_to_npz(prefix, shapes, out):
    out[prefix + "shapes"] = np.array(sorted(f"{k}={'x'.join(map(str, s))}" for k, s in shapes.items()), dtype=str)


def gen_oracle_case(L, Q, out):
    """ViT-VQ fwd + bwd of the reference modules on the oracle's own initialisation (O.init_vitvq_sd)"""
    cfg = ORACLE_CFG
    sd = O.init_vitvq_sd(cfg, seed=7)
    e, d, q = cfg["encoder"], cfg["decoder"], cfg["quantizer"]
    ref = dict(encoder=L.ViTEncoder(48, 8, **e), decoder=L.ViTDecoder(48, 8, **d), quantizer=Q.VectorQuantizer(**q),
               pre_quant=torch.nn.Linear(64, 32), post_quant=torch.nn.Linear(32, 64))
    for name, m in ref.items():
        m.load_state_dict({k[len(name) + 1:]: v for k, v in sd.items() if k.startswith(name + ".")}, strict=True)
    img = torch.rand(2, 3, 48, 48, generator=torch.Generator().manual_seed(3))
    quant, qloss, idx = ref["quantizer"](ref["pre_quant"](ref["encoder"](img)))
    rec = ref["decoder"](ref["post_quant"](quant))
    loss = ((rec - img) ** 2).mean() + qloss
    loss.backward()
    out.update({"oracle.rec": strided_sample(rec.detach().numpy(), 2048).copy(), "oracle.loss": loss.detach().numpy(),
                "oracle.idx": idx.numpy()})
    nograd = []
    for name, m in ref.items():
        for pn, p in m.named_parameters():
            if p.grad is None:
                nograd.append(f"{name}.{pn}")
            else:
                out[f"oracle.grad.{name}.{pn}"] = strided_sample(p.grad.numpy()).copy()
                out[f"oracle.gradnorm.{name}.{pn}"] = np.float64(p.grad.double().norm())
    out["oracle.nograd"] = np.array(nograd, dtype=str)


def gen_gpt_cases(out):
    S = _load("enhancing/modules/stage2/layers.py", "stage2_layers.py", "ref_live.stage2_layers")
    # forward of a config no other fixture covers (no biases, 3-token prefix)
    ref = S.GPT(**GPT_FWD_CFG)
    shapes = param_shapes(ref)
    ref.load_state_dict(seeded_state_dict(shapes, seed=3, gain=1.2), strict=True)
    g = torch.Generator().manual_seed(3)
    codes = torch.randint(0, 33, (2, 21), generator=g)
    conds = torch.randint(0, 7, (2, 3), generator=g)
    _shapes_to_npz("gptfwd.", shapes, out)
    with torch.no_grad():
        out.update({"gptfwd.codes": codes.numpy(), "gptfwd.conds": conds.numpy(), "gptfwd.logits": ref(codes, conds).numpy()})
    # top-k / nucleus sampling with sharp logits
    ref = S.GPT(**GPT_SAMPLE_CFG).eval()
    shapes = param_shapes(ref)
    ref.load_state_dict(seeded_state_dict(shapes, seed=7, gain=1.6), strict=True)
    _shapes_to_npz("gptsample.", shapes, out)
    conds = torch.randint(0, 6, (3, 2), generator=torch.Generator().manual_seed(7))
    out["gptsample.conds"] = conds.numpy()
    for i, kw in enumerate(SAMPLE_KW):
        torch.manual_seed(123)
        with torch.no_grad():
            logits, drawn = ref.sample(conds, use_fp16=False, **kw)
        out[f"gptsample.{i}.logits"], out[f"gptsample.{i}.codes"] = logits.numpy(), drawn.numpy()
    # what the reference's configure_optimizers sorts GPT parameters by (stage2/transformer.py:141-160): the kind of module
    # that owns each parameter
    ref = S.GPT(**GPT_ABI_CFG)
    kinds = (torch.nn.Linear, torch.nn.LayerNorm, torch.nn.Embedding)
    owners = []
    for mn, m in ref.named_modules():
        for pn, _ in m.named_parameters(recurse=False):
            kind = next((k.__name__ for k in kinds if isinstance(m, k)), "other")
            owners.append(f"{mn + '.' if mn else ''}{pn}:{kind}")
    out["gptabi.owners"] = np.array(sorted(owners), dtype=str)


def gen_nonsquare(L, out):
    """ViTEncoder / ViTDecoder with (height, width) patches; the positional tables are the reference's own"""
    enc, dec = L.ViTEncoder(**NONSQUARE_KW), L.ViTDecoder(**NONSQUARE_KW)
    for tag, m in (("enc", enc), ("dec", dec)):
        shapes = {k: s for k, s in param_shapes(m).items() if "pos_embedding" not in k}
        m.load_state_dict(seeded_state_dict(shapes, seed=11), strict=False)
        _shapes_to_npz(f"nonsquare.{tag}.", shapes, out)
    out["nonsquare.en_pos_embedding"] = enc.en_pos_embedding.detach().numpy()
    out["nonsquare.de_pos_embedding"] = dec.de_pos_embedding.detach().numpy()
    img = torch.rand(2, 3, 32, 48, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        h = enc(img)
        rec = dec(h)
    out.update({"nonsquare.h": strided_sample(h.numpy(), 2048).copy(), "nonsquare.h_absmax": np.float64(h.abs().max()),
                "nonsquare.rec": strided_sample(rec.numpy(), 2048).copy(), "nonsquare.rec_absmax": np.float64(rec.abs().max())})


def gen_vitvq_state_dict(out):
    """state-dict keys and shapes of the reference's ViTVQ (stage1/vitvqgan.py) built from its own classes"""
    saved = dict(sys.modules)
    try:
        def stub(name, **attrs):
            m = types.ModuleType(name)
            m.__dict__.update(attrs)
            sys.modules[name] = m
            return m

        class AttrDict(dict):
            __getattr__ = dict.__getitem__

        stub("omegaconf", OmegaConf=AttrDict)
        stub("pytorch_lightning", LightningModule=torch.nn.Module)
        for pkg in ("enhancing", "enhancing.modules", "enhancing.modules.stage1", "enhancing.utils"):
            stub(pkg).__path__ = []
        stub("enhancing.utils.general", initialize_from_config=lambda cfg: torch.nn.Identity())
        L, Q = stage1()
        sys.modules["enhancing.modules.stage1.layers"], sys.modules["enhancing.modules.stage1.quantizers"] = L, Q
        spec = importlib.util.spec_from_file_location("enhancing.modules.stage1.vitvqgan",
                                                      os.path.join(REF, "enhancing", "modules", "stage1", "vitvqgan.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
        kw = VITVQ_KW
        model = mod.ViTVQ(image_key="image", image_size=kw["image_size"], patch_size=kw["patch_size"], encoder=AttrDict(kw["encoder"]),
                          decoder=AttrDict(kw["encoder"]), quantizer=AttrDict(kw["quantizer"]), loss=AttrDict())
        _shapes_to_npz("vitvq.", {k: tuple(v.shape) for k, v in model.state_dict().items()}, out)
    finally:
        for k in set(sys.modules) - set(saved):
            del sys.modules[k]
        sys.modules.update(saved)


def gen_gumbel():
    """GumbelQuantizer of the reference on the CUDA device, training (soft samples, gradients) and eval (hard samples)"""
    _, Q = stage1()
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {}
    for residual in (False, True):
        tag = "res3" if residual else "plain"
        q = Q.GumbelQuantizer(use_residual=residual, num_quantizers=3 if residual else None, **GUMBEL_KW)
        q.load_state_dict(seeded_state_dict(param_shapes(q), seed=5), strict=True)
        q.cuda()
        z0 = torch.randn(2, 96, 32, generator=torch.Generator().manual_seed(6)).cuda()
        q.train()
        z = z0.clone().requires_grad_(True)
        torch.manual_seed(123)
        zq, loss, idx = q(z)
        (zq.square().mean() + loss).backward()
        out.update({f"{tag}.train.zq": strided_sample(zq.detach().cpu().numpy(), 2048).copy(),
                    f"{tag}.train.zq_absmax": np.float64(zq.detach().abs().max()),
                    f"{tag}.train.loss": loss.detach().cpu().numpy(), f"{tag}.train.idx": idx.cpu().numpy(),
                    f"{tag}.train.ge": strided_sample(q.embedding.weight.grad.cpu().numpy(), 2048).copy(),
                    f"{tag}.train.ge_absmax": np.float64(q.embedding.weight.grad.abs().max())})
        if z.grad is not None:
            out[f"{tag}.train.gz"] = strided_sample(z.grad.cpu().numpy(), 2048).copy()
            out[f"{tag}.train.gz_absmax"] = np.float64(z.grad.abs().max())
        q.eval()
        torch.manual_seed(7)
        with torch.no_grad():
            zq, _, idx = q(z0)
        out.update({f"{tag}.eval.zq": zq[:, ::3].cpu().numpy(), f"{tag}.eval.idx": idx.cpu().numpy()})
    out["device"] = np.array(torch.cuda.get_device_name(0))
    return out


def main():
    torch.set_num_threads(4)
    if "--gumbel" in sys.argv:
        rest = sys.argv[sys.argv.index("--gumbel") + 1:]
        dst = rest[0] if rest else OUT
        os.makedirs(dst, exist_ok=True)
        path = os.path.join(dst, "gumbel_cuda.npz")
        np.savez_compressed(path, **gen_gumbel())
    else:
        if not os.path.isdir(REF):
            sys.exit(f"{REF} not present: the reference fixtures can only be generated next to the reference tree")
        out = {}
        L, Q = stage1()
        gen_oracle_case(L, Q, out)
        gen_gpt_cases(out)
        gen_nonsquare(L, out)
        gen_vitvq_state_dict(out)
        path = os.path.join(OUT, "ref_modules.npz")
        np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
