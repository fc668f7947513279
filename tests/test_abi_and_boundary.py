"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol
include/b200vq.h declares, the nn.Module surface matches the reference's constructor /
state-dict contract (SURVEY.md section 8b), and the product path refuses to run on CPU."""
import inspect
import os
import re

import numpy as np
import pytest
import torch

import enhancing_transformers_b200 as etb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "b200vq.h")).read()
    declared = set(re.findall(r"\b(b200vq_\w+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = etb._lib.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in b200vq.h but not exported by libb200vq.so"
    assert declared == set(etb._lib.EXPORTS), declared ^ set(etb._lib.EXPORTS)
    assert lib.b200vq_version() == 202
    assert lib.b200vq_arch() == b"sm_100a"


def test_ctypes_signatures_match_the_header_prototypes():
    """every prototype in include/b200vq.h, parameter by parameter, against the ctypes table the host side calls
    through (a hand-edited ABI must not drift: a missing argument would shift every later one silently)"""
    import ctypes
    hdr = open(os.path.join(ROOT, "include", "b200vq.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    protos = re.findall(r"([\w ]+?[\s\*])\s*(b200vq_\w+)\s*\(([^)]*)\)\s*;", hdr)
    assert len(protos) == len(etb._lib.EXPORTS)

    def kind_of_c(decl: str) -> str:
        decl = decl.strip()
        if decl in ("void", ""):
            return ""
        if "*" in decl:
            return "ptr"
        base = decl.rsplit(" ", 1)[0].strip()
        return {"int": "int", "long long": "ll", "size_t": "size", "float": "float"}[base]

    kind_of_ctypes = {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_int: "int", ctypes.c_longlong: "ll",
                      ctypes.c_size_t: "size", ctypes.c_float: "float"}
    for ret, name, params in protos:
        restype, argtypes = etb._lib._SIGNATURES[name]
        want = [k for k in (kind_of_c(p) for p in params.split(",")) if k]
        got = [kind_of_ctypes[a] for a in argtypes]
        assert got == want, f"{name}: header {want} vs ctypes {got}"
        assert kind_of_ctypes[restype] == ("ptr" if "*" in ret else kind_of_c(ret.strip() + " x")), name


def test_cpu_tensors_are_rejected_loudly():
    enc = etb.ViTEncoder(image_size=32, patch_size=8, dim=64, depth=1, heads=2, mlp_dim=64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        enc(torch.rand(1, 3, 32, 32))
    vq = etb.VectorQuantizer(embed_dim=32, n_embed=64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        vq(torch.randn(1, 4, 32))
    etb.VectorQuantizer(embed_dim=32, n_embed=64, use_norm=False)      # reference-legal (quantizers.py:24): constructs


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from enhancing_transformers_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()


def test_constructor_signatures_match_reference():
    # reference layers.py:154-155,186-187 and quantizers.py:67-68 (keyword names are API: YAML dicts are splatted)
    for cls in (etb.ViTEncoder, etb.ViTDecoder):
        params = list(inspect.signature(cls.__init__).parameters)
        assert params == ["self", "image_size", "patch_size", "dim", "depth", "heads", "mlp_dim", "channels", "dim_head"]
        sig = inspect.signature(cls.__init__)
        assert sig.parameters["channels"].default == 3 and sig.parameters["dim_head"].default == 64
    sig = inspect.signature(etb.VectorQuantizer.__init__)
    assert list(sig.parameters) == ["self", "embed_dim", "n_embed", "beta", "use_norm", "use_residual", "num_quantizers", "kwargs"]
    assert sig.parameters["beta"].default == 0.25 and sig.parameters["use_norm"].default is True


def test_state_dict_keys_and_shapes_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "vit_tiny.npz"))
    ref = {k[3:]: g[k] for k in g.files if k.startswith("sd.")}
    enc = etb.ViTEncoder(image_size=32, patch_size=8, dim=64, depth=2, heads=2, mlp_dim=128)
    dec = etb.ViTDecoder(image_size=32, patch_size=8, dim=96, depth=2, heads=3, mlp_dim=160, dim_head=32)
    vq = etb.VectorQuantizer(embed_dim=32, n_embed=256)
    for pfx, mod in (("encoder.", enc), ("decoder.", dec), ("quantizer.", vq)):
        mine = {pfx + k: tuple(v.shape) for k, v in mod.state_dict().items()}
        theirs = {k: tuple(v.shape) for k, v in ref.items() if k.startswith(pfx)}
        assert mine == theirs
        mod.load_state_dict({k[len(pfx):]: torch.from_numpy(v) for k, v in ref.items() if k.startswith(pfx)}, strict=True)
    # the positional tables are rebuilt bit-exactly and are frozen parameters inside the state dict
    np.testing.assert_array_equal(etb.ViTEncoder(32, 8, 64, 1, 2, 64).en_pos_embedding.numpy(), ref["encoder.en_pos_embedding"])
    assert not enc.en_pos_embedding.requires_grad and not dec.de_pos_embedding.requires_grad
    assert dec.get_last_layer() is dec.to_pixel[-1].weight
    assert enc.num_patches == 16 and enc.patch_dim == 192


def test_quantizer_attributes_read_by_lightning_module():
    vq = etb.VectorQuantizer(embed_dim=32, n_embed=64, use_residual=True, num_quantizers=4)
    assert vq.use_residual is True and vq.num_quantizers == 4 and vq.straight_through is True
    code = torch.tensor([[1, 2, 3, 4]])
    q = vq.norm(vq.embedding(code))              # vitvqgan.py:82-83 on CPU tensors still works (plain torch)
    assert q.shape == (1, 4, 32)
    torch.testing.assert_close(q.norm(dim=-1), torch.ones(1, 4))


def test_init_distributions_follow_reference():
    torch.manual_seed(0)
    enc = etb.ViTEncoder(image_size=64, patch_size=8, dim=256, depth=1, heads=4, mlp_dim=512)
    lin = enc.transformer.layers[0][1].fn.net[0]
    bound = (6.0 / (256 + 512)) ** 0.5
    assert lin.weight.abs().max() <= bound and lin.weight.abs().max() > 0.9 * bound
    assert torch.count_nonzero(lin.bias) == 0
    ln = enc.transformer.norm
    assert torch.all(ln.weight == 1) and torch.all(ln.bias == 0)
    w = enc.to_patch_embedding[0].weight
    assert w.abs().max() <= (6.0 / (256 + 192)) ** 0.5
    vq = etb.VectorQuantizer(32, 4096)
    assert abs(vq.embedding.weight.std().item() - 1.0) < 0.05


def _vitvqgan_stand_in():
    """a module laid out like the reference's stage1/vitvqgan.py as far as this package touches it: module-level names
    Encoder / Decoder / VectorQuantizer that ViTVQ.__init__ looks up when it runs, plain nn.Linear pre/post_quant, and a
    training_step that runs the whole autoencoder and hands the reconstruction to the loss with the optimizer index"""
    import types

    mod = types.ModuleType("vitvqgan_stand_in")

    class ViTVQ(torch.nn.Module):
        def __init__(self, image_size, patch_size, encoder, decoder, quantizer, loss):
            super().__init__()
            self.image_key, self.loss, self.global_step = "image", loss, 0
            self.encoder = mod.Encoder(image_size=image_size, patch_size=patch_size, **encoder)
            self.decoder = mod.Decoder(image_size=image_size, patch_size=patch_size, **decoder)
            self.quantizer = mod.VectorQuantizer(**quantizer)
            self.pre_quant = torch.nn.Linear(encoder["dim"], quantizer["embed_dim"])
            self.post_quant = torch.nn.Linear(quantizer["embed_dim"], decoder["dim"])

        def encode(self, x):
            quant, qloss, _ = self.quantizer(self.pre_quant(self.encoder(x)))
            return quant, qloss

        def decode(self, quant):
            return self.decoder(self.post_quant(quant))

        def forward(self, x):
            quant, qloss = self.encode(x)
            return self.decode(quant), qloss

        def training_step(self, batch, batch_idx, optimizer_idx=0):
            x = batch[self.image_key]
            xrec, qloss = self(x)
            loss, _ = self.loss(qloss, x, xrec, optimizer_idx, self.global_step, batch_idx,
                                last_layer=self.decoder.get_last_layer(), split="train")
            return loss

    mod.ViTVQ = ViTVQ
    return mod


def test_unchanged_lightning_module_constructs_with_patched_classes(golden_dir, monkeypatch):
    """a ViTVQ built on the replacement classes has the state-dict keys and shapes of the reference's own ViTVQ
    (stage1/vitvqgan.py built from its own classes: tests/golden/ref_modules.npz, oracle/gen_golden_live.py), whether the
    names resolve through install_as_reference_modules() or are rebound by patch(); SURVEY.md section 8c"""
    import sys
    import types

    from oracle.gen_golden_live import VITVQ_KW as kw
    from oracle.seeded import parse_shapes
    want = parse_shapes(np.load(os.path.join(golden_dir, "ref_modules.npz"))["vitvq.shapes"])
    for n in ("enhancing.modules.stage1.layers", "enhancing.modules.stage1.quantizers"):
        monkeypatch.delitem(sys.modules, n, raising=False)
    etb.install_as_reference_modules()
    mod = _vitvqgan_stand_in()
    # what the reference's `from .layers import ViTEncoder as Encoder, ...` binds once the package's classes are installed
    mod.Encoder = sys.modules["enhancing.modules.stage1.layers"].ViTEncoder
    mod.Decoder = sys.modules["enhancing.modules.stage1.layers"].ViTDecoder
    mod.VectorQuantizer = sys.modules["enhancing.modules.stage1.quantizers"].VectorQuantizer
    assert mod.Encoder is etb.ViTEncoder and mod.Decoder is etb.ViTDecoder and mod.VectorQuantizer is etb.VectorQuantizer

    def build():
        return mod.ViTVQ(kw["image_size"], kw["patch_size"], kw["encoder"], kw["encoder"], kw["quantizer"], loss=torch.nn.Identity())
    model = build()
    assert isinstance(model.encoder, etb.ViTEncoder) and isinstance(model.quantizer, etb.VectorQuantizer)
    assert {k: tuple(v.shape) for k, v in model.state_dict().items()} == want
    keys = set(model.state_dict())
    # patch() on an already-imported module rebinds the same three names
    mod.Encoder = None
    etb.patch(mod)
    assert mod.Encoder is etb.ViTEncoder
    # ... and makes every ViTVQ built afterwards carry QuantLinear pre/post_quant that share the nn.Linear parameters
    # and state-dict keys; patching twice does not wrap twice
    etb.patch(mod)
    assert mod.ViTVQ.__init__.__wrapped__.__name__ == "__init__" and not hasattr(mod.ViTVQ.__init__.__wrapped__, "__wrapped__")
    model2 = build()
    assert isinstance(model2.pre_quant, etb.QuantLinear) and isinstance(model2.post_quant, etb.QuantLinear)
    assert set(model2.state_dict()) == keys
    model2.load_state_dict(model.state_dict(), strict=True)
    plain = torch.nn.Linear(64, 32)
    fused = etb.QuantLinear.from_linear(plain)
    assert fused.weight is plain.weight and fused.bias is plain.bias and isinstance(fused, torch.nn.Linear)
    # opt-in: the discriminator step's forward (optimizer_idx == 1) runs without an autograd graph
    seen = []

    class Probe(torch.nn.Module):                                # stands in for VQLPIPSWithDiscriminator
        def forward(self, qloss, x, xrec, optimizer_idx, *a, **k):
            seen.append((optimizer_idx, xrec.requires_grad, torch.is_grad_enabled()))
            key = "train/total_loss" if optimizer_idx == 0 else "train/disc_loss"
            return xrec.sum() * 0 + 1.0, {key: torch.tensor(1.0)}

    class Tiny(mod.ViTVQ):                                       # no GPU here: swap the heavy parts for CPU stand-ins
        def __init__(self):
            torch.nn.Module.__init__(self)
            self.image_key, self.loss = "image", Probe()
            self.lin = torch.nn.Linear(4, 4)
            self.decoder = types.SimpleNamespace(get_last_layer=lambda: self.lin.weight)
            self.global_step = 0
        encode = lambda self, x: (self.lin(x), x.sum() * 0)
        decode = lambda self, q: q

    etb.detach_discriminator_forward(Tiny)
    etb.detach_discriminator_forward(Tiny)                       # idempotent
    m = Tiny()
    batch = {"image": torch.randn(2, 4, 4, 4)}
    m.training_step(batch, 0, 0)
    m.training_step(batch, 0, 1)
    m.training_step(batch, 0, 0)
    assert seen == [(0, True, True), (1, False, True), (0, True, True)], seen
    assert mod.ViTVQ.forward is not Tiny.forward                  # only the class it was asked to wrap


def test_fuse_post_quant_pos_keeps_the_checkpoint_abi():
    """SURVEY.md section 8f-1 (opt-in): post_quant borrows the decoder's positional table without registering it a second
    time -- same state-dict keys, same Parameter objects, reversible"""
    import torch

    class Holder(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.decoder = etb.ViTDecoder(32, 8, dim=64, depth=1, heads=2, mlp_dim=128, dim_head=32)
            self.post_quant = torch.nn.Linear(32, 64)

    m = Holder()
    keys, params = set(m.state_dict()), {id(p) for p in m.parameters()}
    w = m.post_quant.weight
    etb.fuse_post_quant_pos(m)
    assert isinstance(m.post_quant, etb.PosQuantLinear) and m.post_quant.weight is w and m.decoder.pos_added_upstream
    assert set(m.state_dict()) == keys and {id(p) for p in m.parameters()} == params
    m.load_state_dict(m.state_dict(), strict=True)
    etb.fuse_post_quant_pos(m, False)
    assert type(m.post_quant) is etb.QuantLinear and m.post_quant.weight is w and not m.decoder.pos_added_upstream
    with pytest.raises(TypeError):
        etb.fuse_post_quant_pos(torch.nn.Linear(2, 2))


def test_unchanged_cond_transformer_constructs_with_patch_stage2(golden_dir):
    """after `etb.patch_stage2` a YAML-style `transformer.target: enhancing.modules.stage2.layers.GPT` resolves by attribute
    lookup (the reference's get_obj_from_str, utils/general.py:29-41) to this package's GPT, whose parameters carry the
    names and owning module kinds (Linear / LayerNorm / Embedding / other) of the reference's own GPT
    (tests/golden/ref_modules.npz, oracle/gen_golden_live.py): what the reference's CondTransformer.configure_optimizers
    (stage2/transformer.py:131-166) sorts into decay / no-decay sets"""
    import types

    from oracle.gen_golden_live import GPT_ABI_CFG
    layers = types.ModuleType("stage2_layers_stand_in")
    layers.GPT = object
    etb.patch_stage2(layers)
    assert layers.GPT is etb.GPT
    gpt = getattr(layers, "GPT")(**GPT_ABI_CFG)
    assert isinstance(gpt, etb.GPT)
    kinds = (torch.nn.Linear, torch.nn.LayerNorm, torch.nn.Embedding)
    owners = []
    for mn, m in gpt.named_modules():
        for pn, _ in m.named_parameters(recurse=False):
            kind = next((k.__name__ for k in kinds if isinstance(m, k)), "other")
            owners.append(f"{mn + '.' if mn else ''}{pn}:{kind}")
    want = np.load(os.path.join(golden_dir, "ref_modules.npz"))["gptabi.owners"].tolist()
    assert sorted(owners) == want, set(owners) ^ set(want)


def test_c_abi_rejects_bad_arguments_before_touching_the_device():
    """error convention of the C ABI (include/b200vq.h): a negative return code and a message from b200vq_last_error();
    argument validation happens before any CUDA call, so it can be exercised on a machine without a GPU"""
    lib = etb._lib.lib()

    def err():
        return lib.b200vq_last_error().decode()
    # stage-2 attention: head size, prefix length
    assert lib.b200vq_attention_causal_fwd(None, None, None, 1, 16, 2, 48, 0.1, 1, 1, 0, None) < 0 and "32 or 64" in err()
    assert lib.b200vq_attention_causal_fwd(None, None, None, 1, 16, 2, 64, 0.1, 17, 1, 0, None) < 0 and "cond_len" in err()
    assert lib.b200vq_attention_causal_bwd(None, None, None, None, None, None, 0, 16, 2, 64, 0.1, 1, 0, 0, None) < 0 and "empty" in err()
    # stream kernels of stage 2
    assert lib.b200vq_time_mix_fwd(None, None, None, 10, 3, 64, 0, None) < 0 and "M % T" in err()
    assert lib.b200vq_time_mix_fwd(None, None, None, 12, 3, 62, 0, None) < 0
    assert lib.b200vq_sqrelu(None, None, None, 6, 0, 0, None) < 0
    assert lib.b200vq_sqrelu(None, None, None, 8, 1, 0, None) < 0 and "gradient" in err()
    assert lib.b200vq_copy_rows(None, None, 2, 9, 5, 6, 0, 5, 64, None) < 0 and "window" in err()
    assert lib.b200vq_decode_attention(None, None, None, None, 2, 2, 64, 10, 10, 0.1, None) < 0 and "position" in err()
    assert lib.b200vq_decode_attention(None, None, None, None, 2, 2, 48, 10, 3, 0.1, None) < 0
    assert lib.b200vq_token_embed_fwd(None, None, None, None, None, None, None, 2, 0, 0, 64, 5, 5, None) < 0
    # stage 1: quantiser width, LayerNorm row length, attention head size
    assert lib.b200vq_vq_fwd(None, None, None, None, None, 128, 256, 16, 1, 0.25, 1, None, 0, None) < 0
    assert lib.b200vq_layernorm_fwd(None, None, None, None, None, None, None, 8, 4096, 0, None) < 0 and "2048" in err()
    assert lib.b200vq_attention_f16_fwd(None, None, None, 1, 16, 2, 32, 0.1, None) < 0 and "64" in err()
    assert lib.b200vq_time_mix_bwd_workspace_bytes(130, 64) == 3 * 64 * 4           # ceil(130 / 64) partial rows
