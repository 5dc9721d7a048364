"""Generate golden fixtures by running the REAL reference (imported from /root/reference).

Run in the authoring container only (the GPU box has no /root/reference):
    python oracle/make_golden.py
Writes small ``.pt`` fixtures to tests/golden/. The oracle (oracle/vqgan_oracle.py) and the CUDA
product are both checked against these files. TEST INFRASTRUCTURE — never imported by the product.
"""
import os
import sys
import types

import torch

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")


def load_reference():
    """SURVEY.md 8c recipe: stub the absent fast_pytorch_kmeans, import reference `models` privately."""
    stub = types.ModuleType("fast_pytorch_kmeans")
    stub.KMeans = object
    sys.modules["fast_pytorch_kmeans"] = stub
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "models" or k.startswith("models.")}
    sys.path.insert(0, REF)
    try:
        import models as ref_models  # noqa
        import models.modules as ref_modules  # noqa
        import models.vqvae as ref_vqvae  # noqa
        import losses.loss_seg as ref_loss_seg  # noqa
        import models.transformer as ref_transformer  # noqa
    finally:
        sys.path.remove(REF)
    out = (ref_models, ref_modules, ref_vqvae, ref_loss_seg, ref_transformer)
    for k in list(sys.modules):
        if k == "models" or k.startswith("models.") or k == "losses" or k.startswith("losses."):
            sys.modules["_ref_" + k] = sys.modules.pop(k)
    sys.modules.update(saved)
    return out


TINY = dict(z_channels=32, in_channels=3, out_channels=3, channels=[32, 32, 64], num_res_blocks=1,
            resolution=16, attn_resolutions=[8], dropout=0.0)
IMG = dict(z_channels=256, in_channels=3, out_channels=3, channels=[128, 128, 128, 256, 512, 512],
           num_res_blocks=2, resolution=512, attn_resolutions=[32], dropout=0.0)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    ref_models, M, V, L, T = load_reference()
    only = None
    for a in sys.argv[1:]:
        if a.startswith("--only="):
            only = set(a[len("--only="):].split(","))
    if only is None or "base" in only:
        base_fixtures(ref_models, M, V, L, T)
    if only is None or "tc" in only:
        tensor_path_block_fixtures(M)
    if only is None or "img256" in only:
        img256_fixture(ref_models)
    if only is None or "codebook" in only:
        codebook_schedule_fixture(M)


def base_fixtures(ref_models, M, V, L, T):

    # ---- G1: tiny VQBASE fwd+bwd, VQ active, train mode --------------------------------------
    torch.manual_seed(0)
    m = ref_models.VQBASE(TINY, 64, 32, 10, 100)
    with torch.no_grad():
        m.quantize.embedding.weight.normal_()
        # make the affine params non-trivial so that gamma/beta paths are exercised
        for n, p in m.named_parameters():
            if "norm" in n or n.startswith("quant_conv.1"):
                p.add_(0.1 * torch.randn_like(p))
    m.quantize.q_counter = 10 ** 6
    m.train()
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(2, 3, 16, 16, generator=g)
    taps = {}
    hooks = []
    for name, mod in list(m.encoder.model.named_children()):
        hooks.append(mod.register_forward_hook(lambda _m, _i, o, n=name: taps.__setitem__("encoder.model." + n, o.detach().clone())))
    for name, mod in list(m.decoder.model.named_children()):
        hooks.append(mod.register_forward_hook(lambda _m, _i, o, n=name: taps.__setitem__("decoder.model." + n, o.detach().clone())))
    hooks.append(m.quant_conv.register_forward_hook(lambda _m, _i, o: taps.__setitem__("quant_conv", o.detach().clone())))
    idx_holder = {}
    hooks.append(m.quantize.register_forward_hook(lambda _m, _i, o: idx_holder.__setitem__("idx", o[2].clone())))
    dec, diff = m(x)
    loss = (x - dec).abs().mean() + diff
    loss.backward()
    for h in hooks:
        h.remove()
    grads = {k: p.grad.clone() for k, p in m.named_parameters()}
    torch.save(dict(ddconfig=TINY, n_embed=64, embed_dim=32, state_dict=sd0, x=x, dec=dec.detach(), diff=diff.detach(),
                    idx=idx_holder["idx"], loss=loss.detach(), grads=grads, taps=taps,
                    running_mean=m.quant_conv[1].running_mean.clone(), running_var=m.quant_conv[1].running_var.clone()),
               os.path.join(OUT, "vqbase_tiny.pt"))
    print("vqbase_tiny: params", sum(p.numel() for p in m.parameters()), "loss", float(loss))

    # ---- G1b: warm-up bypass (q_counter < q_init) and eval mode -------------------------------
    m2 = ref_models.VQBASE(TINY, 64, 32, 10, 100)
    m2.load_state_dict(sd0)
    m2.train()
    dec_b, diff_b = m2(x)
    m2.load_state_dict(sd0)   # undo the running-stat update of the train-mode forward
    m2.eval()
    dec_e, diff_e = m2(x)
    torch.save(dict(dec_bypass=dec_b.detach(), diff_bypass=diff_b.detach(), dec_eval=dec_e.detach(), diff_eval=diff_e.detach()),
               os.path.join(OUT, "vqbase_tiny_modes.pt"))

    # ---- G2: codebook standalone sets (SURVEY.md 8d correctness sets) --------------------------
    sets = {}
    g = torch.Generator().manual_seed(7)
    for name in ("trained", "fresh", "clustered", "duplicated"):
        cb = M.Codebook(256, 64, beta=0.25, init_steps=10, reservoir_size=100)
        cb.eval()
        with torch.no_grad():
            if name == "trained":
                cb.embedding.weight.copy_(torch.randn(256, 64, generator=g))
                z = torch.randn(3, 64, 4, 4, generator=g)
            elif name == "fresh":
                cb.embedding.weight.copy_((torch.rand(256, 64, generator=g) * 2 - 1) / 256)
                z = torch.randn(3, 64, 4, 4, generator=g)
            elif name == "clustered":
                cb.embedding.weight.copy_(torch.randn(256, 64, generator=g))
                j = torch.randint(0, 256, (48,), generator=g)
                z = (cb.embedding.weight[j] + 0.3 * torch.randn(48, 64, generator=g)).view(3, 4, 4, 64).permute(0, 3, 1, 2).contiguous()
            else:
                e = torch.randn(128, 64, generator=g)
                cb.embedding.weight.copy_(torch.cat([e, e], 0))
                z = torch.randn(3, 64, 4, 4, generator=g)
        z = z.clone().requires_grad_(True)
        z_q, loss, idx = cb(z)
        (z_q * torch.linspace(-1, 1, z_q.numel()).view_as(z_q)).sum().add(loss).backward()
        sets[name] = dict(E=cb.embedding.weight.detach().clone(), z=z.detach().clone(), z_q=z_q.detach().clone(),
                          loss=loss.detach().clone(), idx=idx.clone(), grad_z=z.grad.clone(),
                          grad_E=cb.embedding.weight.grad.clone())
        ent = cb.get_codebook_entry(idx, (3, 4, 4, 64))
        sets[name]["entry"] = ent.detach().clone()
    torch.save(sets, os.path.join(OUT, "codebook_sets.pt"))
    print("codebook sets done")

    # ---- G3: individual blocks at real channel widths, small spatial ---------------------------
    blocks = {}
    torch.manual_seed(1)
    g = torch.Generator().manual_seed(11)

    def run_block(mod, x):
        x = x.clone().requires_grad_(True)
        with torch.no_grad():
            for n, p in mod.named_parameters():
                if "norm" in n:
                    p.add_(0.1 * torch.randn_like(p))
        y = mod(x)
        w = torch.linspace(-1, 1, y.numel()).view_as(y)
        (y * w).sum().backward()
        return dict(state_dict={k: v.clone() for k, v in mod.state_dict().items()}, x=x.detach().clone(),
                    y=y.detach().clone(), grad_x=x.grad.clone(),
                    grads={k: p.grad.clone() for k, p in mod.named_parameters()})

    blocks["res_64_64"] = run_block(M.ResnetBlock(in_channels=64, out_channels=64, dropout=0.0), torch.randn(2, 64, 8, 8, generator=g))
    blocks["res_64_128"] = run_block(M.ResnetBlock(in_channels=64, out_channels=128, dropout=0.0), torch.randn(2, 64, 8, 8, generator=g))
    blocks["attn_64"] = run_block(M.AttnBlock(64), torch.randn(2, 64, 4, 4, generator=g))
    blocks["down_32"] = run_block(M.Downsample(32, True), torch.randn(2, 32, 8, 8, generator=g))
    blocks["up_32"] = run_block(M.Upsample(32, True), torch.randn(2, 32, 4, 4, generator=g))
    torch.save(blocks, os.path.join(OUT, "blocks.pt"))
    print("blocks done")

    # ---- G4: img_config model (95 M params, seeded init), small spatial: outputs only ----------
    torch.manual_seed(0)
    big = ref_models.VQBASE(IMG, 8192, 256, 3000, 12500)
    with torch.no_grad():
        big.quantize.embedding.weight.normal_()
    big.quantize.q_counter = 10 ** 6
    big.train()
    checks = {k: (float(v.double().sum()), float(v.double().abs().sum())) for k, v in big.state_dict().items()}
    g = torch.Generator().manual_seed(1234)
    x = torch.rand(2, 3, 64, 64, generator=g)
    qc = {}
    h1 = big.quant_conv.register_forward_hook(lambda _m, _i, o: qc.__setitem__("h", o.detach().clone()))
    h2 = big.quantize.register_forward_hook(lambda _m, _i, o: qc.__setitem__("idx", o[2].clone()))
    dec, diff = big(x)
    loss = (x - dec).abs().mean() + diff
    loss.backward()
    h1.remove(); h2.remove()
    sel = ["encoder.model.0.weight", "encoder.model.1.conv1.weight", "encoder.model.14.q.weight", "decoder.model.28.weight",
           "decoder.model.28.bias", "quantize.embedding.weight", "quant_conv.0.weight", "quant_conv.1.weight",
           "decoder.model.25.norm2.weight", "decoder.model.15.nin_shortcut.weight", "encoder.model.3.conv.weight",
           "decoder.model.22.conv.weight"]
    named = dict(big.named_parameters())
    torch.save(dict(ddconfig=IMG, x=x, dec=dec.detach(), diff=diff.detach(), idx=qc["idx"], quant_in=qc["h"], loss=loss.detach(),
                    param_checks=checks, n_params=sum(p.numel() for p in big.parameters()),
                    grad_norms={k: float(named[k].grad.double().norm()) for k in named},
                    grads_small={k: named[k].grad.clone() for k in sel if named[k].grad.numel() <= 40000}),
               os.path.join(OUT, "vqbase_img_64.pt"))
    print("img 64 done: loss", float(loss), "n_params", sum(p.numel() for p in big.parameters()))

    # ---- G6: tier-2 token transformer (tiny; CPU, non-cached forward + cross-entropy backward) -------------------
    for tag, cfg in (("tiny", dict(num_layers=2, hidden_dim=64, num_attn_heads=4, image_vocab_size=96, seg_vocab_size=48,
                                   text_vocab_size=80 + 12, image_tokens_per_dim=4, seg_tokens_per_dim=3, text_length=12)),
                     ("wide", dict(num_layers=1, hidden_dim=256, num_attn_heads=4, image_vocab_size=128, seg_vocab_size=32,
                                   text_vocab_size=64 + 8, image_tokens_per_dim=4, seg_tokens_per_dim=2, text_length=8))):
        torch.manual_seed(3)
        tm = T.MakeAScene(**cfg)
        tm.device = torch.device("cpu")
        g = torch.Generator().manual_seed(17)
        tt = torch.randint(0, cfg["text_vocab_size"] - cfg["text_length"], (2, cfg["text_length"]), generator=g)
        tt[0, -3:] = 0                                    # padded text positions exercise the pad-id trick (transformer.py:350-353)
        st = torch.randint(0, cfg["seg_vocab_size"], (2, cfg["seg_tokens_per_dim"] ** 2), generator=g)
        it = torch.randint(0, cfg["image_vocab_size"], (2, cfg["image_tokens_per_dim"] ** 2), generator=g)
        logits = tm(tt, st, it)
        loss = torch.nn.functional.cross_entropy(logits.reshape(-1, logits.shape[-1]), it.reshape(-1))
        loss.backward()
        torch.save(dict(cfg=cfg, state_dict={k: v.clone() for k, v in tm.state_dict().items()}, text=tt, seg=st, img=it,
                        logits=logits.detach(), loss=loss.detach(),
                        grads={k: p.grad.clone() for k, p in tm.named_parameters() if p.grad is not None and (tag == "tiny" or p.numel() <= 70000)},
                        grad_norms={k: float(p.grad.double().norm()) for k, p in tm.named_parameters() if p.grad is not None}),
                   os.path.join(OUT, f"transformer_{tag}.pt"))
        print("transformer", tag, "loss", float(loss), "params", sum(p.numel() for p in tm.parameters()))

    # ---- G5: seg loss ---------------------------------------------------------------------------
    g = torch.Generator().manual_seed(5)
    lf = L.BCELossWithQuant(image_channels=159)
    pred = torch.randn(2, 159, 8, 8, generator=g, requires_grad=True)
    tgt = (torch.rand(2, 159, 8, 8, generator=g) > 0.9).float()
    q = torch.tensor(0.37)
    lv = lf(q, tgt, pred)
    lv.backward()
    torch.save(dict(pred=pred.detach().clone(), target=tgt, qloss=q, loss=lv.detach(), grad=pred.grad.clone()),
               os.path.join(OUT, "seg_loss.pt"))
    print("seg loss done")


def tensor_path_block_fixtures(M):
    """G7: blocks at widths / extents that the tcgen05 kernels take (Cout % 128 == 0, H % 16 == 0, W % 8 == 0), run on the
    REAL reference modules. Weights and inputs are regenerated from seeds on both sides (oracle/seeded.py)."""
    import torch.nn as nn
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from seeded import fill_seeded, seeded_input, sample
    specs = {
        "res_128_128": (lambda: M.ResnetBlock(in_channels=128, out_channels=128, dropout=0.0), (2, 128, 32, 32)),
        "res_128_256": (lambda: M.ResnetBlock(in_channels=128, out_channels=256, dropout=0.0), (2, 128, 32, 32)),
        "res_512_512": (lambda: M.ResnetBlock(in_channels=512, out_channels=512, dropout=0.0), (2, 512, 16, 16)),
        "attn_512": (lambda: M.AttnBlock(512), (2, 512, 16, 16)),
        # the AttnBlock's projection epilogue emits the statistics the following ResnetBlock's first GroupNorm consumes
        "attn_res_512": (lambda: nn.Sequential(M.AttnBlock(512), M.ResnetBlock(in_channels=512, out_channels=512, dropout=0.0)),
                         (2, 512, 16, 16)),
        # ... and a ResnetBlock's conv2 epilogue emits those of the next block (res -> res -> attn chain of the decoder)
        "res_res_attn_512": (lambda: nn.Sequential(M.ResnetBlock(in_channels=512, out_channels=512, dropout=0.0),
                                                   M.ResnetBlock(in_channels=512, out_channels=512, dropout=0.0), M.AttnBlock(512)),
                             (2, 512, 16, 16)),
        "up_128": (lambda: M.Upsample(128, True), (2, 128, 16, 16)),
        "down_128": (lambda: M.Downsample(128, True), (2, 128, 32, 32)),
        "up_512": (lambda: M.Upsample(512, True), (1, 512, 16, 16)),
    }
    out = {}
    for i, (name, (ctor, shape)) in enumerate(specs.items()):
        mod = ctor()
        checks = fill_seeded(mod, 100 + i)
        x = seeded_input(shape, 200 + i, 1.5, 0.3).requires_grad_(True)
        y = mod(x)
        w = torch.linspace(-1, 1, y.numel()).view_as(y)
        (y * w).sum().backward()
        grads, norms = {}, {}
        for k, p in mod.named_parameters():
            norms[k] = float(p.grad.double().norm())
            grads[k] = p.grad.clone() if p.grad.numel() <= 70000 else sample(p.grad, 8192)
        out[name] = dict(seed_w=100 + i, seed_x=200 + i, shape=shape, param_checks=checks, y=sample(y, y.numel() // 3),
                         y_norm=float(y.double().norm()), grad_x=sample(x.grad, x.numel() // 3),
                         grad_x_norm=float(x.grad.double().norm()), grads=grads, grad_norms=norms)
        print("tc block", name, "y norm", float(y.norm()))
    torch.save(out, os.path.join(OUT, "blocks_tc.pt"))


def img256_fixture(ref_models):
    """G8: the img_config model at BASELINE's 256x256 (batch 2), fwd + bwd on the REAL reference."""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from seeded import sample
    torch.manual_seed(0)
    big = ref_models.VQBASE(IMG, 8192, 256, 3000, 12500)
    with torch.no_grad():
        big.quantize.embedding.weight.normal_()
    big.quantize.q_counter = 10 ** 6
    big.train()
    x = torch.rand(2, 3, 256, 256, generator=torch.Generator().manual_seed(1234))
    qc = {}
    h1 = big.quant_conv.register_forward_hook(lambda _m, _i, o: qc.__setitem__("h", o))
    def _h2(_m, _i, o):
        o[0].retain_grad()
        qc["idx"], qc["zq"] = o[2].clone(), o[0]
    h2 = big.quantize.register_forward_hook(_h2)
    def _h1(_m, _i, o):
        o.retain_grad()
        qc["h"] = o
    h1.remove()
    h1 = big.quant_conv.register_forward_hook(_h1)
    dec, diff = big(x)
    loss = (x - dec).abs().mean() + diff
    loss.backward()
    h1.remove(); h2.remove()
    named = dict(big.named_parameters())
    grad_samples = {k: sample(p.grad, 512) for k, p in named.items()}
    torch.save(dict(ddconfig=IMG, x_seed=1234, x_shape=(2, 3, 256, 256), x_sum=float(x.double().sum()),
                    idx=qc["idx"], quant_in=qc["h"].detach().clone(), dec_norm=float(dec.double().norm()),
                    dec_sample=sample(dec, 16384), diff=diff.detach(), loss=loss.detach(),
                    g_quant_in=sample(qc["h"].grad, 16384), g_quant_in_norm=float(qc["h"].grad.double().norm()),
                    g_zq=sample(qc["zq"].grad, 16384), g_zq_norm=float(qc["zq"].grad.double().norm()),
                    grad_norms={k: float(p.grad.double().norm()) for k, p in named.items()}, grad_samples=grad_samples),
               os.path.join(OUT, "vqbase_img_256.pt"))
    print("img 256 done: loss", float(loss))


def codebook_schedule_fixture(M):
    """G9: the REAL reference's Codebook through its warm-up steps 1 .. q_init - 1 (init_steps 4: collects from step 5,
    quantises from step 12): per step the output, loss, indices, counter and reservoir, under the same global seeds as
    tests/test_host_logic_vq_cpu.py replays them (reservoir sampling draws two torch.randperm per step)."""
    K, D, init_steps = 16, 8, 4
    torch.manual_seed(3)
    cb = M.Codebook(K, D, 0.25, init_steps, 60)
    cb.train()
    gz = torch.Generator().manual_seed(11)
    zs = [torch.randn(3, D, 4, 4, generator=gz) for _ in range(16)]
    steps = []
    for step, z in enumerate(zs[:11], start=1):
        torch.manual_seed(100 + step)
        z_q, loss, idx = cb(z)
        steps.append(dict(z_q=z_q.detach().clone(), loss=float(loss), idx=idx, q_counter=cb.q_counter,
                          reservoir=None if cb.reservoir is None else cb.reservoir.clone()))
    torch.save(dict(K=K, D=D, init_steps=init_steps, reservoir_size=60, weight=cb.embedding.weight.detach().clone(), steps=steps),
               os.path.join(OUT, "codebook_schedule.pt"))
    print("codebook schedule done")


if __name__ == "__main__":
    main()
