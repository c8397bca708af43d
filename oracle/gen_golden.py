"""Generate tests/golden/*.npz by running the UNMODIFIED reference on CPU (build container only).

    python oracle/gen_golden.py            # needs /root/reference; writes tests/golden/

Each fixture stores the reference's own state_dict (small configs), the inputs and the reference's
outputs, so the oracle (tests/test_oracle_golden.py, CPU) and the CUDA path (tests/test_gpu_*.py)
can both be checked against numbers the reference itself produced.  Inputs that are large are
regenerated from ``portable_uniform`` (numpy Philox: platform independent, exact arithmetic only).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def portable_uniform(seed: int, shape) -> torch.Tensor:
    """U[0,1) fp32 from numpy Philox -- bit-identical on every platform."""
    rng = np.random.Generator(np.random.Philox(seed))
    return torch.from_numpy(rng.random(size=tuple(shape), dtype=np.float32))


def sampler_case_inputs(case: int, B=2, K=256, L=265):
    """(logits (B,K,L), x_t (B,L), t (B,), u (B,K+1,L)) for the posterior/sampler golden cases."""
    scale = [1.0, 6.0, 40.0, 2.0, 12.0][case % 5]
    logits = (portable_uniform(100 + case, (B, K, L)) - 0.5) * scale
    u = portable_uniform(200 + case, (B, K + 1, L))
    t_pair = [(99, 99), (57, 12), (1, 1), (0, 0), (98, 33)][case % 5]
    t = torch.tensor([t_pair[i % 2] for i in range(B)], dtype=torch.long)
    ids = (portable_uniform(300 + case, (B, L)) * K).long().clamp(max=K - 1)
    masked = portable_uniform(400 + case, (B, L)) < ([1.1, 0.35, 0.05, 0.02, 0.9][case % 5])
    x_t = torch.where(masked, torch.full_like(ids, K), ids)
    return logits, x_t, t, u


def sd_np(sd, drop=("attn2.mask",)):
    return {k: v.numpy() for k, v in sd.items() if not any(d in k for d in drop)}


def gen_xf_tiny():
    K, D, NL, NH, CD = 32, 128, 2, 2, 64
    model, _ = rh.build_dalle(K=K, overrides=dict(n_layer=NL, n_embd=D, n_head=NH, condition_dim=CD, dec_ch=32,
                                                  dec_ch_mult=[1, 1, 1, 1, 2], dec_z_channels=64, embed_dim=64), seed=0)
    tr = model.transformer  # DiffusionTransformer
    g = torch.Generator().manual_seed(7)
    # the reference zero-inits biases and unit-inits LayerNorm; perturb so that bias/affine paths are pinned too
    for n, p in tr.named_parameters():
        if n.endswith("bias") or "ln2.weight" in n or "to_logits.0.weight" in n:
            p.add_(torch.randn(p.shape, generator=g) * 0.05)
    B, L = 3, 265
    cond = torch.randn(B, 77, CD, generator=g)
    cond = cond / cond.norm(dim=-1, keepdim=True)
    x_t = torch.randint(0, K + 1, (B, L), generator=g)
    t = torch.tensor([99, 41, 0])
    logits = tr.transformer(x_t.clone(), cond, t)
    log_x = torch.log(torch.nn.functional.one_hot(x_t, K + 1).permute(0, 2, 1).float().clamp(min=1e-30))
    wrapped = model.predict_start_with_truncation(tr.predict_start, "top0.85r")
    lp = wrapped(log_x, cond, t)
    post = tr.q_posterior(lp, log_x, t)
    # free-running reference sample(): global CPU generator, exactly as generate_content would
    model.truncation_forward = True
    tr.predict_start = wrapped
    out = dict(sd_np(tr.state_dict()))
    torch.manual_seed(1234)
    tok = tr.sample(condition_token=None, condition_mask=None, condition_embed=cond, filter_ratio=0, batch_size=B)["content_token"]
    # N1 variants through the reference's own entry points (same truncating predict_start): skip-step sampler and content-conditioned start
    torch.manual_seed(1235)
    tok_fast = tr.sample_fast(condition_token=torch.zeros(B, 1), condition_mask=None, condition_embed=cond, filter_ratio=0, skip_step=3)["content_token"]
    x0 = torch.randint(0, K, (B, L), generator=g)
    torch.manual_seed(1236)
    tok_cond = tr.sample(condition_token=None, condition_mask=None, condition_embed=cond, content_token=x0, filter_ratio=0.3, batch_size=B)["content_token"]
    extra = dict(out_fast3_tokens=tok_fast.numpy().astype(np.int16), in_content=x0.numpy().astype(np.int16), out_cond_tokens=tok_cond.numpy().astype(np.int16))
    np.savez_compressed(os.path.join(GOLD, "xf_tiny.npz"), __cfg=np.array([K, D, NL, NH, CD, B, L]), **extra,
                        in_cond=cond.numpy(), in_x_t=x_t.numpy().astype(np.int16), in_t=t.numpy(),
                        out_logits=logits.numpy(), out_lp=lp.numpy(), out_post=post.numpy(),
                        out_sample_tokens=tok.numpy().astype(np.int16), **{"sd." + k: v for k, v in out.items()})
    print("xf_tiny: logits", tuple(logits.shape), "tokens", tok[0, :8].tolist())
    return model


def gen_train_tiny(model):
    """A13: DiffusionTransformer.forward(return_loss=True) of the reference on the xf_tiny weights, with sample_time pinned
    (harness-side rebinding of the instance attribute; no reference file is edited) and the q_sample uniforms reproduced by seeding
    the global CPU generator.  Stores loss, log_model_prob, x_t and the autograd gradient of every parameter."""
    tr = model.transformer
    K, D, NL, NH, CD, B, L = np.load(os.path.join(GOLD, "xf_tiny.npz"))["__cfg"].tolist()
    g = torch.Generator().manual_seed(11)
    cond = torch.randn(B, 77, CD, generator=g)
    cond = cond / cond.norm(dim=-1, keepdim=True)
    x0 = torch.randint(0, K, (B, L), generator=g)
    t = torch.tensor([57, 0, 99])
    pt = torch.tensor([0.013, 0.004, 0.01])
    tr.__dict__.pop("predict_start", None)  # gen_xf_tiny rebound it to the truncating wrapper; training uses the plain method
    tr.sample_time = lambda b, device, method="uniform": (t, pt)
    tr.Lt_history.zero_(); tr.Lt_count.zero_()
    for p_ in tr.parameters():
        p_.requires_grad_(True)
        p_.grad = None
    seed = 4321
    torch.manual_seed(seed)
    u = torch.rand(B, K + 1, L)
    torch.manual_seed(seed)
    with torch.enable_grad():
        out = tr({"content_token": x0, "condition_embed_token": cond}, return_loss=True)
        out["loss"].backward()
    grads = {"grad." + n: p_.grad.numpy() for n, p_ in tr.named_parameters() if p_.grad is not None}
    missing = [n for n, p_ in tr.named_parameters() if p_.grad is None]
    np.savez_compressed(os.path.join(GOLD, "train_tiny.npz"), in_cond=cond.numpy(), in_x0=x0.numpy().astype(np.int16), in_t=t.numpy(),
                        in_pt=pt.numpy(), in_uniform=u.numpy(), out_loss=out["loss"].detach().numpy(), out_probs=out["logits"].detach().numpy(),
                        out_Lt_history=tr.Lt_history.numpy(), out_Lt_count=tr.Lt_count.numpy(),
                        cfg_aux=np.array([tr.auxiliary_loss_weight, float(tr.adaptive_auxiliary_loss), *tr.mask_weight]), **grads)
    print("train_tiny: loss", float(out["loss"]), "params with grad", len(grads), "without", missing)


def gen_sampler_cases():
    """K=256 posterior + nucleus + Gumbel sampler through the reference's own methods."""
    model, _ = rh.build_dalle(K=256, overrides=dict(n_layer=1, n_embd=64, n_head=1, dec_ch=32, dec_ch_mult=[1, 1, 1, 1, 2]), seed=0)
    tr = model.transformer
    K, L = 256, 265
    res = {}
    for case in range(5):
        logits, x_t, t, u = sampler_case_inputs(case)
        # feed the case logits through the reference's predict_start tail by stubbing the denoiser
        tr.transformer.forward = lambda *_a, _l=logits, **_k: _l
        model.this_save_path = None  # read (unused) by the 'p' branch of predict_start_with_truncation
        for trunc in ("top0.85r", None, "top20p"):
            ps = type(tr).predict_start.__get__(tr)
            if trunc:
                ps = model.predict_start_with_truncation(ps, trunc)
            if case == 0:  # the all-[MASK] start state with its -inf carrier (diffusion_transformer.py:633-636)
                log_x = torch.log(torch.nn.functional.one_hot(x_t, K + 1).permute(0, 2, 1).float())
            else:
                log_x = torch.log(torch.nn.functional.one_hot(x_t, K + 1).permute(0, 2, 1).float().clamp(min=1e-30))
            lp = ps(log_x, None, t)
            post = tr.q_posterior(lp, log_x, t)
            g = -torch.log(-torch.log(u + 1e-30) + 1e-30)
            nxt = (g + post).argmax(1)
            tag = f"c{case}_{ {'top0.85r': 'nuc', None: 'raw', 'top20p': 'topk'}[trunc] }"
            res[tag + "_next"] = nxt.numpy().astype(np.int16)
            res[tag + "_post_head"] = post[:, :, :6].numpy()
            res[tag + "_lp_head"] = lp[:, :, :6].numpy()
            top2 = (g + post).topk(2, dim=1).values
            res[tag + "_margin"] = (top2[:, 0] - top2[:, 1]).numpy()
    np.savez_compressed(os.path.join(GOLD, "sampler_cases.npz"), **res)
    print("sampler_cases:", len(res), "arrays")


def gen_decoder_tiny():
    K = 32
    model, _ = rh.build_dalle(K=K, overrides=dict(n_layer=1, n_embd=64, n_head=1, dec_ch=32, dec_ch_mult=[1, 1, 1, 1, 2],
                                                  dec_z_channels=64, embed_dim=64, grid=(2, 7)), seed=3)
    g = torch.Generator().manual_seed(11)
    cc = model.content_codec
    cc.quantize.embedding.weight.mul_(K * 0.5)  # U(-1/K,1/K) init is tiny; scale to O(1) like a trained codebook
    B, H, W = 2, 2, 7
    ids = torch.randint(0, K, (B, H * W), generator=g)
    mel = model.decode_to_img(ids, (B, 64, H, W))
    sd = {k: v for k, v in model.state_dict().items()
          if k.startswith("content_codec.") and ".encoder." not in k and "quant_conv" not in k.replace("post_quant_conv", "") and ".loss." not in k}
    np.savez_compressed(os.path.join(GOLD, "decoder_tiny.npz"), in_ids=ids.numpy().astype(np.int16), out_mel=mel.numpy(),
                        __cfg=np.array([K, 64, 32, H, W]), **{"sd." + k: v.numpy() for k, v in sd.items()})
    print("decoder_tiny: mel", tuple(mel.shape), float(mel.abs().max()))


def gen_encoder_tiny():
    """N4: the reference tokeniser DALLE.get_tokens (SpecVQGAN Encoder + quant_conv + nearest code + ColumnMajor) on a tiny config."""
    K = 32
    model, _ = rh.build_dalle(K=K, overrides=dict(n_layer=1, n_embd=64, n_head=1, dec_ch=32, dec_ch_mult=[1, 1, 1, 1, 2],
                                                  dec_z_channels=64, embed_dim=64, grid=(2, 7)), seed=3)
    g = torch.Generator().manual_seed(21)
    cc = model.content_codec
    for n_, p_ in cc.encoder.named_parameters():
        if n_.endswith("bias"):
            p_.add_(torch.randn(p_.shape, generator=g) * 0.05)
    mel = torch.rand(2, 1, 32, 112, generator=g) * 2 - 1
    z0 = cc.quant_conv(cc.encoder(mel))
    # a random-init codebook is U(-1/K, 1/K): every latent would map to the same code.  Give the codes the latents' own statistics
    # (per-channel mean + spread) so that the argmin is exercised with realistic margins.
    zf = z0.permute(0, 2, 3, 1).reshape(-1, 64)
    cc.quantize.embedding.weight.copy_(zf.mean(0, keepdim=True) + torch.randn(K, 64, generator=g) * zf.std(0, keepdim=True))
    quant_z, tokens = model.get_tokens(mel)
    z = cc.quant_conv(cc.encoder(mel))
    sd = {k: v for k, v in model.state_dict().items()
          if k.startswith("content_codec.encoder.") or k.startswith("content_codec.quant_conv.") or k.startswith("content_codec.quantize.")}
    np.savez_compressed(os.path.join(GOLD, "encoder_tiny.npz"), in_mel=mel.numpy(), out_z=z.numpy(), out_tokens=tokens.numpy().astype(np.int16),
                        out_quant=quant_z.numpy(), __cfg=np.array([K, 64, 32, 2, 7]), **{"sd." + k: v.numpy() for k, v in sd.items()})
    print("encoder_tiny: z", tuple(z.shape), "tokens", tokens[0].tolist())


CAPTIONS = ["A dog barks while a man is talking", "  Rain falls   on a tin roof, thunder in the distance!  ", "someone's typing on a keyboard & it's loud",
            "Birds chirping; a car passes by (twice) at 60km/h", "A very long caption " + "with many many words " * 30, "", "caf\u00e9 na\u00efve \u00fcber 123 #tag @home",
            "An engine revving and tires squealing &amp; a crowd cheering"]


def gen_tokenizer_cases():
    """N2 (host side): the reference's SimpleTokenizer + clip.tokenize on a few captions (ftfy is not installed here: a pass-through stub,
    which is what ftfy.fix_text does on well-formed text)."""
    import json
    import types
    if "ftfy" not in sys.modules:
        sys.modules["ftfy"] = types.SimpleNamespace(fix_text=lambda t: t)
    rh.install_shims()
    from sound_synthesis.modeling.modules.clip.simple_tokenizer import SimpleTokenizer
    from sound_synthesis.modeling.modules.clip.clip import tokenize
    tk = SimpleTokenizer(end_idx=49152)
    out = tokenize(CAPTIONS, context_length=77, add_start_and_end=True, with_mask=True, pad_value=0, tokenizer=tk)
    raw = [tk.encode(c) for c in CAPTIONS]
    with open(os.path.join(GOLD, "tokenizer_cases.json"), "w") as f:
        json.dump({"captions": CAPTIONS, "token": out["token"].tolist(), "mask": out["mask"].int().tolist(), "encode": raw,
                   "sot": tk.encoder["<|startoftext|>"], "eot": tk.encoder["<|endoftext|>"]}, f)
    print("tokenizer_cases:", [len(r) for r in raw])


TOKENIZE_VARIANT_CAPTIONS = ["Two people talk while a dog barks and a car drives past on a wet road", "wind", "A B C d e f g h i j k l m n o p"]
TOKENIZE_VARIANTS = [(77, True, 0), (256, False, -100), (12, True, 0)]  # (context_length, add_start_and_end, pad_value)
CONFIG_CAPTIONS = ["a dog barks", "rain on a tin roof"]                  # what the caps.yaml test feeds prepare_condition


def gen_tokenize_variants():
    """clip.tokenize's option space (DALL-E style 256 without start/end tokens and -100 padding, a context short enough to truncate)."""
    import json
    import types
    if "ftfy" not in sys.modules:
        sys.modules["ftfy"] = types.SimpleNamespace(fix_text=lambda t: t)
    rh.install_shims()
    from sound_synthesis.modeling.modules.clip.simple_tokenizer import SimpleTokenizer
    from sound_synthesis.modeling.modules.clip.clip import tokenize
    cases = []
    for ctx, sot_eot, pad in TOKENIZE_VARIANTS:
        out = tokenize(TOKENIZE_VARIANT_CAPTIONS, context_length=ctx, add_start_and_end=sot_eot, with_mask=True, pad_value=pad, tokenizer=SimpleTokenizer(end_idx=49152))
        cases.append({"context_length": ctx, "add_start_and_end": sot_eot, "pad_value": pad, "token": out["token"].tolist(), "mask": out["mask"].int().tolist()})
    with open(os.path.join(GOLD, "tokenize_variants.json"), "w") as f:
        json.dump({"captions": TOKENIZE_VARIANT_CAPTIONS, "cases": cases}, f)
    print("tokenize_variants:", len(cases), "cases")


def gen_bpe_merges():
    """The merges of CLIP's BPE table that the reference's SimpleTokenizer applies while encoding every caption the CPU tests encode, with their
    ranks.  Greedy lowest-rank-first merging never applies a pair outside this set, so a table holding these pairs at these ranks (and inert
    pairs elsewhere, tests/helpers.py:golden_bpe_vocab) gives the full table's token ids for these captions."""
    import json
    import types
    if "ftfy" not in sys.modules:
        sys.modules["ftfy"] = types.SimpleNamespace(fix_text=lambda t: t)
    rh.install_shims()
    from sound_synthesis.modeling.modules.clip.simple_tokenizer import SimpleTokenizer

    class Applied(dict):  # SimpleTokenizer.bpe asks `bigram not in self.bpe_ranks` of the pair it is about to merge
        hits = set()

        def __contains__(self, pair):
            found = dict.__contains__(self, pair)
            if found:
                self.hits.add(pair)
            return found
    tk = SimpleTokenizer(end_idx=49152)
    tk.bpe_ranks = Applied(tk.bpe_ranks)
    captions = CAPTIONS + ["A dog barks"] + TOKENIZE_VARIANT_CAPTIONS + CONFIG_CAPTIONS
    for c in captions:
        tk.encode(c)
    merges = sorted([tk.bpe_ranks[p], p[0], p[1]] for p in tk.bpe_ranks.hits)
    with open(os.path.join(GOLD, "bpe_merges.json"), "w") as f:
        json.dump({"n_merges": len(tk.bpe_ranks), "captions": captions, "merges": merges}, f, ensure_ascii=False)
    print("bpe_merges:", len(merges), "of", len(tk.bpe_ranks))


def gen_reference_configs():
    """The `model` blocks of the reference's configs/caps.yaml and evaluation/caps_text.yaml."""
    import json
    with open(os.path.join(GOLD, "reference_configs.json"), "w") as f:
        json.dump({name: rh.load_config(name)["model"] for name in ("configs/caps.yaml", "evaluation/caps_text.yaml")}, f, indent=1)
    print("reference_configs: 2")


def gen_host_policies():
    """Host-side policies of the reference DiffusionTransformer: parameter / buffer names, the AdamW grouping of parameters(name='transformer'),
    and sample_time('importance') before and after the switch-over (tests/test_cpu_host.py:test_host_policies_match_live_reference_module)."""
    import json
    K = 32
    model, _ = rh.build_dalle(K=K, overrides=dict(n_layer=2, n_embd=128, n_head=2, condition_dim=64, dec_ch=32, dec_ch_mult=[1, 1, 1, 1, 2],
                                                  dec_z_channels=64, embed_dim=64), seed=0)
    ref = model.transformer
    import ast
    try:
        ref.parameters(name="transformer")
        groups_error = None
    except AssertionError as e:  # "parameters {<names>} were not separated ...": store the names sorted (a set prints in hash order)
        names, _, rest = str(e).partition(" were not")
        groups_error = {"unseparated": sorted(ast.literal_eval(names[len("parameters "):])), "message": "were not" + rest}
    sample_time = []
    for count, hist in ((0.0, None), (11.0, torch.linspace(0.5, 9.0, 100))):
        ref.Lt_count.fill_(count)
        if hist is not None:
            ref.Lt_history.copy_(hist)
        torch.manual_seed(42)
        t, pt = ref.sample_time(16, torch.device("cpu"), "importance")
        sample_time.append({"t": t.tolist(), "pt": pt.tolist()})
    with open(os.path.join(GOLD, "host_policies.json"), "w") as f:
        json.dump({"state_dict_keys": sorted(ref.state_dict()), "named_groups_error": groups_error, "sample_time": sample_time}, f, indent=1)
    print("host_policies:", len(ref.state_dict()), "keys")


def gen_ema():
    """The reference's EMA (engine/ema.py) over the update sequence of tests/test_cpu_host.py:test_device_resident_ema_matches_reference_ema
    (same module, same seeds: keep the two in step)."""
    rh.install_shims()
    from sound_synthesis.engine.ema import EMA

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(0)
            self.body = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.LayerNorm(32), torch.nn.Linear(32, 8))
            self.register_buffer("steps", torch.zeros(3))

        def get_ema_model(self):
            return self.body
    a = Net()
    ema = EMA(a, decay=0.9, update_interval=2)
    g = torch.Generator().manual_seed(1)
    for it in range(7):
        for p in a.parameters():
            p.data.add_(torch.randn(p.shape, generator=g) * 0.01)
        ema.update(it)
    np.savez_compressed(os.path.join(GOLD, "ema_reference.npz"), **{k: v.numpy() for k, v in ema.state_dict().items()})
    print("ema_reference:", len(ema.state_dict()), "tensors")


def gen_clip_text():
    """N2: the reference's CLIPTextEmbedding.forward (Diffsound flags) on seeded weights.  CLIPTextEmbedding.__init__ downloads CLIP, so the instance
    is assembled by hand from the reference's own sub-modules (clip/model.py Transformer + LayerNorm) and driven through its unmodified forward()."""
    import types
    from oracle import diffsound_oracle as O
    rh.install_shims()
    if "ftfy" not in sys.modules:  # imported by the reference's tokenizer module, unused here
        sys.modules["ftfy"] = types.SimpleNamespace(fix_text=lambda t: t)
    from sound_synthesis.modeling.modules.clip import model as cm
    from sound_synthesis.modeling.embeddings.clip_text_embedding import CLIPTextEmbedding
    NL, V = 3, 2000
    sd = O.make_clip_text_state_dict(n_layer=NL, vocab=V, seed=5)
    emb = object.__new__(CLIPTextEmbedding)
    torch.nn.Module.__init__(emb)
    emb.num_embed, emb.clip_name, emb.normalize, emb.pick_last_embedding, emb.keep_seq_len_dim, emb.additional_last_embedding = V, "none", True, False, False, False
    mask = torch.empty(77, 77).fill_(float("-inf")).triu_(1)
    emb.token_embedding = torch.nn.Embedding(V, 512)
    emb.positional_embedding = torch.nn.Parameter(torch.empty(77, 512))
    emb.transformer = cm.Transformer(width=512, layers=NL, heads=8, attn_mask=mask)
    emb.ln_final = cm.LayerNorm(512)
    emb.text_projection = torch.nn.Parameter(torch.empty(512, 512))
    emb.embed_dim, emb.trainable = 512, False
    missing, unexpected = emb.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(6)
    tok = torch.zeros(3, 77, dtype=torch.long)
    for i, n_ in enumerate((9, 77, 30)):
        tok[i, :n_] = torch.randint(1, V, (n_,), generator=g)
    tok[2, 40] = -100   # padded ids may be negative (Tokenize pad_value=-100 configs): the reference clamps them to 0 in place
    out = emb(tok.clone())
    np.savez_compressed(os.path.join(GOLD, "clip_text.npz"), in_tokens=tok.numpy(), out_features=out.numpy(), __cfg=np.array([NL, V, 5]))
    print("clip_text:", tuple(out.shape), float(out.norm(dim=-1).mean()))


def gen_melgan():
    rh.install_shims()
    from vocoder.modules import Generator
    torch.manual_seed(5)
    gen = Generator(80, 4, 3).eval()
    g = torch.Generator().manual_seed(13)
    with torch.no_grad():
        for n, p in gen.named_parameters():  # weights_init gives N(0,0.02) v with g=|v|; make g and bias non-trivial
            if n.endswith("weight_g"):
                p.mul_(1 + 0.2 * torch.randn(p.shape, generator=g))
            if n.endswith("bias"):
                p.add_(0.05 * torch.randn(p.shape, generator=g))
        mel = torch.rand(2, 80, 24, generator=g)
        wav = gen(mel)
    np.savez_compressed(os.path.join(GOLD, "melgan_tiny.npz"), in_mel=mel.numpy(), out_wav=wav.numpy(),
                        **{"sd." + k: v.numpy() for k, v in gen.state_dict().items()})
    # real shipped checkpoint: only input/output are committed; the weights travel in oracle/_ref/
    real = rh.build_vocoder(real_weights=True)
    mel = torch.rand(1, 80, 40, generator=g)
    with torch.no_grad():
        wav = real(mel)
    np.savez_compressed(os.path.join(GOLD, "melgan_real_io.npz"), in_mel=mel.numpy(), out_wav=wav.numpy())
    print("melgan: tiny wav", tuple(gen(torch.rand(1, 80, 8)).shape), "real wav absmax", float(wav.abs().max()))


def gen_schedule():
    model, _ = rh.build_dalle(K=256, overrides=dict(n_layer=1, n_embd=64, n_head=1, dec_ch=32, dec_ch_mult=[1, 1, 1, 1, 2]), seed=0)
    tr = model.transformer
    names = ["log_at", "log_bt", "log_ct", "log_cumprod_at", "log_cumprod_bt", "log_cumprod_ct", "log_1_min_ct", "log_1_min_cumprod_ct"]
    np.savez_compressed(os.path.join(GOLD, "schedule_k256.npz"), **{n: getattr(tr, n).numpy() for n in names})


if __name__ == "__main__":
    assert rh.available(), "reference tree not found"
    os.makedirs(GOLD, exist_ok=True)
    torch.set_grad_enabled(False)
    gen_schedule()
    gen_train_tiny(gen_xf_tiny())
    gen_sampler_cases()
    gen_decoder_tiny()
    gen_encoder_tiny()
    gen_tokenizer_cases()
    gen_tokenize_variants()
    gen_bpe_merges()
    gen_reference_configs()
    gen_host_policies()
    gen_ema()
    gen_clip_text()
    gen_melgan()
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)) // 1024, "KB")
