"""CPU-side checks (no GPU): C-ABI surface, drop-in module construction / checkpoint-key compatibility, config factory,
no-fallback behaviour, the sharded driver's host logic over gloo, and the reference-arm bench line."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from tests.helpers import ROOT, golden_bpe_vocab, load_golden, load_golden_json

import _pkg

_pkg.load()


def test_cabi_library_exports_every_declared_symbol():
    from diffsound_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "diffsound_b200.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(dsb_\w+)\s*\(", hdr, flags=re.M))
    assert len(declared) >= 20
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name), f"libdiffsound_b200.so does not export {name}"
    assert declared - {"dsb_last_error"} == set(_lib.SIGNATURES), "ctypes signatures out of sync with the header"
    assert L.dsb_version() == 100


def test_gemm_descriptor_layout_matches_header():
    """sizeof(struct dsb_gemm_desc) as laid out by ctypes == what a C compiler produces for the header."""
    from diffsound_b200 import _lib
    import ctypes, tempfile
    src = '#include <stdio.h>\n#include "diffsound_b200.h"\nint main(){printf("%zu %zu %zu", sizeof(dsb_gemm_desc), __builtin_offsetof(dsb_gemm_desc, tap_shift), __builtin_offsetof(dsb_gemm_desc, alpha));return 0;}'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")], check=True)
        out = subprocess.run([os.path.join(d, "t")], capture_output=True, text=True, check=True).stdout.split()
    assert int(out[0]) == ctypes.sizeof(_lib.GemmDesc)
    assert int(out[1]) == _lib.GemmDesc.tap_shift.offset and int(out[2]) == _lib.GemmDesc.alpha.offset


def test_ops_refuse_cpu_tensors_no_fallback():
    from diffsound_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.round_tf32(torch.zeros(8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.gemm(torch.zeros(4, 32), torch.zeros(4, 32))


def _dt(K, D, NL, NH, CD):
    from tests.test_gpu_transformer import build_dt
    real_cuda = torch.nn.Module.cuda
    torch.nn.Module.cuda = lambda self, *a, **k: self
    try:
        return build_dt(K, D, NL, NH, CD)
    finally:
        torch.nn.Module.cuda = real_cuda


def test_dropin_modules_keep_reference_state_dict_keys():
    sd, g = load_golden("xf_tiny.npz")
    K, D, NL, NH, CD, B, L = [int(v) for v in g["__cfg"]]
    m = _dt(K, D, NL, NH, CD)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and all("attn2.mask" in k for k in missing)
    assert m.num_classes == K + 1 and m.shape == 265 and m.num_timesteps == 100
    with pytest.raises(RuntimeError, match="CUDA"):
        m.sample(None, None, torch.zeros(B, 77, CD), filter_ratio=0, batch_size=B)
    # decoder + vocoder
    from tests.test_gpu_decoder import build_vq
    from diffsound_b200.vocoder.modules import Generator
    dsd, dg = load_golden("decoder_tiny.npz")
    real_cuda = torch.nn.Module.cuda
    torch.nn.Module.cuda = lambda self, *a, **k: self
    try:
        vq = build_vq(int(dg["__cfg"][0]), int(dg["__cfg"][1]), int(dg["__cfg"][2]), (1, 1, 1, 1, 2), dsd)
    finally:
        torch.nn.Module.cuda = real_cuda
    assert not vq.engine.packed
    msd, _ = load_golden("melgan_tiny.npz")
    Generator(80, 4, 3).load_state_dict(msd, strict=True)
    with pytest.raises(RuntimeError):
        Generator(80, 4, 3)(torch.zeros(1, 80, 8))


def test_stage_methods_stay_rebindable_and_truncation_parses():
    from diffsound_b200.modeling.transformers.diffusion_transformer import parse_truncation
    assert parse_truncation("top0.85r") == (1, 0.85, 0)
    assert parse_truncation("top100p") == (2, 0.0, 100)
    assert parse_truncation("top0.85r,fast3") == (1, 0.85, 0)
    assert parse_truncation("normal") == (0, 0.0, 0) and parse_truncation(None) == (0, 0.0, 0)
    m = _dt(32, 128, 1, 2, 64)
    assert not m._stages_overridden()
    m.predict_start = (lambda f: (lambda *a, **k: f(*a, **k)))(m.predict_start)  # what the reference DALLE does (dalle_spec.py:209)
    assert m._stages_overridden()


def test_config_factory_and_retarget():
    from diffsound_b200.utils.misc import instantiate_from_config, retarget_config
    cfg = {"target": "sound_synthesis.modeling.models.dalle_spec.DALLE", "params": {
        "content_codec_config": {"target": "sound_synthesis.modeling.codecs.spec_codec.vqgan.VQModel", "params": {
            "ckpt_path": None, "embed_dim": 64, "n_embed": 32, "lossconfig": {"target": "specvqgan.modules.losses.DummyLoss"},
            "ddconfig": dict(double_z=False, z_channels=64, resolution=848, in_channels=1, out_ch=1, ch=32, ch_mult=[1, 1, 1, 1, 2],
                             num_res_blocks=2, attn_resolutions=[53], dropout=0.0)}},
        "condition_codec_config": None,
        "first_stage_permuter_config": {"target": "specvqgan.modules.transformer.permuter.ColumnMajor", "params": {"H": 5, "W": 53}},
        "diffusion_config": {"target": "sound_synthesis.modeling.transformers.diffusion_transformer.DiffusionTransformer", "params": {
            "diffusion_step": 100, "alpha_init_type": "alpha1", "auxiliary_loss_weight": 5.0e-4, "adaptive_auxiliary_loss": True, "mask_weight": [1, 1],
            "condition_emb_config": None,
            "transformer_config": {"target": "sound_synthesis.modeling.transformers.transformer_utils.Text2ImageTransformer", "params": dict(
                attn_type="selfcross", n_layer=1, condition_seq_len=77, content_seq_len=265, content_spatial_size=[5, 53], n_embd=64, condition_dim=64,
                n_head=1, attn_pdrop=0.0, resid_pdrop=0.0, block_activate="GELU2", timestep_type="adalayernorm", mlp_hidden_times=4)},
            "content_emb_config": {"target": "sound_synthesis.modeling.embeddings.dalle_mask_image_embedding.DalleMaskImageEmbedding", "params": dict(
                num_embed=32, spatial_size=(5, 53), embed_dim=64, trainable=True, pos_emb_type="embedding")}}}}}
    new = retarget_config(cfg)
    assert new["target"].startswith("diffsound_b200.") and cfg["target"].startswith("sound_synthesis.")  # input not mutated
    model = instantiate_from_config(new)
    keys = set(model.state_dict().keys())
    assert "transformer.transformer.blocks.0.attn1.query.weight" in keys and "content_codec.decoder.conv_in.weight" in keys
    assert "first_stage_permuter.forward_shuffle_idx" in keys and "transformer.log_cumprod_at" in keys
    ids = torch.arange(265).view(1, 265)
    perm = model.first_stage_permuter
    assert torch.equal(perm(perm(ids), reverse=True), ids)
    assert perm(ids)[0, 1].item() == 53  # column-major: second token is row 1 of column 0


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import _pkg
    _pkg.load()
    from diffsound_b200 import pipeline

    class FakeDalle:
        device = torch.device("cpu")

        def generate_content(self, *, batch, **kw):
            c = batch["condition_embed"]
            tok = (c[:, 0, :3].sum(-1, keepdim=True) * 1000).long().expand(-1, 5) + torch.randint(0, 1 << 20, (1,))  # seed-dependent
            return {"content": torch.zeros(c.shape[0], 1, 2, 4), "content_token": tok}

    cond = torch.arange(8 * 77 * 4, dtype=torch.float32).view(8, 77, 4) / 100
    out = pipeline.synthesize_sharded(FakeDalle(), lambda s: s.sum(-1, keepdim=True).unsqueeze(1), cond, base_seed=7)
    q.put((rank, out["tokens"].clone(), out["wav"].shape))
    dist.destroy_process_group()


def test_sharded_driver_over_gloo_world2():
    import torch.multiprocessing as mp
    import socket
    ctx = mp.get_context("spawn")
    res = None
    for attempt in range(3):  # a stale TIME_WAIT socket on the rendezvous port must not fail the suite
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        q = ctx.Queue()
        procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
        [p.start() for p in procs]
        try:
            res = sorted([q.get(timeout=120) for _ in procs], key=lambda r: r[0])
        except Exception:
            res = None
        [p.join(60) for p in procs]
        if res is not None and all(p.exitcode == 0 for p in procs):
            break
        [p.kill() for p in procs if p.is_alive()]
        res = None
    assert res is not None, "gloo world-size-2 run failed three times"
    (r0, t0, s0), (r1, t1, s1) = res
    assert torch.equal(t0, t1) and t0.shape == (8, 5) and s0 == s1  # every rank holds all 8 clips, in caption order
    # rank-local seeds differ (base_seed + rank), captions are contiguous blocks of 4
    torch.manual_seed(7); a = torch.randint(0, 1 << 20, (1,))
    torch.manual_seed(8); b = torch.randint(0, 1 << 20, (1,))
    cond = torch.arange(8 * 77 * 4, dtype=torch.float32).view(8, 77, 4) / 100
    base = (cond[:, 0, :3].sum(-1, keepdim=True) * 1000).long().expand(-1, 5)
    assert torch.equal(t0[:4], base[:4] + a) and torch.equal(t0[4:], base[4:] + b)


def test_bench_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--layers", "1", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "clips/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0


def test_save_clip_writes_reference_layout(tmp_path):
    import wave
    import numpy as np
    from diffsound_b200 import pipeline
    mel = torch.linspace(-1, 1, 80 * 848).view(1, 80, 848)
    wav = torch.sin(torch.linspace(0, 100, 22050)).view(1, -1) * 0.5
    stem = pipeline.save_clip(str(tmp_path), "Y123", 3, mel, wav)
    assert stem.endswith("Y123_mel_sample_3")
    spec = np.load(stem + ".npy")
    assert spec.shape == (80, 848) and abs(float(spec.min())) < 1e-6 and abs(float(spec.max()) - 1.0) < 1e-6  # [0,1] as generate_samples_batch.py:181
    with wave.open(stem + ".wav", "rb") as f:
        assert (f.getnchannels(), f.getsampwidth(), f.getframerate(), f.getnframes()) == (1, 3, 22050, 22050)
        raw = np.frombuffer(f.readframes(4), dtype=np.uint8).reshape(-1, 3).astype(np.int32)
    val = raw[:, 0] | (raw[:, 1] << 8) | (raw[:, 2] << 16)
    val = np.where(val >= 1 << 23, val - (1 << 24), val)
    assert np.allclose(val / 8388607.0, wav[0, :4].numpy(), atol=2e-7)


def test_training_host_logic_without_gpu():
    """A13 host side on the CPU: optimizer groups of parameters(name=...), sample_time policy, the flat gradient layout of the training engine
    (every parameter a non-overlapping, correctly shaped view) -- no kernel is launched."""
    import _pkg
    _pkg.load()
    from diffsound_b200.modeling.transformers.diffusion_transformer import DiffusionTransformer
    K, D, NL = 32, 128, 2
    m = DiffusionTransformer(
        content_emb_config=dict(target="diffsound_b200.modeling.embeddings.dalle_mask_image_embedding.DalleMaskImageEmbedding",
                                params=dict(num_embed=K, spatial_size=(5, 53), embed_dim=D, trainable=True, pos_emb_type="embedding")),
        condition_emb_config=None,
        transformer_config=dict(target="diffsound_b200.modeling.transformers.transformer_utils.Text2ImageTransformer",
                                params=dict(attn_type="selfcross", n_layer=NL, condition_seq_len=77, content_seq_len=265, content_spatial_size=[5, 53],
                                            n_embd=D, condition_dim=64, n_head=2, attn_pdrop=0.0, resid_pdrop=0.0, block_activate="GELU2",
                                            timestep_type="adalayernorm", mlp_hidden_times=4)),
        diffusion_step=100, alpha_init_type="alpha1", auxiliary_loss_weight=5.0e-4, adaptive_auxiliary_loss=True, mask_weight=[1, 1])
    # optimizer groups (reference diffusion_transformer.py:483-537): Linear weights decayed, everything else not; every parameter exactly once
    decay, no_decay = m.parameters(name="transformer")
    assert decay["weight_decay"] == 0.01 and no_decay["weight_decay"] == 0.0
    ids = [id(p) for p in decay["params"] + no_decay["params"]]
    assert len(ids) == len(set(ids)) == len(list(m.transformer.parameters()))
    assert all(p.dim() == 2 for p in decay["params"])
    assert any(p.shape == (K + 1, D) for p in no_decay["params"])  # the token embedding is an nn.Embedding: not decayed
    # sample_time (:379-406): uniform until every Lt_count > 10, then importance sampling proportional to sqrt(Lt_history) with entry 0 <- entry 1
    torch.manual_seed(0)
    t, pt = m.sample_time(64, "cpu", "importance")
    assert t.shape == (64,) and torch.all(pt == 0.01) and int(t.max()) < 100
    m.Lt_count.fill_(11.0)
    m.Lt_history.copy_(torch.linspace(1.0, 4.0, 100))
    t, pt = m.sample_time(64, "cpu", "importance")
    w = torch.sqrt(m.Lt_history + 1e-10) + 0.0001
    w[0] = w[1]
    assert torch.allclose(pt, (w / w.sum())[t])
    # flat gradient layout of the training engine
    eng = m.transformer.train_engine
    eng.D, eng.H, eng.n_layer, eng.Cd = D, 2, NL, 64
    layout, total = eng._grad_layout()
    views = eng._grad_views(torch.zeros(total))
    spans = []
    for n, p in m.transformer.named_parameters():
        v = views[n]
        assert v.shape == p.shape and v.is_contiguous(), n
        spans.append((v.data_ptr(), v.data_ptr() + v.numel() * 4))
    spans.sort()
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:])), "parameter gradient views overlap"
    assert all(o % 64 == 0 for _, _, o in layout)


def test_clip_tokenizer_matches_reference_cases(tmp_path):
    """N2 host side: the re-implemented CLIP BPE tokenizer + Tokenize codec vs token ids produced by the reference's own SimpleTokenizer /
    clip.tokenize (tests/golden/tokenizer_cases.json), over the golden merge table (CLIP's own table is not redistributed here)."""
    import json
    import _pkg
    _pkg.load()
    from diffsound_b200.modeling.modules.clip.simple_tokenizer import SimpleTokenizer
    from diffsound_b200.modeling.codecs.text_codec.tokenize import Tokenize
    bpe = golden_bpe_vocab(tmp_path)
    with open(os.path.join(ROOT, "tests", "golden", "tokenizer_cases.json")) as f:
        g = json.load(f)
    tk = SimpleTokenizer(end_idx=49152, bpe_path=bpe)
    assert tk.encoder["<|startoftext|>"] == g["sot"] and tk.encoder["<|endoftext|>"] == g["eot"] and len(tk.encoder) == 49408
    for cap, ref in zip(g["captions"], g["encode"]):
        assert tk.encode(cap) == ref, cap
    assert tk.decode(tk.encode("A dog barks")).strip() == "a dog barks"
    codec = Tokenize(context_length=77, add_start_and_end=True, with_mask=True, pad_value=0, clip_embedding=False,
                     tokenizer_config={"target": "diffsound_b200.modeling.modules.clip.simple_tokenizer.SimpleTokenizer", "params": {"end_idx": 49152, "bpe_path": bpe}})
    out = codec.get_tokens(g["captions"])
    assert out["token"].tolist() == g["token"] and out["mask"].int().tolist() == g["mask"]
    assert int(out["token"][4, 76]) == g["eot"] and bool(out["mask"][4].all())  # the over-long caption is truncated but keeps <|endoftext|>


def test_reference_yaml_retargets_to_dropins_including_text_front_end(tmp_path):
    """The `model` block of the reference's own configs/caps.yaml (tests/golden/reference_configs.json) -> retarget_config -> every `target:` of the
    hot path resolves to a drop-in class, the model builds on the CPU (modules only hold parameters), and its state_dict carries the reference's
    key families."""
    from diffsound_b200.utils.misc import instantiate_from_config, retarget_config
    cfg = load_golden_json("reference_configs.json")["configs/caps.yaml"]
    cfg["params"]["content_codec_config"]["params"]["ckpt_path"] = None          # no checkpoints in the tree
    new = retarget_config(cfg)

    def targets(c):
        if isinstance(c, dict):
            return ([c["target"]] if isinstance(c.get("target"), str) else []) + [t for v in c.values() for t in targets(v)]
        return [t for v in c for t in targets(v)] if isinstance(c, (list, tuple)) else []
    left = [t for t in targets(new) if not t.startswith("diffsound_b200.")]
    assert left == ["specvqgan.modules.losses.DummyLoss"], left                    # the (unused) stage-1 loss is the only reference class left
    new["params"]["content_codec_config"]["params"]["lossconfig"] = None
    new["params"]["condition_codec_config"]["params"]["tokenizer_config"]["params"]["bpe_path"] = golden_bpe_vocab(tmp_path)
    model = instantiate_from_config(new)
    keys = set(model.state_dict().keys())
    for k in ("transformer.condition_emb.transformer.resblocks.11.attn.in_proj_weight", "transformer.condition_emb.token_embedding.weight",
              "transformer.transformer.blocks.18.mlp.2.weight", "transformer.transformer.to_logits.1.bias", "content_codec.encoder.down.4.attn.1.q.weight",
              "content_codec.decoder.up.4.attn.2.proj_out.bias", "content_codec.quantize.embedding.weight", "transformer.Lt_history"):
        assert k in keys, k
    assert model.transformer.condition_emb.embed_dim == 512 and model.transformer.transformer.content_emb.num_embed == 257
    cond = model.prepare_condition({"text": ["a dog barks", "rain on a tin roof"]})
    tk = model.condition_codec.tokenizer
    want = sum(len(tk.encode(t)) + 2 for t in ("a dog barks", "rain on a tin roof"))  # <|startoftext|> ... <|endoftext|>
    assert cond["condition_token"].shape == (2, 77) and cond["condition_mask"].dtype == torch.bool and int(cond["condition_mask"].sum()) == want
    assert int(cond["condition_token"][0, 0]) == tk.encoder["<|startoftext|>"]


def test_device_resident_ema_matches_reference_ema():
    """N4 remainder: engine_utils.ema.EMA (shadow weights kept on the model's device, fused multi-tensor update) vs the reference's EMA class
    (CPU state_dict round trip) over several updates, plus the swap-in / swap-out used around validation (solver_spec.py).  The reference's
    shadow weights after this update sequence are tests/golden/ema_reference.npz (oracle/gen_golden.py:gen_ema: keep the two in step)."""
    import numpy as np
    from diffsound_b200.engine_utils.ema import EMA

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(0)
            self.body = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.LayerNorm(32), torch.nn.Linear(32, 8))
            self.register_buffer("steps", torch.zeros(3))

        def get_ema_model(self):
            return self.body

        @property
        def device(self):
            return torch.device("cpu")

    b = Net()
    mine = EMA(b, decay=0.9, update_interval=2)
    g = torch.Generator().manual_seed(1)
    for it in range(7):
        for pb in b.parameters():
            pb.data.add_(torch.randn(pb.shape, generator=g) * 0.01)
        mine.update(it)
    with np.load(os.path.join(ROOT, "tests", "golden", "ema_reference.npz")) as z:
        ref = {k: torch.from_numpy(z[k]) for k in z.files}
    assert set(ref) == set(mine.state_dict())
    assert all(torch.allclose(ref[k], mine.state_dict()[k], rtol=0, atol=2e-6) for k in ref)
    assert not torch.allclose(mine.state_dict()["0.weight"], b.body[0].weight)  # the shadow lags the live weights
    live = {k: v.clone() for k, v in b.body.state_dict().items()}
    mine.modify_to_inference()
    assert all(torch.equal(b.body.state_dict()[k], mine.state_dict()[k]) for k in live)
    mine.modify_to_train()
    assert all(torch.equal(b.body.state_dict()[k], live[k]) for k in live)
    assert not any(p.requires_grad for p in mine.ema_model.parameters())


def test_generate_samples_cli_dry_run_on_reference_yaml(tmp_path):
    """tools/generate_samples.py (the generate_samples_batch.py flow on the drop-ins): config retargeting, caption grouping, sample_type string.
    The config is the `model` block of the reference's evaluation/caps_text.yaml (tests/golden/reference_configs.json)."""
    import yaml
    cfgp = tmp_path / "caps_text.yaml"
    cfgp.write_text(yaml.safe_dump({"model": load_golden_json("reference_configs.json")["evaluation/caps_text.yaml"]}))
    import importlib.util
    spec = importlib.util.spec_from_file_location("generate_samples", os.path.join(ROOT, "tools", "generate_samples.py"))
    gs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gs)
    csvp = tmp_path / "val.csv"
    csvp.write_text("file_name,caption\nY1.wav,a dog barks\nY1.wav,\"a dog barks, twice\"\nY2.wav,rain\n")
    ck = os.path.join(ROOT, "oracle", "_ref", "best_netG.pt")
    argv = ["--config", str(cfgp), "--bpe", golden_bpe_vocab(tmp_path), "--captions", str(csvp), "--out", str(tmp_path / "o"), "--fast", "3",
            "--dry-run"] + (["--vocoder-ckpt", ck] if os.path.exists(ck) else [])
    model, vocoder, caps, st = gs.main(argv)
    assert caps == {"Y1.wav": ["a dog barks", "a dog barks, twice"], "Y2.wav": ["rain"]} and st == "top0.85r,fast2"
    assert type(model).__module__.startswith("diffsound_b200.") and model.condition_codec is not None
    assert model.transformer.condition_emb is not None and (vocoder is None or type(vocoder).__module__.startswith("diffsound_b200."))


def test_synthesize_captions_sharding_and_replication_logic():
    """pipeline.synthesize_captions: single process (no group) keeps every caption; replicate repeats the whole caption block, as generate_content's
    torch.cat does; the caption index list says which caption each clip belongs to."""
    from diffsound_b200 import pipeline

    class FakeDalle:
        def generate_content(self, *, batch, filter_ratio, replicate, sample_type):
            n = len(batch["text"]) * replicate
            ids = torch.tensor([len(t) for t in batch["text"]] * replicate)
            return {"content": ids.float().view(n, 1, 1, 1).expand(n, 1, 2, 4).contiguous(), "content_token": ids.view(n, 1)}

    caps = ["a", "bb", "ccc"]
    out = pipeline.synthesize_captions(FakeDalle(), lambda s: s.sum(-1, keepdim=True).unsqueeze(1), caps, replicate=2, seed=5)
    assert out["caption_index"] == [0, 1, 2, 0, 1, 2]
    assert out["tokens"].view(-1).tolist() == [1, 2, 3, 1, 2, 3] and out["mel"].shape == (6, 1, 2, 4) and out["wav"].shape == (6, 1, 2, 1)
    assert pipeline.synthesize_captions(FakeDalle(), None, caps)["wav"] is None


def test_host_policies_match_live_reference_module():
    """sample_time (importance / uniform) and the AdamW grouping of parameters(name=...) against what the reference's own DiffusionTransformer of
    the same configuration gives (tests/golden/host_policies.json)."""
    K = 32
    ref = load_golden_json("host_policies.json")
    from diffsound_b200.modeling.transformers.diffusion_transformer import DiffusionTransformer
    mine = DiffusionTransformer(
        content_emb_config=dict(target="diffsound_b200.modeling.embeddings.dalle_mask_image_embedding.DalleMaskImageEmbedding",
                                params=dict(num_embed=K, spatial_size=(5, 53), embed_dim=128, trainable=True, pos_emb_type="embedding")),
        condition_emb_config=None,
        transformer_config=dict(target="diffsound_b200.modeling.transformers.transformer_utils.Text2ImageTransformer",
                                params=dict(attn_type="selfcross", n_layer=2, condition_seq_len=77, content_seq_len=265, content_spatial_size=[5, 53],
                                            n_embd=128, condition_dim=64, n_head=2, attn_pdrop=0.0, resid_pdrop=0.0, block_activate="GELU2",
                                            timestep_type="adalayernorm", mlp_hidden_times=4)),
        diffusion_step=100, alpha_init_type="alpha1", auxiliary_loss_weight=5.0e-4, adaptive_auxiliary_loss=True, mask_weight=[1, 1])
    # identical parameter / buffer names
    assert set(ref["state_dict_keys"]) == {k for k in mine.state_dict()}
    # AdamW groups: the reference's named branch cannot run -- its decay / no_decay names carry the 'transformer.' prefix while its param_dict does
    # not, so its own completeness assert fires (diffusion_transformer.py:522-529; the shipped configs only use name='none').  The drop-in
    # implements the documented intent (minGPT split) and must cover every parameter exactly once.
    assert "were not separated" in ref["named_groups_error"]["message"]
    decay, no_decay = mine.parameters(name="transformer")
    names = {id(p): n for n, p in mine.transformer.named_parameters()}
    d, nd = {names[id(p)] for p in decay["params"]}, {names[id(p)] for p in no_decay["params"]}
    assert not (d & nd) and (d | nd) == set(names.values()) >= set(ref["named_groups_error"]["unseparated"])
    assert all(n.endswith("weight") and "emb" not in n and "ln2" not in n and "to_logits.0" not in n for n in d)
    # sample_time: same generator stream -> same (t, pt), before and after the importance switch-over
    for (count, hist), want in zip(((0.0, None), (11.0, torch.linspace(0.5, 9.0, 100))), ref["sample_time"]):
        mine.Lt_count.fill_(count)
        if hist is not None:
            mine.Lt_history.copy_(hist)
        torch.manual_seed(42)
        t_m, pt_m = mine.sample_time(16, torch.device("cpu"), "importance")
        assert torch.equal(torch.tensor(want["t"]), t_m) and torch.equal(torch.tensor(want["pt"], dtype=pt_m.dtype), pt_m)


@pytest.mark.parametrize("ctx,sot_eot,pad", [(77, True, 0), (256, False, -100), (12, True, 0)])
def test_tokenize_variants_match_live_reference(ctx, sot_eot, pad, tmp_path):
    """Tokenize / clip.tokenize option space (DALL-E style 256 without start/end tokens and -100 padding, and a context short enough to truncate)
    against what the reference's own functions give (tests/golden/tokenize_variants.json)."""
    from diffsound_b200.modeling.codecs.text_codec.tokenize import Tokenize
    g = load_golden_json("tokenize_variants.json")
    ref = next(c for c in g["cases"] if (c["context_length"], c["add_start_and_end"], c["pad_value"]) == (ctx, sot_eot, pad))
    mine = Tokenize(context_length=ctx, add_start_and_end=sot_eot, with_mask=True, pad_value=pad,
                    tokenizer_config={"target": "diffsound_b200.modeling.modules.clip.simple_tokenizer.SimpleTokenizer",
                                      "params": {"end_idx": 49152, "bpe_path": golden_bpe_vocab(tmp_path)}}).get_tokens(g["captions"])
    assert (mine["token"].dtype, mine["mask"].dtype) == (torch.int64, torch.bool)  # the reference's dtypes
    assert mine["token"].tolist() == ref["token"] and mine["mask"].int().tolist() == ref["mask"]
