"""CLIP text tower without a GPU: key layout and parameter count of the full-width model against transformers'
CLIPTextModel, the loader, the host model (kernels emulated in torch, causal attention included) against transformers in
fp32, the tokenizer against transformers' CLIPTokenizer on a tiny vocabulary, the composition's prompt stack against
the golden seams, the argument checks of mvoc_attn_causal_fwd, and the scripts' text paths."""
import collections
import json
import os

import pytest
import torch
import torch.nn.functional as F

from tests import cpu_ops_emulation as emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
FULL_PARAMS = 340_387_840
FULL = dict(vocab_size=49408, hidden_size=1024, intermediate_size=4096, num_hidden_layers=23, num_attention_heads=16,
            max_position_embeddings=77)   # the reference checkpoint's text_encoder/config.json (layer count assumed)
# head_dim 64 like the checkpoint, widths multiples of 64 like the kernels need
SMALL = dict(vocab_size=1000, hidden_size=256, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4,
             max_position_embeddings=77)


def _hf_model(**kw):
    transformers = pytest.importorskip("transformers")
    cfg = transformers.CLIPTextConfig(hidden_act="gelu", layer_norm_eps=1e-5, **kw)
    cfg._attn_implementation = "eager"
    return transformers.CLIPTextModel(cfg).eval()


def _small_cfg(**over):
    from mvoc_b200.clip_text import CLIPTextConfig

    return CLIPTextConfig(**{**SMALL, **over})


def test_full_width_layout_and_parameter_count():
    from mvoc_b200.clip_text import CLIPTextEncoder

    with torch.device("meta"):
        ours = CLIPTextEncoder()
        ref = _hf_model(**FULL)
    mine = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    theirs = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert mine == theirs
    assert sum(v.numel() for v in ours.parameters()) == FULL_PARAMS
    assert "text_model.final_layer_norm.weight" in mine and "text_model.encoder.layers.22.mlp.fc2.bias" in mine
    assert all(layer.self_attn.causal for layer in ours.text_model.encoder.layers)


# ------------------------------------------------------------------ loader
@pytest.fixture()
def small_files(tmp_path):
    torch.manual_seed(0)
    sd = _hf_model(**SMALL).state_dict()
    from safetensors.torch import save_file

    pt, st = str(tmp_path / "text.pt"), str(tmp_path / "text.safetensors")
    torch.save(sd, pt)
    save_file({k: v.contiguous() for k, v in sd.items()}, st)
    return sd, pt, st


@pytest.mark.parametrize("fmt", ["pt", "safetensors"])
def test_loader_round_trip(small_files, fmt):
    from mvoc_b200.clip_text import load_clip_text_encoder

    sd, pt, st = small_files
    enc = load_clip_text_encoder(pt if fmt == "pt" else st, "cpu", torch.float32, cfg=_small_cfg())
    got = enc.state_dict()
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    assert all(k.startswith("text_model.") for k in got)


def test_loader_ignores_the_other_tower_and_position_ids(small_files, tmp_path):
    from mvoc_b200.clip_text import load_clip_text_encoder

    sd, _, _ = small_files
    extra = dict(sd)
    extra["text_model.embeddings.position_ids"] = torch.arange(77).view(1, -1)
    extra["vision_model.post_layernorm.weight"] = torch.zeros(4)
    extra["visual_projection.weight"] = torch.zeros(4, 4)
    extra["text_projection.weight"] = torch.zeros(4, 4)
    extra["logit_scale"] = torch.tensor(1.0)
    p = str(tmp_path / "full.pt")
    torch.save(extra, p)
    enc = load_clip_text_encoder(p, "cpu", torch.float32, cfg=_small_cfg())
    assert set(enc.state_dict()) == set(sd)


def test_loader_names_the_bad_key(small_files, tmp_path):
    from mvoc_b200.clip_text import load_clip_text_encoder

    sd, _, _ = small_files
    key = "text_model.encoder.layers.1.self_attn.k_proj.weight"
    missing = {k: v for k, v in sd.items() if k != key}
    torch.save(missing, tmp_path / "missing.pt")
    with pytest.raises(KeyError, match=key.replace(".", r"\.")):
        load_clip_text_encoder(str(tmp_path / "missing.pt"), "cpu", cfg=_small_cfg())
    bad = dict(sd)
    bad[key] = torch.zeros(7, 3)
    torch.save(bad, tmp_path / "shape.pt")
    with pytest.raises(ValueError, match=key.replace(".", r"\.")):
        load_clip_text_encoder(str(tmp_path / "shape.pt"), "cpu", cfg=_small_cfg())
    # a layer count other than the configuration's: the first extra or missing key is named
    torch.save(_hf_model(**{**SMALL, "num_hidden_layers": 3}).state_dict(), tmp_path / "deeper.pt")
    with pytest.raises(KeyError, match=r"unexpected CLIP text encoder key 'text_model\.encoder\.layers\.2\."):
        load_clip_text_encoder(str(tmp_path / "deeper.pt"), "cpu", cfg=_small_cfg())
    with pytest.raises(KeyError, match=r"missing CLIP text encoder key 'text_model\.encoder\.layers\.2\."):
        load_clip_text_encoder(small_files[1], "cpu", cfg=_small_cfg(num_hidden_layers=3))
    with pytest.raises(FileNotFoundError, match="CLIP text encoder"):
        load_clip_text_encoder(str(tmp_path / "absent.pt"), "cpu", cfg=_small_cfg())


# ------------------------------------------------------------------ host model with emulated kernels
def attention_causal(q, k, v, heads, scale=None, out=None):
    """The contract of mvoc_attn_causal_fwd: one [B, N, H*64] shape, views with a contiguous last dim and 16-byte
    strides; query row r attends to keys 0..r."""
    assert q.shape == k.shape == v.shape
    for t in (q, k, v):
        assert t.dim() == 3 and t.shape[-1] == heads * 64 and t.stride(-1) == 1
        assert all(s % 8 == 0 for s in t.stride()[:-1])
    B, N, C = q.shape
    sp = lambda t: t.reshape(B, N, heads, 64).transpose(1, 2)
    o = F.scaled_dot_product_attention(sp(q), sp(k), sp(v), scale=scale, is_causal=True)
    return o.transpose(1, 2).reshape(B, N, C)


def linear_gelu(x, weight, bias=None, out=None, variant=None):
    n, k = weight.shape
    assert n % 64 == 0 and k % 64 == 0 and weight.is_contiguous() and x.stride(-1) == 1
    return F.gelu(F.linear(x, weight, bias))


@pytest.fixture()
def emulated_ops():
    from mvoc_b200 import ops

    saved = emu.install()
    extra = {n: getattr(ops, n) for n in ("attention_causal", "linear_gelu")}
    ops.attention_causal, ops.linear_gelu = attention_causal, linear_gelu
    yield
    for n, f in extra.items():
        setattr(ops, n, f)
    emu.uninstall(saved)


def _small_pair(seed=0):
    from mvoc_b200.clip_text import CLIPTextEncoder

    torch.manual_seed(seed)
    ref = _hf_model(**SMALL)
    ours = CLIPTextEncoder(_small_cfg()).eval()
    ours.load_state_dict(ref.state_dict(), strict=True)
    return ref, ours


def test_host_model_vs_transformers(emulated_ops):
    ref, ours = _small_pair()
    ids = torch.randint(0, SMALL["vocab_size"], (3, 77), generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        want = ref(input_ids=ids).last_hidden_state
        got = ours(ids)
        short = ours(ids[:, :20])                    # a shorter sequence: the causal rows do not see the tail
    assert got.shape == want.shape == (3, 77, 256)
    err = float((got - want).norm() / want.norm())
    assert err <= 1e-5, err
    assert torch.allclose(short, got[:, :20], rtol=1e-5, atol=1e-5)


def test_encode_prompt_needs_both_halves_and_chunks(emulated_ops, tmp_path):
    from mvoc_b200.pipeline import I2VGenXLPipeline

    tok = _tokenizer(tmp_path, "!")
    _, ours = _small_pair()
    with pytest.raises(RuntimeError, match="text encoder"):
        I2VGenXLPipeline(None, "cpu", text_encoder=ours).encode_prompt(["a"])
    pipe = I2VGenXLPipeline(None, "cpu", text_encoder=ours, tokenizer=tok)
    prompts = ["a boat", None, "the surfer", "", "blurry"]
    a, b = pipe.encode_prompt(prompts, encode_chunk_size=2), pipe.encode_prompt(prompts, encode_chunk_size=5)
    assert a.shape == (5, 77, 256)
    assert torch.allclose(a, b, rtol=1e-4, atol=1e-5)      # CPU GEMMs of other row counts (the GPU test: bits)
    assert torch.equal(pipe.encode_prompt(None), pipe.encode_prompt([""]))
    with torch.no_grad():
        assert torch.allclose(a, ours(tok(["a boat", "", "the surfer", "", "blurry"])), rtol=1e-4, atol=1e-5)


# ------------------------------------------------------------------ tokenizer
CORPUS = ("a boat and a surfer on the sea it's the blurry sky over the boats café naïve surfing surfers they'll "
          "photo of 1 dog running").split() * 3
CASES = [
    "",                                                         # empty prompt
    "a boat and a surfer on the sea",
    "Hello, World!! (yes) -- ok...",                            # punctuation
    "it's THE boat's sail; they'll've we'd I'M",                # apostrophes and upper case
    "2024 boats, 3.14 and 10,000",                              # digits (one per token)
    "café naïve Ünïcödé cafe\u0301",                            # accents, precomposed and combining (NFC)
    "  many   spaces\n\nand\tnewlines  \r\n",                   # whitespace runs
    "A BOAT",
    "abc!",                                                     # special-token text: "!" when it is the pad token
    "x<|endoftext|>y <|startoftext|>z",
    "<|ENDOFTEXT|> and <|EndOfText|>",                          # not special (case), split by the byte-level regex
    "emoji 🏄 and 中文",
    " ".join(["surfer"] * 80),                                  # longer than 75 tokens: truncated
    " ".join(str(i % 10) for i in range(120)),
]


def _learn_merges(corpus, n_merges):
    """A few BPE merges learned on `corpus` (byte-level symbols, </w> word ends), most frequent pair first."""
    from mvoc_b200.clip_text import _bytes_to_unicode

    bt = _bytes_to_unicode()
    words = collections.Counter()
    for w in corpus:
        s = "".join(bt[b] for b in w.encode())
        words[tuple(s[:-1]) + (s[-1] + "</w>",)] += 1
    merges = []
    for _ in range(n_merges):
        pairs = collections.Counter()
        for w, c in words.items():
            for p in zip(w, w[1:]):
                pairs[p] += c
        if not pairs:
            break
        best = max(pairs, key=lambda p: (pairs[p], p))
        merges.append(best)
        nw = collections.Counter()
        for w, c in words.items():
            out, i = [], 0
            while i < len(w):
                if i + 1 < len(w) and (w[i], w[i + 1]) == best:
                    out.append(w[i] + w[i + 1])
                    i += 2
                else:
                    out.append(w[i])
                    i += 1
            nw[tuple(out)] += c
        words = nw
    return merges


def tiny_vocab():
    """CLIP's vocabulary layout at a small size: the 256 byte symbols ("!" is id 0), the same with </w>, the merges,
    then <|startoftext|> and <|endoftext|>."""
    from mvoc_b200.clip_text import _bytes_to_unicode

    base = list(_bytes_to_unicode().values())
    merges = _learn_merges(CORPUS, 60)
    vocab = {t: i for i, t in enumerate(base + [c + "</w>" for c in base] + [a + b for a, b in merges])}
    vocab["<|startoftext|>"] = len(vocab)
    vocab["<|endoftext|>"] = len(vocab)
    return vocab, merges


def write_tokenizer_dir(path, pad=None, pad_in="tokenizer_config"):
    """A tokenizer/ folder like a diffusers checkpoint's: vocab.json, merges.txt (with its #version line) and the
    special tokens in tokenizer_config.json (AddedToken dicts) and / or special_tokens_map.json (strings)."""
    vocab, merges = tiny_vocab()
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "vocab.json"), "w", encoding="utf-8") as f:
        json.dump(vocab, f, ensure_ascii=False)
    with open(os.path.join(path, "merges.txt"), "w", encoding="utf-8") as f:
        f.write("#version: 0.2\n" + "".join(f"{a} {b}\n" for a, b in merges))
    tok = lambda s: {"__type": "AddedToken", "content": s, "lstrip": False, "normalized": True, "rstrip": False,
                     "single_word": False}
    conf = {"bos_token": tok("<|startoftext|>"), "eos_token": tok("<|endoftext|>"), "unk_token": tok("<|endoftext|>"),
            "model_max_length": 77, "tokenizer_class": "CLIPTokenizer", "do_lower_case": True}
    smap = {"bos_token": "<|startoftext|>", "eos_token": "<|endoftext|>", "unk_token": "<|endoftext|>"}
    if pad is not None and pad_in in ("tokenizer_config", "both"):
        conf["pad_token"] = tok(pad)
    if pad is not None and pad_in in ("special_tokens_map", "both"):
        smap["pad_token"] = pad
    with open(os.path.join(path, "tokenizer_config.json"), "w") as f:
        json.dump(conf, f)
    with open(os.path.join(path, "special_tokens_map.json"), "w") as f:
        json.dump(smap, f)
    return vocab, merges


def _tokenizer(tmp_path, pad):
    from mvoc_b200.clip_text import CLIPTokenizer

    write_tokenizer_dir(str(tmp_path / "tokenizer"), pad)
    return CLIPTokenizer.from_dir(str(tmp_path / "tokenizer"))


def _reference_ids(vocab, merges, pad, prompts):
    transformers = pytest.importorskip("transformers")
    ref = transformers.CLIPTokenizer(vocab=dict(vocab), merges=[tuple(m) for m in merges], pad_token=pad)
    return ref(prompts, padding="max_length", max_length=77, truncation=True).input_ids


@pytest.mark.parametrize("pad", ["!", "<|endoftext|>"])
def test_tokenizer_matches_transformers(pad):
    from mvoc_b200.clip_text import CLIPTokenizer

    vocab, merges = tiny_vocab()
    ours = CLIPTokenizer(vocab, [" ".join(m) for m in merges], pad_token=pad)
    got = ours(CASES)
    want = _reference_ids(vocab, merges, pad, CASES)
    assert got.shape == (len(CASES), 77) and got.dtype == torch.int64
    for prompt, g, w in zip(CASES, got.tolist(), want):
        assert g == w, f"{prompt!r}: {g} != transformers {w}"
    assert got[0].tolist() == [vocab["<|startoftext|>"], vocab["<|endoftext|>"]] + [vocab[pad]] * 75
    long = got[CASES.index(" ".join(["surfer"] * 80))]
    assert long[-1] == vocab["<|endoftext|>"] and vocab[pad] not in long.tolist()[1:-1]
    bang = ours.encode("abc!")
    assert (bang[-1] == 0) == (pad == "!")         # "!" is split out as the pad token, not encoded as "!</w>"


@pytest.mark.parametrize("pad_in", ["tokenizer_config", "special_tokens_map", "both", "neither"])
def test_tokenizer_folder_reads_the_pad_token(tmp_path, pad_in):
    from mvoc_b200.clip_text import CLIPTokenizer

    path = str(tmp_path / "tokenizer")
    vocab, merges = write_tokenizer_dir(path, "!", pad_in)
    tok = CLIPTokenizer.from_dir(path)
    pad = "<|endoftext|>" if pad_in == "neither" else "!"     # transformers' default when no file names one
    assert tok.pad_token == pad and tok.pad_id == vocab[pad]
    assert tok(CASES).tolist() == _reference_ids(vocab, merges, pad, CASES)
    transformers = pytest.importorskip("transformers")
    assert transformers.CLIPTokenizer.from_pretrained(path).pad_token == pad
    os.remove(os.path.join(path, "merges.txt"))
    with pytest.raises(FileNotFoundError, match="merges.txt"):
        CLIPTokenizer.from_dir(path)


# ------------------------------------------------------------------ the prompt stacks against the golden seams
def _stand_in_encoder(calls):
    from tests.golden import spec

    def encode(prompts):
        calls.append(list(prompts))
        return torch.cat([spec.text_embedding(p) for p in prompts])

    return encode


def test_composition_prompt_stack_is_the_golden_seam():
    """[ddim_inv_prompt x (n+1), negative_prompt, prompt] with spec.text_embedding standing in for the encoder gives
    the encoder_hidden_states the reference's own loop produced, bit for bit; each distinct string is encoded once."""
    from mvoc_b200.clip_text import composition_prompt_embeds, composition_prompts
    from tests.golden import spec

    fx = spec.loop_fixture()
    golden = torch.load(os.path.join(GOLDEN, "composition_loop_tiny4.pt"), map_location="cpu")
    calls = []
    got = composition_prompt_embeds(_stand_in_encoder(calls), fx["n_obj"], fx["prompt"], fx["negative_prompt"],
                                    fx["ddim_inv_prompt"])
    assert torch.equal(got, golden["seam"]["encoder_hidden_states"])
    assert calls == [["", "blurry", "a boat and a surfer on the sea"]]
    assert composition_prompts(2, "p", None, None) == ["", "", "", "", "p"]


def test_inversion_prompt_is_the_golden_seam():
    from mvoc_b200.clip_text import encode_distinct
    from tests.golden import spec

    fx = spec.inversion_fixture()
    golden = torch.load(os.path.join(GOLDEN, "inversion_loop_tiny4.pt"), map_location="cpu")
    got = encode_distinct(_stand_in_encoder([]), [fx["prompt"]])
    assert torch.equal(got, golden["seam"]["encoder_hidden_states"])


# ------------------------------------------------------------------ entry argument checks (no GPU touched)
def test_attn_causal_entry_rejects_bad_arguments():
    from mvoc_b200 import _cabi

    lib = _cabi.load()
    st = [77 * 3072, 3072, 64] * 3 + [77 * 1024, 1024, 64]

    def call(p=16, Nq=77, Nk=77, D=64, dtype=0, strides=st):
        return lib.mvoc_attn_causal_fwd(p, 16, 16, 16, 2, 16, Nq, Nk, D, *strides, 0.125, dtype, None)

    assert call(p=None) == -1 and b"null pointer" in lib.mvoc_last_error()
    assert call(Nk=78) == -2 and b"Nq == Nk" in lib.mvoc_last_error()
    assert call(Nq=128, Nk=77) == -2 and b"Nq=128 Nk=77" in lib.mvoc_last_error()
    assert call(D=80) == -2 and b"head_dim 80" in lib.mvoc_last_error()
    assert call(p=24) == -1 and b"16-byte aligned" in lib.mvoc_last_error()
    assert call(dtype=2) == -2 and b"dtype" in lib.mvoc_last_error()
    assert call(strides=[77 * 3072, 3076, 64] + st[3:]) == -2 and b"multiple of 8" in lib.mvoc_last_error()
    assert call(Nq=0, Nk=0) == -1 and b"empty problem" in lib.mvoc_last_error()
    assert call(strides=st[:4] + [0] + st[5:]) == -2 and b"mvoc_attn_causal_fwd" in lib.mvoc_last_error()


def test_attention_causal_wrapper_needs_cuda_tensors():
    from mvoc_b200 import ops

    x = torch.zeros(1, 4, 128)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.attention_causal(x, x, x, 2)


# ------------------------------------------------------------------ the scripts' text paths
@pytest.mark.parametrize("script", ["inverse", "composite"])
def test_scripts_pair_the_text_flags(script, tmp_path):
    """One of --text_encoder_state_dict / --tokenizer_dir without the other fails before any weights are built."""
    from mvoc_b200 import composite, inverse

    main = inverse.main if script == "inverse" else composite.main
    template = os.path.join(ROOT, "configs", f"group_{'inversion' if script == 'inverse' else 'composite'}",
                            "template.yaml")
    for kw in (dict(text_encoder_state_dict=str(tmp_path / "t.pt")), dict(tokenizer_dir=str(tmp_path))):
        with pytest.raises(ValueError, match="--text_encoder_state_dict and --tokenizer_dir go together"):
            main(template, str(tmp_path / "absent.json"), synthetic_inputs=True, device="cpu", **kw)
    for flag in ("--text_encoder_state_dict", "--tokenizer_dir"):
        mod = inverse if script == "inverse" else composite
        assert getattr(mod.build_parser().parse_args([flag, "x"]), flag[2:]) == "x"


def test_composite_prompts_come_from_the_config(tmp_path, emulated_ops):
    from mvoc_b200 import config as cfgmod
    from mvoc_b200.composite import branch_prompt_embeds
    from mvoc_b200.config import Config
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, ours = _small_pair()
    pipe = I2VGenXLPipeline(None, "cpu", text_encoder=ours, tokenizer=_tokenizer(tmp_path, "!"))
    cfg = Config({"obj_mask_path": ["m0", "m1"], "prompt": "a boat and a surfer", "negative_prompt": "blurry",
                  "ddim_inv_prompt": "the sea"})
    emb = branch_prompt_embeds(pipe, cfg)
    want = pipe.encode_prompt(["the sea", "blurry", "a boat and a surfer"])
    assert emb.shape == (5, 77, 256)
    for i, j in ((0, 0), (1, 0), (2, 0), (3, 1), (4, 2)):
        assert torch.equal(emb[i], want[j])
    # the template's defaults are "" for all three
    template = cfgmod.load_template(os.path.join(ROOT, "configs", "group_composite", "template.yaml"))
    assert (template["prompt"], template["negative_prompt"], template["ddim_inv_prompt"]) == ("", "", "")
    emb = branch_prompt_embeds(pipe, Config({"obj_mask_path": ["m0"], "prompt": "", "negative_prompt": "",
                                             "ddim_inv_prompt": ""}))
    assert emb.shape == (4, 77, 256) and all(torch.equal(emb[i], emb[0]) for i in range(4))


def test_inverse_runs_without_inputs_when_every_key_is_computed(tmp_path, emulated_ops, monkeypatch):
    """With the VAE, image and text flags together inverse.py needs no --inputs file (nor --synthetic); the prompt
    embeddings that reach the loop are encode_prompt(inverse_config.prompt).  The UNet is the reduced configuration
    and the frame encoders are stubbed: this checks the script's wiring, the GPU test runs the towers."""
    from mvoc_b200 import clip_text, inverse, unet3d
    from mvoc_b200.pipeline import I2VGenXLPipeline

    _, ours = _small_pair()
    weights = str(tmp_path / "text_encoder.pt")
    torch.save(ours.state_dict(), weights)
    write_tokenizer_dir(str(tmp_path / "tokenizer"), "!")
    real_load = clip_text.load_clip_text_encoder
    monkeypatch.setattr(clip_text, "load_clip_text_encoder",
                        lambda p, device: real_load(p, device, torch.float32, cfg=_small_cfg()))
    monkeypatch.setattr(unet3d.UNetConfig, "full", staticmethod(unet3d.UNetConfig.reduced))
    unet_weights = str(tmp_path / "unet.pt")
    torch.save(unet3d.I2VGenXLUNet(unet3d.UNetConfig.reduced()).state_dict(), unet_weights)
    monkeypatch.setattr("mvoc_b200.vae.load_vae_encoder", lambda p, device: object())
    monkeypatch.setattr("mvoc_b200.clip.load_clip_image_encoder", lambda p, device: object())
    lat = torch.zeros(1, 4, 2, 8, 8)
    monkeypatch.setattr(inverse, "encode_entry", lambda pipe, config, idx, syn, device: (lat, lat))
    monkeypatch.setattr(inverse, "image_embeddings_entry", lambda pipe, config, idx, syn: torch.zeros(1, 1, 1024))
    seen = {}

    def record(self, latents, prompt_embeds, image_embeddings, image_latents, fps, **kw):
        seen.update(pipe=self, prompt_embeds=prompt_embeds)
        return {}

    monkeypatch.setattr(I2VGenXLPipeline, "invert", record)
    cfg = tmp_path / "group.json"
    cfg.write_text(json.dumps([{"active": True, "force_recompute_latents": True, "video_name": "clip",
                                "data_dir": str(tmp_path), "image_size": [64, 64], "n_frames": 2,
                                "inverse_config": {"prompt": "a boat and a surfer"}}]))
    template = os.path.join(ROOT, "configs", "group_inversion", "template.yaml")
    assert inverse.main(template, str(cfg), unet_weights, device="cpu", vae_state_dict="vae",
                        image_encoder_state_dict="clip", text_encoder_state_dict=weights,
                        tokenizer_dir=str(tmp_path / "tokenizer")) == 1
    pipe = seen["pipe"]
    want = pipe.encode_prompt(["a boat and a surfer"])
    assert seen["prompt_embeds"].shape == (1, 77, 256)
    assert torch.equal(seen["prompt_embeds"], want.to(seen["prompt_embeds"].dtype))
    # without the text flags the same call still needs --inputs
    with pytest.raises(FileNotFoundError, match="--inputs"):
        inverse.main(template, str(cfg), unet_weights, device="cpu", vae_state_dict="vae",
                     image_encoder_state_dict="clip")
