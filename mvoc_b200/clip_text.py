"""CLIP text tower, product side: prompts -> prompt embeddings on the library's kernels (bf16 on one B200).

The module tree and parameter names are those of transformers' ``CLIPTextModel`` (the reference's ``text_encoder/``
folder: vocabulary 49408, width 1024, 16 heads of 64, MLP 4096, 77 positions), so its state dict loads unchanged.  The
reference calls it from ``I2VGenXLPipeline.encode_prompt`` (diffusers 0.27.2) with ``clip_skip=None`` and no attention
mask: the output is ``last_hidden_state`` after ``final_layer_norm`` at all 77 positions, pad positions included.

Per encoder layer the image tower's layer runs (mvoc_b200.clip.CLIPEncoderLayer) with the causal attention
``mvoc_attn_causal_fwd`` in place of the dense head_dim-80 one: ``mvoc_layernorm``, one fused q/k/v ``mvoc_linear``,
causal attention on the three column slices, ``out_proj`` with the residual in the epilogue, ``mvoc_layernorm``,
``fc1`` with the exact GELU in the epilogue, ``fc2`` with the residual in the epilogue.  The token gather and the
position add are torch ops; ``final_layer_norm`` is ``mvoc_layernorm`` on every token.  Nothing on this path goes to
cuDNN or cuBLAS.

``CLIPTokenizer`` reads the checkpoint's ``tokenizer/`` folder (``vocab.json``, ``merges.txt``,
``tokenizer_config.json`` / ``special_tokens_map.json``) and produces the ids of transformers' ``CLIPTokenizer``
(transformers 5.5, tokenizers backend) with ``padding="max_length", max_length=77, truncation=True``.
"""
from __future__ import annotations

import json
import os
import unicodedata
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence

import regex
import torch
import torch.nn as nn

from . import ops
from .clip import CLIPEncoder, _layernorm


@dataclass
class CLIPTextConfig:
    """The reference checkpoint's CLIPTextConfig (text_encoder/config.json of i2vgen-xl); LayerNorm eps 1e-5 and the
    erf GELU (hidden_act "gelu") are fixed.  The layer count 23 is the published config's value as recalled, not read
    from a checkpoint: the loader rejects a checkpoint with another count and names the first key that differs."""
    vocab_size: int = 49408
    hidden_size: int = 1024
    intermediate_size: int = 4096
    num_hidden_layers: int = 23
    num_attention_heads: int = 16
    max_position_embeddings: int = 77
    layer_norm_eps: float = 1e-5


class CLIPTextEmbeddings(nn.Module):
    def __init__(self, cfg: CLIPTextConfig):
        super().__init__()
        self.token_embedding = nn.Embedding(cfg.vocab_size, cfg.hidden_size)
        self.position_embedding = nn.Embedding(cfg.max_position_embeddings, cfg.hidden_size)

    def forward(self, input_ids: torch.Tensor) -> torch.Tensor:
        n = input_ids.shape[1]
        return self.token_embedding.weight[input_ids] + self.position_embedding.weight[:n]


class CLIPTextTransformer(nn.Module):
    def __init__(self, cfg: CLIPTextConfig):
        super().__init__()
        self.embeddings = CLIPTextEmbeddings(cfg)
        self.encoder = CLIPEncoder(cfg, causal=True)
        self.final_layer_norm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)


class CLIPTextEncoder(nn.Module):
    """transformers' CLIPTextModel (same module tree and state-dict names): input_ids [n, N <= 77] (int64) ->
    last_hidden_state [n, N, hidden_size] in the weights' dtype."""

    def __init__(self, cfg: CLIPTextConfig = None):
        super().__init__()
        self.cfg = cfg or CLIPTextConfig()
        self.text_model = CLIPTextTransformer(self.cfg)

    @property
    def dtype(self):
        return self.text_model.final_layer_norm.weight.dtype

    def forward(self, input_ids: torch.Tensor) -> torch.Tensor:
        tm = self.text_model
        if input_ids.dim() != 2 or input_ids.shape[1] > self.cfg.max_position_embeddings:
            raise ValueError(f"CLIP text tower: input_ids must be [n, <= {self.cfg.max_position_embeddings}], got "
                             f"{tuple(input_ids.shape)}")
        x = tm.embeddings(input_ids.to(tm.embeddings.token_embedding.weight.device))
        for layer in tm.encoder.layers:
            x = layer(x)
        return _layernorm(tm.final_layer_norm, x)


# keys of a full CLIPModel / older transformers checkpoints that the text tower does not use
_IGNORED = ("vision_model.", "visual_projection.", "text_projection.", "logit_scale",
            "text_model.embeddings.position_ids")


def load_clip_text_encoder(path: str, device, dtype=torch.bfloat16, cfg: CLIPTextConfig = None) -> CLIPTextEncoder:
    """CLIP text tower from a transformers ``CLIPTextModel`` state dict (``.safetensors`` or a torch file):
    ``text_model.*``.  The image tower's and the projections' keys and the position_ids buffer of older checkpoints are
    ignored; a missing or unexpected key, or a tensor of the wrong shape, raises an error that names it.  `cfg`
    defaults to the reference checkpoint's configuration."""
    from .vae import _load_part

    return _load_part(path, lambda: CLIPTextEncoder(cfg), "CLIP text encoder", _IGNORED, device, dtype,
                      kind="CLIP text encoder")


def check_text_flags(text_encoder_state_dict: Optional[str], tokenizer_dir: Optional[str]) -> None:
    """The scripts' --text_encoder_state_dict and --tokenizer_dir go together."""
    if (text_encoder_state_dict is None) != (tokenizer_dir is None):
        raise ValueError("--text_encoder_state_dict and --tokenizer_dir go together: the text tower needs both the "
                         "weights and the checkpoint's tokenizer/ folder")


def load_text_tower(text_encoder_state_dict: Optional[str], tokenizer_dir: Optional[str], device):
    """(CLIPTextEncoder, CLIPTokenizer) from the scripts' two flags, or (None, None) when neither is given."""
    check_text_flags(text_encoder_state_dict, tokenizer_dir)
    if text_encoder_state_dict is None:
        return None, None
    return load_clip_text_encoder(text_encoder_state_dict, device), CLIPTokenizer.from_dir(tokenizer_dir)


# ------------------------------------------------------------------ tokenizer
# CLIP's pre-tokenizer split (transformers' CLIPTokenizer): the two special strings, contractions, letter runs, single
# digits, runs of anything else but whitespace
_SPLIT = regex.compile(r"""<\|startoftext\|>|<\|endoftext\|>|'s|'t|'re|'ve|'m|'ll|'d|[\p{L}]+|[\p{N}]|[^\s\p{L}\p{N}]+""")
# then byte-level BPE's GPT-2 split inside each piece (of CLIP's pieces it only splits the two special strings, which
# reach it when the prompt spells them in another case)
_SPLIT_BYTE_LEVEL = regex.compile(r"""'s|'t|'re|'ve|'m|'ll|'d| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+""")
_SPACES = regex.compile(r"\s+")


def _bytes_to_unicode() -> Dict[int, str]:
    """GPT-2's byte -> printable character table of byte-level BPE."""
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(ord("¡"), ord("¬") + 1)) + list(range(ord("®"), ord("ÿ") + 1))
    cs = bs[:]
    n = 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    return dict(zip(bs, (chr(c) for c in cs)))


class CLIPTokenizer:
    """Byte-level BPE of CLIP with ``</w>`` word ends.  ``tokenizer(prompts)`` gives what transformers'
    ``CLIPTokenizer(prompts, padding="max_length", max_length=77, truncation=True).input_ids`` gives on the same files:
    special-token strings in the text are split out first (longest first, as written); every other piece is NFC
    normalised, whitespace runs collapse to one space, lower-cased, split by CLIP's regex and then by byte-level BPE's
    GPT-2 regex; each piece is encoded as UTF-8 bytes through the byte table, merged by rank and looked up (unknown
    symbols become the unk token).  The ids are truncated to BOS + max_length-2 + EOS and right-padded with the pad
    token.  ftfy's mojibake repair (transformers' slow tokenizer, when ftfy is installed) is not applied; transformers
    5.5's tokenizer does not apply it either."""

    DEFAULTS = dict(bos_token="<|startoftext|>", eos_token="<|endoftext|>", unk_token="<|endoftext|>",
                    pad_token="<|endoftext|>")   # transformers' CLIPTokenizer defaults

    def __init__(self, vocab: Dict[str, int], merges: Sequence[str], model_max_length: int = 77, **special):
        self.vocab = dict(vocab)
        self.ranks = {}
        for i, m in enumerate(merges):
            a, b = m.split()
            self.ranks[(a, b)] = i
        self.model_max_length = int(model_max_length)
        tokens = {**self.DEFAULTS, **{k: v for k, v in special.items() if v is not None}}
        for name, tok in tokens.items():
            if tok not in self.vocab:
                raise KeyError(f"CLIP tokenizer: {name} {tok!r} is not in the vocabulary")
            setattr(self, name, tok)
        self.bos_id, self.eos_id = self.vocab[self.bos_token], self.vocab[self.eos_token]
        self.unk_id, self.pad_id = self.vocab[self.unk_token], self.vocab[self.pad_token]
        specials = sorted(set(tokens.values()), key=len, reverse=True)
        self._special = regex.compile("(" + "|".join(regex.escape(t) for t in specials) + ")")
        self._byte = _bytes_to_unicode()
        self._cache: Dict[str, List[str]] = {}

    @classmethod
    def from_dir(cls, path: str) -> "CLIPTokenizer":
        """A checkpoint's ``tokenizer/`` folder: vocab.json, merges.txt and the special tokens (bos / eos / unk / pad)
        and model_max_length of tokenizer_config.json, overridden by special_tokens_map.json where both name one;
        a token neither file names takes transformers' default."""
        for name in ("vocab.json", "merges.txt"):
            if not os.path.isfile(os.path.join(path, name)):
                raise FileNotFoundError(f"CLIP tokenizer: {os.path.join(path, name)!r} not found")
        with open(os.path.join(path, "vocab.json"), encoding="utf-8") as f:
            vocab = json.load(f)
        with open(os.path.join(path, "merges.txt"), encoding="utf-8") as f:
            merges = [ln for ln in f.read().split("\n") if ln.strip() and not ln.startswith("#version")]
        kw = {}
        for name in ("tokenizer_config.json", "special_tokens_map.json"):
            p = os.path.join(path, name)
            if not os.path.isfile(p):
                continue
            with open(p, encoding="utf-8") as f:
                conf = json.load(f)
            for key in cls.DEFAULTS:
                if key in conf and conf[key] is not None:
                    v = conf[key]
                    kw[key] = v["content"] if isinstance(v, dict) else v
            if "model_max_length" in conf:
                kw["model_max_length"] = conf["model_max_length"]
        return cls(vocab, merges, **kw)

    def _bpe(self, word: str) -> List[str]:
        if word in self._cache:
            return self._cache[word]
        parts = list(word[:-1]) + [word[-1] + "</w>"]
        while len(parts) > 1:
            rank, i = min((self.ranks.get(p, float("inf")), i) for i, p in enumerate(zip(parts, parts[1:])))
            if rank == float("inf"):
                break
            a, b = parts[i], parts[i + 1]
            merged, j = [], 0
            while j < len(parts):
                if j + 1 < len(parts) and parts[j] == a and parts[j + 1] == b:
                    merged.append(a + b)
                    j += 2
                else:
                    merged.append(parts[j])
                    j += 1
            parts = merged
        self._cache[word] = parts
        return parts

    def encode(self, text: str) -> List[int]:
        """Token ids of `text` without BOS / EOS, truncation or padding."""
        ids = []
        for k, piece in enumerate(self._special.split(text)):
            if k % 2:                                   # a special-token string
                ids.append(self.vocab[piece])
                continue
            piece = _SPACES.sub(" ", unicodedata.normalize("NFC", piece)).strip().lower()
            for word in (w for p in _SPLIT.findall(piece) for w in _SPLIT_BYTE_LEVEL.findall(p)):
                sym = "".join(self._byte[b] for b in word.encode("utf-8"))
                ids.extend(self.vocab.get(t, self.unk_id) for t in self._bpe(sym))
        return ids

    def __call__(self, prompts) -> torch.Tensor:
        """One prompt or a list -> input_ids [n, model_max_length] int64."""
        prompts = [prompts] if isinstance(prompts, str) else list(prompts)
        n = self.model_max_length
        rows = []
        for p in prompts:
            ids = [self.bos_id] + self.encode(p)[:n - 2] + [self.eos_id]
            rows.append(ids + [self.pad_id] * (n - len(ids)))
        return torch.tensor(rows, dtype=torch.int64).view(len(rows), n)


# ------------------------------------------------------------------ the composition's prompt stack
def composition_prompts(n_obj: int, prompt: str, negative_prompt: Optional[str] = None,
                        ddim_inv_prompt: Optional[str] = None) -> List[str]:
    """The prompts of a composition's n_obj + 3 branches (SURVEY Appendix B #9): the inversion prompt for the
    background and every object, then the negative prompt (uncond composite), then the prompt (cond composite).
    None becomes "", as in encode_prompt."""
    inv = ddim_inv_prompt or ""
    return [inv] * (n_obj + 1) + [negative_prompt or "", prompt or ""]


def encode_distinct(encode: Callable[[List[str]], torch.Tensor], prompts: Sequence[str]) -> torch.Tensor:
    """encode(prompts) with every distinct string encoded once: encode(distinct) [k, ...] gathered back to
    [len(prompts), ...] (the rows are copies, bit for bit)."""
    distinct = list(dict.fromkeys(prompts))
    emb = encode(distinct)
    return emb[torch.tensor([distinct.index(p) for p in prompts], device=emb.device)]


def composition_prompt_embeds(encode: Callable[[List[str]], torch.Tensor], n_obj: int, prompt: str,
                              negative_prompt: Optional[str] = None, ddim_inv_prompt: Optional[str] = None):
    """prompt_embeds [n_obj + 3, ...] of a composition, in branch order [inv x (n_obj + 1), negative, prompt]."""
    return encode_distinct(encode, composition_prompts(n_obj, prompt, negative_prompt, ddim_inv_prompt))
