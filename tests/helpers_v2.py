"""Test helpers for the 80-mel checkpoints (large-v2, distil-large-v2, medium, small, base): the v2 special-token layout,
seeded weight variants with 80 mel bins, a synthetic v2-layout tokenizer and the 80-bin log-mel reference.
No dependency on transformers at import time (the GPU box tests must not need HF model classes)."""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

import helpers
from oracle import logmel_ref as L
from oracle import whisper_ref as R

# helpers.TINY widths with the 80-mel front end and the 51865-id vocabulary
TINY_V2 = dict(helpers.TINY, n_mels=80, vocab=51865)
N_MELS = 80

# generation_config.json layout of openai/whisper-large-v2 and older multilingual checkpoints: the large-v3 layout
# without <|yue|> (50358 there), so every special from <|translate|> on sits one id lower
EOS, SOT = 50257, 50258
LANG_FIRST, LANG_LAST = 50259, 50357
TRANSLATE, TRANSCRIBE = 50358, 50359
NO_TIMESTAMPS = 50363
TIMESTAMP_BEGIN = 50364
VOCAB = 51865
# the large-v3 list with its last five ids (translate, transcribe, startoflm, startofprev, nospeech) shifted down
SUPPRESS_TOKENS = R.SUPPRESS_TOKENS[:-5] + [50358, 50359, 50360, 50361, 50362]
BEGIN_SUPPRESS_TOKENS = [220, 50257]


def languages():
    from transformers.models.whisper.tokenization_whisper import LANGUAGES
    return [l for l in LANGUAGES if l != "yue"]


def ref_dims() -> R.WhisperDims:
    return R.WhisperDims(**TINY_V2)


def gen_config() -> R.GenConfig:
    """Oracle settings with the v2 ids."""
    return R.GenConfig(no_timestamps_token_id=NO_TIMESTAMPS, suppress_tokens=list(SUPPRESS_TOKENS),
                       begin_suppress_tokens=list(BEGIN_SUPPRESS_TOKENS),
                       lang_ids=list(range(LANG_FIRST, LANG_LAST + 1)),
                       task_to_id={"transcribe": TRANSCRIBE, "translate": TRANSLATE})


def generation_settings():
    """The engine's GenerationSettings with the v2 ids (what GenerationSettings.from_hf reads from a v2 checkpoint)."""
    from turbo_whisper_workspace_b200.config import GenerationSettings
    return GenerationSettings(no_timestamps_token_id=NO_TIMESTAMPS, suppress_tokens=list(SUPPRESS_TOKENS),
                              begin_suppress_tokens=list(BEGIN_SUPPRESS_TOKENS), lang_first=LANG_FIRST,
                              lang_last=LANG_LAST, task_to_id={"transcribe": TRANSCRIBE, "translate": TRANSLATE})


def variant_state_dict(dims, variant: str, seed: int = 0) -> Dict[str, torch.Tensor]:
    """helpers.variant_state_dict for the v2 layout: the timestamp boost starts at <|0.00|> = 50364."""
    emb_scale, ts_boost = {"decisive": (0.2, 0.6), "varied": (0.1, 0.3)}[variant]
    sd = helpers.random_state_dict(dims, seed, "unit")
    E = sd["model.decoder.embed_tokens.weight"]
    E.mul_(emb_scale / 0.5)
    g = torch.Generator().manual_seed(seed + 1)
    d = torch.randn(dims.d_model, generator=g)
    d /= d.norm()
    E[TIMESTAMP_BEGIN:] += ts_boost * d
    sd["model.decoder.layer_norm.bias"] = sd["model.decoder.layer_norm.bias"] + 2.0 * d
    return sd


def build_tokenizer():
    """Synthetic WhisperTokenizer with the v2 id layout (51865 ids): as helpers.build_tokenizer() without <|yue|>."""
    from transformers import WhisperTokenizer

    bs = list(range(33, 127)) + list(range(161, 173)) + list(range(174, 256))
    cs = bs[:]
    n = 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    b2u = dict(zip(bs, map(chr, cs)))
    vocab = {}
    for b in range(256):
        vocab[b2u[b]] = len(vocab)
    i = 0
    while len(vocab) < 50257:
        s = "".join(b2u[ord(c)] for c in f"w{i}")
        vocab.setdefault(s, len(vocab))
        i += 1
    tok = WhisperTokenizer(vocab=vocab, merges=[])
    tok.add_special_tokens({"additional_special_tokens": ["<|startoftranscript|>"] + [f"<|{l}|>" for l in languages()] +
                            ["<|translate|>", "<|transcribe|>", "<|startoflm|>", "<|startofprev|>", "<|nospeech|>",
                             "<|notimestamps|>"]})
    tok.add_tokens(["<|%.2f|>" % (k * 0.02) for k in range(1501)])
    tok.pad_token = "<|endoftext|>"
    assert len(tok) == VOCAB and tok.convert_tokens_to_ids("<|notimestamps|>") == NO_TIMESTAMPS
    assert tok.convert_tokens_to_ids("<|0.00|>") == TIMESTAMP_BEGIN
    return tok


def hf_generation_config(**overrides):
    """A transformers GenerationConfig with the v2 fields, as a multilingual v2 checkpoint ships it."""
    from transformers import GenerationConfig
    kw = dict(begin_suppress_tokens=list(BEGIN_SUPPRESS_TOKENS), suppress_tokens=list(SUPPRESS_TOKENS),
              max_initial_timestamp_index=50, max_length=448, is_multilingual=True, no_timestamps_token_id=NO_TIMESTAMPS,
              lang_to_id={f"<|{l}|>": LANG_FIRST + i for i, l in enumerate(languages())},
              task_to_id={"transcribe": TRANSCRIBE, "translate": TRANSLATE}, return_timestamps=False, pad_token_id=EOS,
              bos_token_id=EOS, eos_token_id=EOS, decoder_start_token_id=SOT)
    kw.update(overrides)
    return GenerationConfig(**kw)


def hf_model(variant: str):
    """Random tiny 80-mel WhisperForConditionalGeneration with the v2 vocabulary and generation config."""
    from transformers import WhisperConfig, WhisperForConditionalGeneration
    T = helpers.TINY
    cfg = WhisperConfig(vocab_size=VOCAB, num_mel_bins=N_MELS, d_model=T["d_model"], encoder_layers=T["enc_layers"],
                        decoder_layers=T["dec_layers"], encoder_attention_heads=T["heads"],
                        decoder_attention_heads=T["heads"], encoder_ffn_dim=T["ffn"], decoder_ffn_dim=T["ffn"],
                        max_source_positions=1500, max_target_positions=448, pad_token_id=EOS, bos_token_id=EOS,
                        eos_token_id=EOS, decoder_start_token_id=SOT)
    model = WhisperForConditionalGeneration(cfg).eval()
    sd = variant_state_dict(ref_dims(), variant)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all("proj_out" in m for m in missing), (missing, unexpected)
    model.tie_weights()
    model.generation_config = hf_generation_config()
    return model, sd


# ---------------------------------------------------------------------------------------------- 80-bin log-mel
def log_mel(pcm: np.ndarray, n_mels: int = N_MELS) -> np.ndarray:
    """oracle.logmel_ref.log_mel with an n_mels filterbank: [n_mels, 3000] fp32 features of one clip of <= 30 s."""
    x, _ = L.pad_or_trim(pcm)
    xp = np.pad(x, (L.N_FFT // 2, L.N_FFT // 2), mode="reflect")
    n_frames = 1 + (len(xp) - L.N_FFT) // L.HOP
    idx = np.arange(L.N_FFT)[None, :] + L.HOP * np.arange(n_frames)[:, None]
    frames = xp[idx] * L.hann_periodic().astype(np.float32)[None, :]
    power = (np.abs(np.fft.rfft(frames.astype(np.float32), axis=1)) ** 2).astype(np.float32)[:-1]
    logspec = np.log10(np.maximum(power @ L.mel_filter_bank(n_mels=n_mels).astype(np.float32), 1e-10)).T
    logspec = np.maximum(logspec, logspec.max() - 8.0)
    return ((logspec + 4.0) / 4.0).astype(np.float32)


def log_mel_long(pcm: np.ndarray, n_mels: int = N_MELS) -> np.ndarray:
    """oracle.logmel_ref.log_mel_long with an n_mels filterbank: [n_mels, n // 160] features of a clip > 30 s."""
    x = np.asarray(pcm, dtype=np.float32).reshape(-1)
    xp = np.pad(x, (L.N_FFT // 2, L.N_FFT // 2), mode="reflect")
    n_frames = 1 + (len(xp) - L.N_FFT) // L.HOP
    win = L.hann_periodic().astype(np.float32)[None, :]
    fb = L.mel_filter_bank(n_mels=n_mels).astype(np.float32)
    out = np.empty((n_mels, n_frames - 1), dtype=np.float32)
    for f0 in range(0, n_frames - 1, 4096):
        f1 = min(n_frames - 1, f0 + 4096)
        idx = np.arange(L.N_FFT)[None, :] + L.HOP * np.arange(f0, f1)[:, None]
        power = (np.abs(np.fft.rfft((xp[idx] * win).astype(np.float32), axis=1)) ** 2).astype(np.float32)
        out[:, f0:f1] = np.log10(np.maximum(power @ fb, 1e-10)).T
    out = np.maximum(out, out.max() - 8.0)
    return ((out + 4.0) / 4.0).astype(np.float32)
