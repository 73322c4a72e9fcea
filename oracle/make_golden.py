"""Generate tests/golden/* by running the REFERENCE ITSELF (needs a checkout of the reference, see oracle/ref_import.py).

    python -m oracle.make_golden [generator ...]      # default: all of them

Inputs are the seeded synthetic weights/prompts of chattts_b200.synth / .prompts (identical on
every box); outputs are what the reference's own ``GPT.generate`` / ``DVAE`` / host classes produce on
them with stubs for the three absent third-party packages (oracle/ref_import.py).  The tests
load these files, so they do not need the reference at run time.
"""
from __future__ import annotations

import json
import os
import pathlib
import sys

import numpy as np
import torch

from chattts_b200.config import Config
from chattts_b200.prompts import synth_prompt_batch
from chattts_b200.synth import synth_dvae_state, synth_embed_state, synth_gpt_state
from oracle.ref_models import build_reference_dvae, build_reference_gpt, reference_generate

TESTS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests")
OUT = os.path.join(TESTS, "golden")


def _sample(t: torch.Tensor, n: int, seed: int):
    """A fixed, seeded sample of ``n`` elements of ``t`` as (flat indices, values): keeps large outputs small on disk."""
    flat = t.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return idx.numpy().astype(np.int32), flat[idx].numpy()


GPT_CASES = {
    # name: (lengths, prompt_seed, sampler_seed, steps, kwargs)
    "gpt_audio_b1": ([16], 1, 1234, 24, {}),
    "gpt_audio_b3_ragged": ([5, 12, 9], 1, 42, 16, {}),
    "gpt_audio_b2_nopenalty_topk5": ([8, 8], 2, 7, 12, dict(repetition_penalty=1.0, top_K=5, top_P=0.9)),
    "gpt_text_b2": ([7, 4], 3, 7, 8, dict(text=True)),
}


def gen_gpt():
    gs, es = synth_gpt_state(0), synth_embed_state(1)
    gpt, embed = build_reference_gpt(gs, es)
    for name, (lengths, pseed, sseed, steps, kw) in GPT_CASES.items():
        ids, mask, tmask = synth_prompt_batch(lengths, seed=pseed)
        if kw.get("text"):
            ref = reference_generate(gpt, embed, ids, mask, tmask, temperature=[0.7], eos_token=21001,
                                     max_new_token=steps, repetition_penalty=1.0, num_code=21178, infer_text=True,
                                     return_hidden=False, manual_seed=sseed)
            hid = np.zeros((0,), np.float32)
        else:
            ref = reference_generate(gpt, embed, ids, mask, tmask, temperature=[0.3] * 4, eos_token=625,
                                     max_new_token=steps, min_new_token=steps, manual_seed=sseed,
                                     top_P=kw.get("top_P", 0.7), top_K=kw.get("top_K", 20),
                                     repetition_penalty=kw.get("repetition_penalty", 1.05))
            hid = torch.stack([h for h in ref.hiddens]).numpy()
        lens = np.array([len(i) for i in ref.ids])
        pad = np.full((len(lengths), steps, 4), -1, np.int64)
        for b, t in enumerate(ref.ids):
            pad[b, : len(t)] = t.numpy() if t.dim() == 2 else t.numpy()[:, None]
        np.savez_compressed(os.path.join(OUT, name + ".npz"), lengths=np.array(lengths), prompt_seed=pseed,
                            sampler_seed=sseed, steps=steps, ids=pad, n=lens, hiddens=hid.astype(np.float32))
        print(name, lens, pad[0, :2].tolist())


def gen_sampler():
    """Rows of logits pushed through the reference's own processor objects + torch.multinomial."""
    from oracle.ref_import import load_reference

    load_reference()
    from ChatTTS.model import gen_logits

    g = torch.Generator().manual_seed(11)
    rows, V, n_gen = 16, 626, 20
    logits = torch.randn(rows, V, generator=g) * 2.0
    gen_ids = torch.randint(0, 40, (rows, n_gen), generator=g)  # small id range => repeats in the window
    temp = torch.tensor([0.3, 0.5, 0.7, 1.0])
    out = {}
    for tag, (tp, tk, rp) in {"default": (0.7, 20, 1.05), "p95k3": (0.95, 3, 1.2), "nop": (None, 20, 1.0),
                              "nok": (0.5, None, 1.05)}.items():
        warp, proc = gen_logits(num_code=625, top_P=tp, top_K=tk, repetition_penalty=rp)
        x = logits / temp.repeat(rows // 4)[:, None]
        for pr in (*proc, *warp):
            x = pr(gen_ids, x)
        scores = torch.softmax(x, -1)
        idx = torch.multinomial(scores, 1, generator=torch.Generator().manual_seed(99))
        out["idx_" + tag] = idx[:, 0].numpy()
        out["keep_" + tag] = torch.isfinite(x).numpy()
    np.savez_compressed(os.path.join(OUT, "sampler_rows.npz"), logits=logits.numpy(), gen_ids=gen_ids.numpy(),
                        temperature=temp.numpy(), seed=99, **out)
    print("sampler", {k: v[:6].tolist() for k, v in out.items() if k.startswith("idx")})


def gen_dvae():
    cfg = Config()
    st = synth_dvae_state(2, cfg.decoder, cfg.decoder.idim)
    ref = build_reference_dvae(st, cfg.decoder, cfg.decoder.idim)
    g = torch.Generator().manual_seed(21)
    x = torch.randn(2, 768, 12, generator=g)
    with torch.no_grad():
        mel = ref(x.clone(), "decode")
    np.savez_compressed(os.path.join(OUT, "dvae_decoder_hidden.npz"), x=x.numpy(), mel=mel.numpy())
    print("dvae", mel.shape, float(mel.abs().mean()))


def gen_dvae_encode():
    """Encode branch: mel and encoder output from the REFERENCE's modules (torchaudio mel, downsample convs, encoder
    stack); ids / margins from the oracle's FSQ restatement applied to the reference's encoder output (third-party
    quantiser absent - parity unpinned for that last step)."""
    from chattts_b200.synth import synth_speech_like
    from oracle.dvae_oracle import fsq_quantize
    from oracle.ref_models import build_reference_dvae_encoder

    cfg = Config()
    st = synth_dvae_state(3, cfg.dvae.decoder, cfg.dvae.decoder.idim, cfg.dvae.vq, encoder=cfg.dvae.encoder)
    ref = build_reference_dvae_encoder(st, cfg.dvae.decoder, cfg.dvae.encoder, cfg.dvae.decoder.idim)
    seconds, seed = 1.37, 7                      # 32 880 samples: not a multiple of the hop, odd frame count
    wav = synth_speech_like(seconds, seed)
    with torch.inference_mode():
        mel = ref.preprocessor_mel(wav.clone())
        mel = mel / ref.coef.view(100, 1)
        x = ref.encoder(ref.downsample_conv(mel).unsqueeze(0))
    ids, margin = fsq_quantize(x.transpose(1, 2).clone(), st)
    np.savez_compressed(os.path.join(OUT, "dvae_encode.npz"), seconds=seconds, seed=seed, mel_over_coef=mel.numpy(),
                        ids=ids.numpy().astype(np.int32), margin=margin.numpy())
    print("dvae encode", tuple(ids.shape), "frames", mel.shape[1], "min margin", float(margin.min()))


def gen_oracle_pins():
    """What tests/test_oracle_vs_reference.py compares the oracle with: the reference's GPT, Embed, DVAE decode branch and
    encode-side modules on that test's inputs."""
    from chattts_b200.synth import synth_speech_like
    from oracle.ref_models import build_reference_dvae_encoder

    gs, es = synth_gpt_state(0), synth_embed_state(1)
    gpt, embed = build_reference_gpt(gs, es)
    out = {}
    for lengths, seed in (([16], 1234), ([5, 12, 9], 42)):
        ids, mask, tmask = synth_prompt_batch(lengths, seed=1)
        ref = reference_generate(gpt, embed, ids, mask, tmask, temperature=[0.3] * 4, eos_token=625,
                                 max_new_token=12, min_new_token=12, manual_seed=seed)
        out[f"audio_{seed}_ids"] = torch.stack(ref.ids).numpy()
        out[f"audio_{seed}_hid_idx"], out[f"audio_{seed}_hid"] = _sample(torch.stack(ref.hiddens), 2048, seed)
    ids, mask, tmask = synth_prompt_batch([7, 4], seed=3)
    ref = reference_generate(gpt, embed, ids, mask, tmask, temperature=[0.7], eos_token=21001, max_new_token=6,
                             repetition_penalty=1.0, num_code=21178, infer_text=True, return_hidden=False, manual_seed=7)
    out["text_ids"] = np.full((2, 6), -1, np.int64)
    for b, t in enumerate(ref.ids):
        out["text_ids"][b, : len(t)] = t.numpy()
    out["text_n"] = np.array([len(t) for t in ref.ids])
    ids, mask, tmask = synth_prompt_batch([6, 3], seed=5)
    tmask[0, -2:] = False
    ids[0, -2:] = torch.randint(0, 626, (2, 4), generator=torch.Generator().manual_seed(5))
    out["embed_idx"], out["embed"] = _sample(embed(ids, tmask), 2048, 5)

    cfg = Config()
    st = synth_dvae_state(2, cfg.decoder, cfg.decoder.idim)
    x = torch.randn(2, 768, 20, generator=torch.Generator().manual_seed(20))
    with torch.no_grad():
        out["dvae_mel"] = build_reference_dvae(st, cfg.decoder, cfg.decoder.idim)(x, "decode").numpy()

    st = synth_dvae_state(3, cfg.dvae.decoder, cfg.dvae.decoder.idim, cfg.dvae.vq, encoder=cfg.dvae.encoder)
    ref = build_reference_dvae_encoder(st, cfg.dvae.decoder, cfg.dvae.encoder, cfg.dvae.decoder.idim)
    for seconds, seed in ((1.3, 0), (2.0, 1)):
        wav = synth_speech_like(seconds, seed)
        with torch.inference_mode():
            mel = ref.preprocessor_mel(wav.clone())
            enc = ref.encoder(ref.downsample_conv(mel / ref.coef.view(100, 1)).unsqueeze(0))
        out[f"enc{seed}_mel_shape"], out[f"enc{seed}_x_shape"] = np.array(mel.shape), np.array(enc.shape)
        out[f"enc{seed}_mel_idx"], out[f"enc{seed}_mel"] = _sample(mel, 2048, seed)
        out[f"enc{seed}_x_idx"], out[f"enc{seed}_x"] = _sample(enc, 4096, seed)
        out[f"enc{seed}_x_absmax"] = np.float32(enc.abs().max())
    np.savez_compressed(os.path.join(OUT, "reference_oracle.npz"), **out)
    print("oracle pins", sorted(out))


def gen_host_pins():
    """What the host-side tests compare with: the reference's own Normalizer, Speaker and Tokenizer on the inputs those
    tests define (imported from them), and the reference's ``spk_stat`` asset."""
    import tempfile

    from oracle.ref_import import load_reference

    load_reference()
    from ChatTTS.config import Config as RefConfig
    from ChatTTS.model.speaker import Speaker as RefSpeaker
    from ChatTTS.model.tokenizer import Tokenizer as RefTokenizer
    from ChatTTS.norm import Normalizer as RefNormalizer

    sys.path.insert(0, TESTS)
    import test_norm_audio
    import test_speaker
    import test_tokenizer

    js, arrays = {"spk_stat": RefConfig().spk_stat}, {}

    fd, path = tempfile.mkstemp(suffix=".json")
    with os.fdopen(fd, "w", encoding="utf-8") as f:
        json.dump(test_norm_audio.HOMO, f, ensure_ascii=False)
    norm = RefNormalizer(path)
    os.unlink(path)
    assert norm.register("en", lambda s: s.upper())
    js["normalizer"] = [[text, n, h, lang, norm(text, n, h, lang)] for text, n, h, lang in test_norm_audio.normalizer_inputs()]

    ref = object.__new__(RefSpeaker)
    emb, vec, ids = test_speaker.apply_inputs()
    a = ref.apply(emb.clone(), vec, ids, 21143, torch.device("cpu"))
    changed = (a != emb).any(-1)
    arrays["apply_changed"], arrays["apply_rows"] = changed.numpy(), a[changed].numpy()
    js["decorate_code"] = []
    for spk_emb, smp in test_speaker.DECORATE_CASES:
        texts = list(test_speaker.DECORATE_TEXTS)
        js["decorate_code"].append([ref.decorate_code_prompts(texts, "[speed_5]", smp, spk_emb), texts])
    js["decorate_text"] = ref.decorate_text_prompts(["a", "b"], "[oral_2]")

    with tempfile.TemporaryDirectory() as tmp:
        tok = RefTokenizer(test_tokenizer._write_vocab(pathlib.Path(tmp)))
    if not hasattr(tok._tokenizer, "encode_plus"):       # API drift: transformers >= 5 removed encode_plus (same as __call__)
        tok._tokenizer.encode_plus = tok._tokenizer.__call__
    js["tokenizer"] = {"len": tok.len, "spk_emb_ids": tok.spk_emb_ids, "break_0_ids": tok.break_0_ids,
                       "eos_token": tok.eos_token, "decode": tok.decode(test_tokenizer.DECODE_IDS)}
    for tag, prompt in (("noprompt", None), ("prompt", test_tokenizer.PROMPT)):
        for name, t in zip(("ids", "attention_mask", "text_mask"),
                           tok.encode(list(test_tokenizer.TEXTS), 4, prompt=None if prompt is None else prompt.clone())):
            arrays[f"tok_{tag}_{name}"] = t.numpy()

    with open(os.path.join(OUT, "reference_host.json"), "w", encoding="utf-8") as f:
        json.dump(js, f, ensure_ascii=False, indent=0)
        f.write("\n")
    np.savez_compressed(os.path.join(OUT, "reference_host.npz"), **arrays)
    print("host pins", sorted(js), sorted(arrays))


GENERATORS = {f.__name__: f for f in (gen_gpt, gen_sampler, gen_dvae, gen_dvae_encode, gen_oracle_pins, gen_host_pins)}

if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    for name in sys.argv[1:] or GENERATORS:
        GENERATORS[name]()
