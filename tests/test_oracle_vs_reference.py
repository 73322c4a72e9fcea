"""Pin oracle/*_oracle.py against what the reference's own code computed on the same inputs.

The reference outputs are stored in tests/golden/reference_oracle.npz (generator: ``python -m oracle.make_golden
gen_oracle_pins``); large outputs are a fixed, seeded sample of their elements (``<name>_idx`` = flat indices)."""
import os

import numpy as np
import pytest
import torch

from chattts_b200.prompts import synth_prompt_batch
from chattts_b200.synth import synth_embed_state, synth_gpt_state
from oracle.gpt_oracle import GPTOracle, SamplerParams

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_oracle.npz"))


def _sampled(t, name):
    return t.reshape(-1)[torch.from_numpy(GOLD[name + "_idx"]).long()].numpy()


@pytest.fixture(scope="module")
def orc():
    return GPTOracle(synth_gpt_state(0), synth_embed_state(1))


@pytest.mark.parametrize("lengths,seed", [([16], 1234), ([5, 12, 9], 42)])
def test_audio_generate_ids_and_hiddens(orc, lengths, seed):
    ids, mask, tmask = synth_prompt_batch(lengths, seed=1)
    out = orc.generate(orc.embed_prompt(ids, tmask), ids, torch.tensor([0.3] * 4), 625, attention_mask=mask,
                       max_new_token=12, min_new_token=12, sampler=SamplerParams(), return_hidden=True,
                       manual_seed=seed)
    ref_ids = GOLD[f"audio_{seed}_ids"]
    assert ref_ids.shape == (len(lengths), 12, 4)
    for b in range(len(lengths)):
        assert np.array_equal(ref_ids[b], out.ids[b].numpy()), (b, ref_ids[b], out.ids[b])
    hid = _sampled(torch.stack(out.hiddens), f"audio_{seed}_hid")
    assert np.abs(hid - GOLD[f"audio_{seed}_hid"]).max() < 2e-5


def test_text_generate_ids(orc):
    ids, mask, tmask = synth_prompt_batch([7, 4], seed=3)
    out = orc.generate(orc.embed_prompt(ids, tmask), ids, torch.tensor([0.7]), 21001, attention_mask=mask,
                       max_new_token=6, sampler=SamplerParams(repetition_penalty=1.0, penalty_max_ids=21178),
                       infer_text=True, manual_seed=7)
    for b in range(2):
        assert np.array_equal(GOLD["text_ids"][b, : int(GOLD["text_n"][b])], out.ids[b].numpy())


def test_embed_prompt_matches(orc):
    ids, mask, tmask = synth_prompt_batch([6, 3], seed=5)
    tmask[0, -2:] = False  # mixed text / code positions (audio prompt splice, tokenizer.py:115-124)
    ids[0, -2:] = torch.randint(0, 626, (2, 4), generator=torch.Generator().manual_seed(5))
    assert np.array_equal(_sampled(orc.embed_prompt(ids, tmask), "embed"), GOLD["embed"])


def test_dvae_decoder_branch_matches_reference():
    """DVAE(decoder_config, dim=384) decode branch (the default use_decoder=True path)."""
    from chattts_b200.config import Config
    from chattts_b200.synth import synth_dvae_state
    from oracle.dvae_oracle import dvae_decode

    cfg = Config()
    st = synth_dvae_state(2, cfg.decoder, cfg.decoder.idim)
    x = torch.randn(2, 768, 20, generator=torch.Generator().manual_seed(20))
    want = torch.from_numpy(GOLD["dvae_mel"])
    got = dvae_decode(x, st)
    assert want.shape == got.shape == (2, 100, 40)
    assert (want - got).abs().max() < 1e-5 * max(1.0, float(want.abs().max()))


def test_dvae_encode_branch_matches_reference_up_to_the_quantizer():
    """Encode branch (dvae.py:265-274) piece by piece against the reference's own modules: MelSpectrogramFeatures
    (torchaudio), downsample_conv, encoder stack.  The FSQ quantiser itself is third-party and absent (parity unpinned)."""
    from chattts_b200.config import Config
    from chattts_b200.synth import synth_dvae_state, synth_speech_like
    from oracle.dvae_oracle import dvae_encode, mel_features

    cfg = Config()
    st = synth_dvae_state(3, cfg.dvae.decoder, cfg.dvae.decoder.idim, cfg.dvae.vq, encoder=cfg.dvae.encoder)
    for seconds, seed in ((1.3, 0), (2.0, 1)):
        wav = synth_speech_like(seconds, seed)
        mel = mel_features(wav)
        assert mel.shape == tuple(GOLD[f"enc{seed}_mel_shape"]) == (100, wav.numel() // 256 + 1)
        # same stft; the filterbank matmul runs in another order
        assert np.abs(_sampled(mel, f"enc{seed}_mel") - GOLD[f"enc{seed}_mel"]).max() < 2e-4
        ids, margin, _, x = dvae_encode(wav, st, return_parts=True)
        assert x.shape == tuple(GOLD[f"enc{seed}_x_shape"]) == (1, 1024, (wav.numel() // 256 + 1) // 2)
        tol = 1e-4 * max(1.0, float(GOLD[f"enc{seed}_x_absmax"]))
        assert np.abs(_sampled(x, f"enc{seed}_x") - GOLD[f"enc{seed}_x"]).max() < tol
        assert ids.shape == (1, 4, x.shape[2]) and int(ids.min()) >= 0 and int(ids.max()) < 625
