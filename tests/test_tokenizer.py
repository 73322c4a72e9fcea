"""chattts_b200.tokenizer.Tokenizer against the reference's Tokenizer on a small BERT vocabulary written on the fly."""
import json
import os

import numpy as np
import torch

SPECIAL = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", "[Stts]", "[Ptts]", "[spk_emb]", "[empty_spk]", "[Sbreak]",
           "[Pbreak]", "[Ebreak]", "[break_0]", "[uv_break]", "[speed_5]", "[oral_2]"]
WORDS = ["hello", "there", "world", "hi", "a", "b", "test", "##ing", "speech", ".", ","]


def _write_vocab(tmp_path):
    from transformers import BertTokenizerFast

    tok = BertTokenizerFast(vocab={w: i for i, w in enumerate(SPECIAL + WORDS)}, do_lower_case=True)
    tok.add_special_tokens({"additional_special_tokens": SPECIAL[5:]})
    out = tmp_path / "tok"
    tok.save_pretrained(str(out))
    return str(out)


def test_layout_left_padding_and_audio_prompt(tmp_path):
    from chattts_b200.tokenizer import Tokenizer

    t = Tokenizer(_write_vocab(tmp_path))
    assert t.len == len(SPECIAL) + len(WORDS)
    assert (t.spk_emb_ids, t.break_0_ids, t.eos_token) == (7, 12, 11)
    ids, att, tm = t.encode(["[Stts][spk_emb]hello there world[Ptts]", "[Stts][empty_spk]hi[Ptts]"], 4)
    assert ids.shape == (2, 6, 4) and att.shape == tm.shape == (2, 6)
    assert att.tolist() == [[1] * 6, [0, 0, 1, 1, 1, 1]] and torch.equal(tm, att.bool())
    assert ids[0, :, 0].tolist() == [5, 7, 16, 17, 18, 6] and bool((ids == ids[:, :, :1]).all())
    prompt = torch.arange(12).view(4, 3)
    ids2, att2, tm2 = t.encode(["hello", "hi there"], 4, prompt=prompt)
    assert ids2.shape == (2, 5, 4)
    assert att2.tolist() == [[0, 1, 1, 1, 1], [1, 1, 1, 1, 1]]
    assert tm2.tolist() == [[False, True, False, False, False], [True, True, False, False, False]]
    assert torch.equal(ids2[0, 2:], prompt.t()) and torch.equal(ids2[1, 2:], prompt.t())
    assert t.decode(ids[:, :, 0])[1].replace(" ", "").endswith("[Stts][empty_spk]hi[Ptts]")


TEXTS = ("[Stts][spk_emb]hello there world[Ptts]", "[Stts][empty_spk]hi[Ptts]", "testing speech, a b.")
PROMPT = torch.randint(0, 626, (4, 7), generator=torch.Generator().manual_seed(3))
DECODE_IDS = [[16, 17, 11], [19, 12]]


def test_matches_reference_tokenizer(tmp_path):
    """Against the reference Tokenizer's outputs on the same vocabulary and inputs (tests/golden/reference_host.*,
    ``python -m oracle.make_golden gen_host_pins``)."""
    from chattts_b200.tokenizer import Tokenizer

    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    with open(os.path.join(gold, "reference_host.json"), encoding="utf-8") as f:
        ref = json.load(f)["tokenizer"]
    arrays = np.load(os.path.join(gold, "reference_host.npz"))
    ours = Tokenizer(_write_vocab(tmp_path))
    assert (ours.len, ours.spk_emb_ids, ours.break_0_ids, ours.eos_token) == \
        (ref["len"], ref["spk_emb_ids"], ref["break_0_ids"], ref["eos_token"])
    for tag, prompt in (("noprompt", None), ("prompt", PROMPT)):
        a = ours.encode(list(TEXTS), 4, prompt=prompt)
        for x, name in zip(a, ("ids", "attention_mask", "text_mask")):
            y = torch.from_numpy(arrays[f"tok_{tag}_{name}"])
            assert x.dtype == y.dtype and torch.equal(x, y), (tag, name)
    assert ours.decode(DECODE_IDS) == ref["decode"]
