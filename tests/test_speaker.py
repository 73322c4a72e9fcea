"""Speaker strings / base16384 / prompt decoration (SURVEY.md 8f N3, host side) - CPU only.

The reference's outputs are stored in tests/golden/reference_host.{json,npz} (``python -m oracle.make_golden gen_host_pins``)."""
import json
import lzma
import os

import numpy as np
import pytest
import torch

from chattts_b200 import b14
from chattts_b200.speaker import Speaker

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _reference_host():
    with open(os.path.join(GOLD, "reference_host.json"), encoding="utf-8") as f:
        return json.load(f)


def test_base16384_round_trip_every_tail_length():
    rng = np.random.default_rng(0)
    for n in list(range(0, 40)) + [1535, 1536, 3072, 10_001]:
        data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        s = b14.encode_to_string(data)
        assert len(s) == (n // 7) * 4 + (0, 2, 3, 3, 4, 4, 5)[n % 7]
        assert all(0x4E00 <= ord(c) < 0x4E00 + (1 << 14) for c in (s[:-1] if n % 7 else s))
        assert b14.decode_from_string(s) == data


def test_base16384_known_answers():
    # 7 bytes -> 4 characters of 14 bits, most significant bit first
    assert b14.encode_to_string(b"\x00" * 7) == "一一一一"
    assert b14.encode_to_string(b"\xff" * 7) == chr(0x4E00 + 0x3FFF) * 4
    assert b14.encode_to_string(bytes([0x80, 0, 0, 0, 0, 0, 0x01])) == chr(0x4E00 + 0x2000) + "一一" + chr(0x4E01)
    assert b14.encode_to_string(b"\xff") == chr(0x4E00 + 0x3FC0) + chr(0x3D01)
    with pytest.raises(ValueError):
        b14.decode_from_string("abc")


def test_speaker_strings_start_like_the_reference_ones():
    """Every speaker string of the reference begins with "蘁淰" (examples/web/funcs.py:178): the LZMA2 chunk header
    E0 05 FF .. of a 1536-byte payload read as 14-bit groups.  Only the right bit order reproduces it."""
    stat = b14.encode_to_string(np.concatenate([np.full(768, 2.0, np.float16), np.zeros(768, np.float16)]).tobytes())
    spk = Speaker(768, stat)
    torch.manual_seed(0)
    s = spk.sample_random()
    assert s.startswith("蘁淰")
    emb = spk._decode(s)
    assert emb.shape == (768,) and emb.dtype == np.float16 and abs(float(emb.astype(np.float32).std()) - 2.0) < 0.3
    raw = b14.decode_from_string(s)
    assert len(lzma.decompress(raw, format=lzma.FORMAT_RAW,
                               filters=[{"id": lzma.FILTER_LZMA2, "preset": 9 | lzma.PRESET_EXTREME}])) == 1536


def test_reference_spk_stat_decodes_to_std_and_mean():
    """config.py:132: the reference's own base16384 asset decodes to exactly 2 x 768 fp16 with a positive std half."""
    stat = _reference_host()["spk_stat"]
    raw = b14.decode_from_string(stat)
    assert len(raw) == 2 * 768 * 2
    spk = Speaker(768, stat)
    assert torch.isfinite(spk.std).all() and float(spk.std.min()) > 0 and torch.isfinite(spk.mean).all()
    assert b14.encode_to_string(raw) == stat


def test_prompt_round_trip_and_shape_header():
    p = torch.randint(0, 626, (4, 37))
    s = Speaker.encode_prompt(p)
    back = Speaker.decode_prompt(s)
    assert back.dtype == torch.int32 and torch.equal(back, p.int())
    assert np.frombuffer(b14.decode_from_string(s)[:4], dtype="<u2").tolist() == [4, 37]
    with pytest.raises(AssertionError):
        Speaker.encode_prompt(torch.zeros(3, dtype=torch.int64))


def apply_inputs():
    torch.manual_seed(1)
    emb = torch.randn(3, 6, 768)
    vec = torch.randn(768)
    ids = torch.randint(0, 50, (3, 6, 4))
    ids[0, 2, 0] = ids[2, 5, 0] = 21143
    return emb, vec, ids


DECORATE_CASES = ((None, None), ("x", None), ("x", "sample text"))
DECORATE_TEXTS = ("  hi [Stts] there[spk_emb] ", "[empty_spk]b")


def test_apply_and_decoration_match_the_reference_speaker():
    """Against the reference Speaker's outputs on the same inputs: ``apply`` changed the rows ``apply_changed`` of the
    embedding to ``apply_rows``; decoration results and the in-place stripped text lists."""
    host, arrays = _reference_host(), np.load(os.path.join(GOLD, "reference_host.npz"))
    ours = object.__new__(Speaker)
    emb, vec, ids = apply_inputs()
    a = emb.clone()
    a[torch.from_numpy(arrays["apply_changed"])] = torch.from_numpy(arrays["apply_rows"])
    b = ours.apply(emb.clone(), vec, ids, 21143, torch.device("cpu"))
    assert torch.equal(a, b) and not torch.equal(a, emb)
    c = ours.apply(emb, vec, ids, 21143, torch.device("cpu"), inplace=False)
    assert torch.equal(c, a) and not torch.equal(emb, a)
    assert len(host["decorate_code"]) == len(DECORATE_CASES)
    for (spk_emb, smp), (want, stripped) in zip(DECORATE_CASES, host["decorate_code"]):
        t1 = list(DECORATE_TEXTS)
        assert ours.decorate_code_prompts(t1, "[speed_5]", smp, spk_emb) == want
        assert t1 == stripped                              # the caller's list is stripped in place by both
    assert ours.decorate_text_prompts(["a", "b"], "[oral_2]") == host["decorate_text"]


def test_decoration_golden():
    assert Speaker.decorate_code_prompts(["hi"], "", None, None) == ["[Stts][empty_spk]hi[Ptts]"]
    assert Speaker.decorate_code_prompts(["hi"], "[speed_5]", "ref", "e") == ["[Stts][spk_emb]ref[speed_5]hi[Ptts]"]
    assert Speaker.decorate_text_prompts(["hi"], "[oral_2]") == ["[Sbreak]hi[Pbreak][oral_2]"]
