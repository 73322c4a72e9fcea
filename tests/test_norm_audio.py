"""Host pre/post-processing (SURVEY.md 8f N4): chattts_b200.norm.Normalizer against what the reference's own Normalizer
returned on the same inputs, stored in tests/golden/reference_host.json (``python -m oracle.make_golden gen_host_pins``)."""
import json
import os

import numpy as np
import pytest

from chattts_b200.audio import float_to_int16, pcm_to_wav_bytes, strip_silence
from chattts_b200.norm import Normalizer, combine_tags, split_tags

HOMO = {"粘": "年", "呐": "那", "嗯": "恩", "A": "B"}
CASES = [
    "你好，世界！这是一个测试：ChatTTS（语音）合成。",
    "Hello, world! This is a test: (speech) synthesis - version 2.",
    "带标签的文本[uv_break]继续说话[laugh]结束。",
    "mixed 中文 and English words，符号#￥%……&*都有",
    "粘呐嗯 ABC [speed_5] tail",
    "no_invalid chars here, only letters. and commas",
    "stray ] bracket [x] and [unterminated",
    "nested [a[b]c] text",
    "数字123和符号@#都会被删除",
]


def normalizer_inputs():
    """(text, do_text_normalization, do_homophone_replacement, lang) for every case and flag combination; both sides
    have an "en" normaliser registered that upper-cases."""
    return [(text, norm, homo, lang) for text in CASES for norm in (True, False) for homo in (True, False)
            for lang in (None, "zh", "en")]


def test_normalizer_matches_reference_on_every_case_and_flag_combination():
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_host.json"),
              encoding="utf-8") as f:
        expected = json.load(f)["normalizer"]
    assert [tuple(r[:4]) for r in expected] == normalizer_inputs()
    ours = Normalizer(homophones=HOMO)
    assert ours.register("en", lambda s: s.upper())
    for text, norm, homo, lang, want in expected:
        assert ours(text, norm, homo, lang) == want, (text, norm, homo, lang)


def test_normalizer_golden_strings():
    n = Normalizer(homophones=HOMO)
    assert n("你好，世界！这是一个测试：ChatTTS（语音）合成。") == "你好，世界。这是一个测试，ChatTTS，语音，合成。"
    assert n("Hello, world! This is a test: (speech) synthesis - version 2.") == \
        "Hello, world. This is a test, ,speech, synthesis , version ."
    assert n("带标签的文本[uv_break]继续说话[laugh]结束。") == "带标签的文本[uv_break]继续说话[laugh]结束。"
    assert n("粘呐嗯 ABC [speed_5] tail") == "年那恩 BBC [speed_5] tail"
    assert n("no_invalid chars here", do_homophone_replacement=False) == "noinvalid chars here"


def test_split_and_combine_tags_round_trip_and_quirks():
    t, g = split_tags("a[x]b[y]c")
    assert (t, g) == (["a", "b", "c"], ["[x]", "[y]"]) and combine_tags(t, g) == "a[x]b[y]c"
    assert split_tags("abc") == (["abc"], [])
    assert split_tags("a[unterminated") == (["a"], [])            # the reference drops an unterminated tag
    assert split_tags("a]b") == (["a]b"], [""])                   # ... and records an empty tag for a stray ']'
    assert split_tags("a[b[c]d") == (["a", "", "d"], ["[c]"])     # a second '[' restarts the tag


def test_register_contract():
    n = Normalizer(homophones={})
    assert n.register("en", lambda s: s.lower())
    assert not n.register("en", lambda s: s)            # already registered
    assert not n.register("bad", lambda s: 123)         # must return str
    assert not n.register("boom", lambda s: 1 / 0)      # exceptions are reported, not raised
    assert n("HELLO There", lang="en") == "hello there"
    n.unregister("en")
    assert n("HELLO There", lang="en") == "HELLO There"


def test_float_to_int16_and_wav_container():
    x = np.array([0.0, 0.5, -1.0, 0.25], dtype=np.float32)
    y = float_to_int16(x)
    assert y.dtype == np.int16 and y.tolist() == [0, 16383, -32767, 8191]
    loud = float_to_int16(np.array([1.5, -3.0], dtype=np.float32))   # ceil(3.0) = 3 -> scale 10922
    assert loud.tolist() == [16383, -32766]
    with pytest.raises(ZeroDivisionError):
        float_to_int16(np.zeros(4, dtype=np.float32))
    b = pcm_to_wav_bytes(y)
    assert b[:4] == b"RIFF" and b[8:12] == b"WAVE" and len(b) == 44 + 8
    assert strip_silence(np.array([0.0, 1e-6, 2e-5, -0.5], dtype=np.float32)).tolist() == pytest.approx([2e-5, -0.5])
