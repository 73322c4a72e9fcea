"""Import the *unmodified* reference (``/root/reference``) inside the build container.

TEST INFRASTRUCTURE ONLY.  Nothing under ``chattts_b200/`` may import this module; only
``oracle/make_golden.py`` uses it, to write the fixtures under ``tests/golden/`` that the
tests compare with, so no test needs the reference at run time.

The reference cannot be imported as-is here (SURVEY.md §8c): ``vocos``,
``vector_quantize_pytorch`` and ``pybase16384`` are not installed and there is no network.
None of the three is needed for the arithmetic we pin (they are only *names* at import
time), so we register empty stub modules for them, plus one shim for a transformers API
drift (``DynamicCache.get_max_cache_shape`` returns -1 in transformers>=4.48/5.x, which
breaks ``ChatTTS/model/gpt.py:190-232``).
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("CHATTTS_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "ChatTTS"))


def load_reference():
    """Return the imported ``ChatTTS`` reference package (with stubs installed)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    for name in ("vocos", "vocos.pretrained", "pybase16384", "vector_quantize_pytorch"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["vocos"].Vocos = object
    sys.modules["vocos.pretrained"].instantiate_class = lambda *a, **k: None
    sys.modules["vector_quantize_pytorch"].GroupedResidualFSQ = object
    from transformers.cache_utils import DynamicCache

    DynamicCache.get_max_cache_shape = lambda self, *a, **k: None
    import ChatTTS  # noqa: F401  (the reference package)

    return sys.modules["ChatTTS"]
