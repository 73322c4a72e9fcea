"""CPU oracle for the two ChatTTS hot paths.  TEST INFRASTRUCTURE, NOT PRODUCT.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / reference
arm may import this package, and only as the checker (or the timed CPU baseline).  The
product path (``chattts_b200``) never imports it and fails loudly without its CUDA library.

Pin status (DESIGN.md §oracle):
* ``gpt_oracle``  - pinned against committed fixtures of what the reference's own
  ``GPT.generate`` / ``Embed`` / ``gen_logits`` + HF warpers + ``torch.multinomial`` computed
  (``tests/golden/*``, generator ``oracle/make_golden.py``; ``tests/test_oracle_golden.py``,
  ``tests/test_oracle_vs_reference.py``).
* ``dvae_oracle`` - ``DVAEDecoder``/``DVAE`` decode branch pinned the same way; the Vocos
  backbone/ISTFT head and GroupedResidualFSQ dequant are third-party code absent from
  ``/root/reference`` -> restated from the reference's call sites: **parity unpinned**
  for those two pieces (no reference test or golden vector exists for them).
"""
