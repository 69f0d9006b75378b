"""CPU oracle for the ConsistentID denoising hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import it, and there only as
the checker or the timed CPU baseline.  The product path
(``consistentid_b200``) never imports this package and fails loudly when its
CUDA library is missing.

What is restated here
---------------------
* ``processors_ref``  - the reference's own code for the path:
  ``attention.py:90-174`` (Consistent_AttProcessor) and ``attention.py:177-294``
  (Consistent_IPAttProcessor).  PINNED: ``tests/golden/*.pt`` hold outputs
  of the reference ``attention.py`` imported verbatim (through the 2-symbol
  ``oracle/diffusers_shim``; ``tests/golden/make_golden.py``,
  ``tests/golden/make_pinned_golden.py``) and ``tests/test_oracle_cpu.py``
  compares.
* ``unet_ref`` / ``schedulers_ref`` - the third-party dependency the reference
  calls for ~99 % of the arithmetic: ``diffusers==0.23.0``
  (``requirements.txt:36``; not vendored in /root/reference, not installable
  here).  Its published algorithm is restated from SURVEY.md Appendix A.  The
  reference has no tests / golden vectors for this part, so for it PARITY IS
  UNPINNED (anchored only on the reference's call sites:
  ``pipline_StableDiffusion_ConsistentID.py:536-579``,
  ``pipline_StableDiffusionXL_ConsistentID.py:611-667``).
* ``loop_ref`` - the denoising-loop bodies of the reference pipelines.
* ``controlnet_ref`` - diffusers ``ControlNetModel`` with default processors (config 5; unpinned like ``unet_ref``).
* ``embed_ref`` - the embedding producers ``ProjPlusModel`` / ``AttentionMLP`` / ``FuseModule`` / ``FacialEncoder``
  (``functions.py:389-592``, ``attention.py:10-88``).  PINNED on golden vectors generated from the reference's own classes
  (``tests/golden/make_embed_golden.py``).
* ``clip_ref`` - CLIP ViT image encoder up to ``hidden_states[-2]``.  PINNED on the ``transformers`` implementation installed in this
  image (``tests/test_clip_cpu.py``).
* ``vae_ref`` - diffusers ``AutoencoderKL`` decode (unpinned; anchored on the decoder's published 49,490,179 parameters).
* ``synth`` - seeded synthetic weights / prompts / latents (SURVEY.md 8d).
"""
