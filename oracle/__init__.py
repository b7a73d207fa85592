"""CPU oracle for the MFCC + FFN VAD hot path of nameofuser1/vad.

TEST INFRASTRUCTURE ONLY.  Nothing under ``vad_b200/`` may import this package.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs use it, and there only as the checker or as the timed
CPU baseline -- never as the thing shipped.

Pinning status
--------------
* MFCC / delta / analyser-feature math (``ref_math``): the reference ships no
  tests and no golden vectors (SURVEY.md section 4), so the restatement is pinned
  against the *unmodified reference code executed in the build container*
  (``oracle/reference_shim.py`` imports /root/reference/mfcc.py,
  dataset/file_processing.py and realtime_analysis/sklearn_analyser.py).
  ``oracle/make_golden.py`` froze those outputs into ``tests/golden/*.npz``;
  ``tests/test_oracle.py`` re-checks the restatement against the fixtures.
* FFN forward (``ref_math.ffn_forward``): **parity unpinned**.  The reference
  only defines the architecture (learning/ffn_trainer.py:104-116); it never
  runs inference, ships no weights, and its arithmetic lives in Keras 1.x
  (unvendored, unpinned, absent here).  The oracle restates Keras-1 ``Dense``
  semantics (y = act(x.W + b), W:(in,out), glorot_uniform, zero bias).
"""
