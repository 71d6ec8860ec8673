"""CPU oracle for the box-supervised mask-loss hot path.

THIS PACKAGE IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it, and only as the *checker* (or as the timed CPU
baseline) -- never as the thing shipped.  ``boxinstseg_b200`` must not import it.

Every function restates, in independent code, the arithmetic of one reference function
and cites the reference file:line it follows (paths relative to ``/root/reference``).

Parity pinning status (see DESIGN.md "Oracle"):
  * The reference ships no tests / golden vectors for this path (SURVEY.md section 4), so
    the pin is "outputs of the reference itself": ``oracle/make_golden.py`` AST-extracts
    the reference's own pure-PyTorch functions from ``/root/reference`` (runs only in the
    authoring container), runs them on seeded inputs and commits inputs+outputs under
    ``tests/golden``; ``tests/test_oracle_golden.py`` checks this oracle against them.
  * The MST restatement is pinned against the reference's own ``boruvka.cpp`` compiled
    from where it lies into ``oracle/_ref/`` (``oracle/Makefile``), and the committed
    edge-set fixtures produced from it.
  * The reference's CUDA extensions (``mmdet/ops/pairwise``, ``mmdet/ops/tree_filter``) are compiled
    UNMODIFIED by ``oracle/Makefile`` into ``oracle/_ref/*.so`` (an empty ``THC/THC.h`` shim under
    ``oracle/csrc/shim`` replaces the header PyTorch no longer ships); they run only on a GPU:
    ``oracle/make_golden_ref_ext.py`` stores their outputs as the golden vectors that
    ``tests/test_reference_ext_gpu.py`` and ``tests/test_config_a_gpu.py`` compare the product's kernels with,
    ``bench.py`` times the reference's GPU loss path around its pairwise op (``gpu_reference``).
  * ``skimage.color.rgb2lab`` and ``mmcv.tensor2imgs`` are third-party code absent from
    ``/root/reference`` (scikit-image unpinned; mmcv-full 1.3.17-1.6.0): their published
    algorithms are restated and pinned on known-answer colours + OpenCV's independent
    implementation -> "parity unpinned" for those two functions only.
  * ``oracle/solo_targets.py`` (SOLO grid targets, box_solov2_head.py:390-472) is pinned on the reference's own METHOD:
    ``oracle/make_golden_solo.py`` AST-extracts ``BoxSOLOv2Head.solo_target_single``, runs it and asserts equality; its
    ``mmcv.imrescale`` (third party, absent) is the ``cv2.resize`` call mmcv makes, OpenCV being importable here.
"""
