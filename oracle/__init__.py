"""CPU oracle for the multimodal timing-prediction hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is product code: only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it, and there only as the checker or the
CPU arm being timed.  The product path (the package
``multimodal-fusion-based-pre-routing-timing-prediction-_b200``) never imports
this package and fails loudly when its CUDA library is missing.

Layout
------
``restate.py``    pure-PyTorch CPU restatement of the reference arithmetic
                  (``src/model.py``, ``src/Unet.py``, ``src/train.py:465-555``);
                  travels to the GPU box.
``levelize.py``   plain-Python / numpy restatement of
                  ``verilog_parser_asap7.py:1452-1517`` (level construction),
                  ``:1433-1450`` (critical-path trace) and ``:1302-1369``
                  (path-mask rasterisation), plus the in-edge CSR definition.
``fake_dgl.py``   ~100-line stand-in for the DGL graph surface the reference
                  touches (``pull`` semantics per SURVEY.md Appendix A).
``dgl_stub/``     inert ``dgl.function`` so the reference's ``model.py`` imports.
``ref_loader.py`` imports the UNMODIFIED reference modules from the original
                  project's ``src/`` (``TM_REFERENCE_SRC``; not in this repository).
``make_golden.py``runs the unmodified reference on seeded inputs and writes
                  ``tests/golden/*.npz`` -- the committed fixtures the oracle
                  restatement and the CUDA path are pinned against.

Parity status: the torch-only parts (MLP, UNet, LayoutNet, PathModel head) are
pinned against the reference's own classes executed here.  ``PathConv`` is
pinned against the reference's own ``forward``/UDFs executed through
``fake_dgl`` -- DGL itself is absent (no version is pinned by the reference, no
network), so the DGL ``pull`` semantics are restated, not executed:
**parity unpinned at the DGL boundary** (see DESIGN.md).
"""
