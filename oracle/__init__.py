"""CPU oracle of the SimpleAICV data-parallel training hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` may be imported by the product package
(``simpleaicv_pytorch_training_examples_b200``); only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s cpu_baseline / ``--impl reference`` legs use it, and only as the checker or
the reported CPU baseline.

The reference is pure Python on top of PyTorch (torch is un-pinned in its requirements.txt;
its README names 2.5.1 / 2.8.0, this image has 2.11.0): the arithmetic of the path lives in
``torch.nn.functional``.  The oracle therefore restates the reference's *model code* as
functional fp32 torch-CPU code driven by a plain state dict (no nn.Module of the reference is
needed at run time), citing reference file:line for each function.

Pinning: the reference has no tests or golden vectors (SURVEY.md §4).  The oracle is pinned
against outputs of the reference itself: ``tests/golden/make_golden.py`` imports the reference
(copied into oracle/_ref by oracle/install_ref.sh) and writes small fixtures (inputs, logits, loss,
gradient digests) that ``tests/test_oracle_golden.py`` replays anywhere;
``tests/golden/make_reference_snapshots.py`` does the same for ``tests/test_oracle_vs_reference.py``
and the other tests that compare with the reference.
"""
