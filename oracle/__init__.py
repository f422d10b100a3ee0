"""Oracle for the ST-encoder hot path -- TEST INFRASTRUCTURE ONLY.

Nothing under ``oracle/`` is product code.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it, and only as the checker or the timed
CPU baseline -- never as a fallback for the CUDA path.

Contents
--------
``encoder_oracle``  pure-torch CPU restatement of the reference algorithm
                    (every function cites the reference file:line it follows).
``ref_loader``      imports the LIVE reference from ``/root/reference`` with the
                    in-process shims of SURVEY.md F1/F2/F11 (only usable in the
                    build container; the GPU box has no ``/root/reference``).
``make_golden``     regenerates ``tests/golden/*.pt`` from the live reference.
``golden``          saves / loads those fixtures (one of more than 1 MB as parts of at most 1 MB).

Parity pinning: the reference's own test-suite holds NO golden vector for this
path (SURVEY.md section 4 / 8c) -- "parity unpinned" by the reference's suite.  The
oracle is therefore pinned against (a) outputs of the live reference run in the
build container (``tests/golden/*.pt``, generator committed) and (b) the
hand-derivable CTC-compression known-answer vector of SURVEY.md section 3.5.
"""
