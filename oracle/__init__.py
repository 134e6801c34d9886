"""CPU oracle for the wavelet-monodepth decoder hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in ``wavelet_monodepth_b200`` (the product)
imports this package.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it, and
there only as the checker or as the timed CPU arm.

What it is: a torch-CPU (fp32) restatement of the reference's decoder path,
written from the reference sources, each function citing the reference
file:line it follows (paths relative to the reference checkout):

* ``oracle.haar``       - Haar DWT / IDWT as the un-vendored ``pytorch_wavelets``
                          dependency (latest release 1.3.0, un-pinned by the
                          reference, README.md:58-65) computes them; also usable
                          as a drop-in ``pytorch_wavelets`` stand-in when the
                          reference itself is imported by ``oracle/pin_against_reference.py``.
* ``oracle.sparse_ops`` - KITTI/layers.py:335-508 and NYUv2/networks/layers.py:82-223.
* ``oracle.kitti``      - KITTI/networks/decoders/depth_decoder.py:72-428.
* ``oracle.nyu``        - NYUv2/networks/decoders/densedepth_decoder.py:92-148,224-409.

Pinning status (see DESIGN.md "Oracle"):
* decoders + sparse ops: PINNED - ``oracle/pin_against_reference.py`` imports the
  unmodified reference from /root/reference (possible only in the build
  container) and checks every output of the restatement against it, then
  writes the golden vectors under ``tests/golden/``.
* known-answer values from the reference's notebooks (17 473 692 295 and
  33 463 546 800 ops) are reproduced (tests/test_opcount.py).
* Haar DWT/IDWT arithmetic: the reference's own closed form ``my_iwt_once``
  (depth_decoder.py:225-239) pins it algebraically (checked to <=1e-6); the
  third-party package itself is absent from the container, so bit-level parity
  with ``pytorch_wavelets`` proper is UNPINNED ("parity unpinned" for that
  dependency only).
"""

# Intra-op threads of the process that writes and checks the golden vectors.  The CPU GEMMs split their sums by thread
# count, so the restatement reproduces the reference's fp32 outputs bit for bit only at the count they were written with.
GOLDEN_THREADS = 8
