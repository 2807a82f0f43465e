"""oracle/ -- TEST INFRASTRUCTURE ONLY.

CPU restatements of the reference's superquadric optimisation path, used as the
checker for the CUDA product path.  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import this
package; nothing under ``odam_b200/`` does (tests/test_boundary.py enforces it).

Contents
--------
sq_oracle.c          plain-C fp32 restatement (sampler + forward + analytic backward + Adam)
c_oracle.py          ctypes binding of the above (+ of oracle/_ref/libref_sampler.so)
torch_oracle.py      op-for-op PyTorch/autograd restatement of sq_libs.py's run loop
grad64.py            float64 restatement of one step's gradient with its discrete decisions held fixed
Makefile             builds _build/*.so and, when /root/reference is present, _ref/
"""
