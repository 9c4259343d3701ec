"""CPU oracle for the ensemble Kalman update path of agarbuno/ces.

TEST INFRASTRUCTURE ONLY.  Nothing under ``ces_b200/`` may import this
package; only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` do, and there only
as the checker or as the timed CPU baseline, never as the product path.

Modules
-------
eks_oracle       numpy restatement of ``sampling.eks_update*`` /
                 ``timestep_method`` / metrics (ces/calibrate.py:243-529).
                 Parity PINNED: checked against the real reference (run here,
                 tab-expanded in memory) and against tests/golden/*.npz that
                 were generated from it (tests/golden/make_golden.py).
forward_oracle   numpy restatement of the ``ces.utils`` map-type forward
                 models (ces/utils.py:5-122).  Parity PINNED the same way.
darcy_oracle     scipy restatement of ces/darcy.py + utilities/mfiles/*.m.
                 PARITY UNPINNED: the reference needs a MATLAB engine that is
                 not available and stores no Darcy output anywhere.
mcmc_oracle      numpy restatement of ``MCMC.model_mh`` (ces/sample.py:121-196).  Parity
                 PINNED: reproduces the golden chains of the real reference
                 (tests/golden/mcmc_cases.npz; tests/test_oracle_mcmc.py).
darcy_pcg_oracle / lorenz_oracle   restatements of the device's own solver / RK4 scheme (see
                 their headers).
philox_oracle    numpy restatement of the device's Philox4x32-10 streams
                 (``ces_fill_normal`` and the MH chains beside chain 0).  Parity
                 PINNED to the Random123 known-answer vectors
                 (tests/test_philox_oracle.py).
reference_loader loads the real reference from /root/reference when present
                 (never at run time on the GPU box).
"""
