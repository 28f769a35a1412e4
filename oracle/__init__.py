"""CPU oracle for the PILCO moment-matching rollout path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is imported by the product
packages (``pilco_b200`` / ``pilco``).  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it, and
only as the checker (or as the timed CPU reference arm), never as the thing shipped.

Contents
--------
matlab_port   loop-form numpy transcription of the reference's MATLAB oracle files
              (``tests/Matlab Code/{gp0,gp1,gp2,maha,conlin,gSin,reward,propagate,pred}.m``).
python_port   vectorised numpy transcription of the reference's Python hot path
              (``pilco/models/mgpr.py``, ``smgpr.py``, ``controllers.py``, ``rewards.py``,
              ``pilco/models/pilco.py``), materialising the [E,E,N,N] tensors like TF does.
torch_port    the same vectorised form in torch fp64 (autograd = gradient oracle; threaded
              CPU execution = the timed "reference-equivalent" CPU arm of bench.py).
staged        numpy statement of the *algorithm the CUDA kernels implement* (W-form mean,
              Cholesky-form pair prologue, A+B+u.zeta exponent, staged VJP) so that device
              workspaces can be compared stage by stage.
safe_port     numpy/torch transcription of the reference's safe_pilco_extension (parity unpinned: the
              reference has no test or golden vector for it).
fitc_staged   numpy statement of the FITC training objective with hand-derived adjoints (the algorithm a
              device SMGPR trainer implements), checked against torch autograd.
mrun          a small MATLAB-subset interpreter that executes the reference's ``.m`` files
              (the unmodified copies under ``tests/reference_tests/Matlab Code``) to pin the
              transcriptions and to generate ``tests/golden/*.npz``.

Pinning status: the reference commits NO golden vectors (its tests call Octave live) and
TensorFlow/GPflow/Octave are not installable here.  The oracle is pinned by (1) executing the
reference's own ``.m`` oracle files with ``oracle/mrun.py`` (transcriptions match to <=2e-12;
outputs committed as ``tests/golden/*.npz`` with ``tests/golden/make_golden.py``) and (2) the
cross-agreement of the two independent transcriptions -- the exact relation the reference's tests
assert at rtol 1e-4; ours agree to <=1e-9.  The reference's Python/TensorFlow side itself was never
executed here (not installable).  Gradients and optimiser trajectories: parity unpinned by the
reference (no reference test checks them); gradients are checked against torch autograd.
See DESIGN.md section 8.
"""
