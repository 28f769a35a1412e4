"""ctypes binding of ``libpilco_b200.so`` (the C ABI declared in ``include/pilco_b200.h``).

The product path has no CPU fallback: if the shared library is missing the import of this module
raises, and every compute entry point raises unless a CUDA device is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PILCO_B200_LIB") or os.path.join(_HERE, "libpilco_b200.so")   # env: diagnostics builds

c_dp = C.c_void_p          # device pointers are passed as integers (tensor.data_ptr())
c_ll = C.c_longlong


class GpModel(C.Structure):
    """mirror of ``pilco_gp_model``"""
    _fields_ = [("n", C.c_int), ("D", C.c_int), ("E", C.c_int), ("mode", C.c_int),
                ("X", c_dp), ("X_bs", c_ll),
                ("ell", c_dp), ("ell_bs", c_ll),
                ("sf2", c_dp), ("sf2_bs", c_ll),
                ("beta", c_dp), ("beta_bs", c_ll),
                ("iK", c_dp), ("ldk", C.c_int)]


class Policy(C.Structure):
    """mirror of ``pilco_policy``"""
    _fields_ = [("kind", C.c_int), ("Ds", C.c_int), ("U", C.c_int), ("squash", C.c_int),
                ("max_action", c_dp),
                ("W", c_dp), ("W_bs", c_ll), ("b", c_dp), ("b_bs", c_ll),
                ("rbf", GpModel)]


class RewardTerm(C.Structure):
    """mirror of ``pilco_reward_term``"""
    _fields_ = [("kind", C.c_int), ("channel", C.c_int), ("coef", C.c_double), ("W", c_dp), ("t", c_dp)]


class Rollout(C.Structure):
    """mirror of ``pilco_rollout``"""
    _fields_ = [("R", C.c_int), ("H", C.c_int),
                ("dyn", GpModel), ("pol", Policy),
                ("n_rewards", C.c_int), ("rewards", RewardTerm * 8),
                ("m0", c_dp), ("m0_bs", c_ll), ("S0", c_dp), ("S0_bs", c_ll),
                ("traj_m", c_dp), ("traj_S", c_dp), ("reward", c_dp), ("step_reward", c_dp),
                ("info", c_dp), ("ws", c_dp), ("ws_bytes", C.c_size_t),
                ("mult_mu", C.c_double), ("step_risk", c_dp),
                ("tape", c_dp), ("tape_bytes", C.c_size_t)]


class RolloutGrad(C.Structure):
    """mirror of ``pilco_rollout_grad``"""
    _fields_ = [("gW", c_dp), ("gb", c_dp), ("gXc", c_dp), ("gYc", c_dp), ("gell", c_dp), ("pol_L", c_dp),
                ("gm0", c_dp), ("gS0", c_dp), ("ws", c_dp), ("ws_bytes", C.c_size_t)]


POLICY_LINEAR, POLICY_RBF = 0, 1
REWARD_EXP, REWARD_LINEAR, REWARD_BOX = 0, 1, 2
CHANNEL_ADD, CHANNEL_MULT = 0, 1
ABI_VERSION = 3

# name -> (restype, argtypes); every symbol declared in include/pilco_b200.h
SIGNATURES = {
    "pilco_version": (C.c_int, []),
    "pilco_status_string": (C.c_char_p, [C.c_int]),
    "pilco_pad_n": (C.c_int, [C.c_int]),
    "pilco_mm_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "pilco_mm_forward": (C.c_int, [C.POINTER(GpModel), C.c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                   c_dp, C.c_size_t, c_dp]),
    "pilco_gp_factorize_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "pilco_gp_factorize": (C.c_int, [C.c_int] * 4 + [c_dp, c_ll] * 5 + [c_dp, C.c_int, c_dp, c_dp,
                                                                        c_dp, C.c_size_t, c_dp]),
    "pilco_gp_append_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "pilco_gp_append": (C.c_int, [C.c_int] * 4 + [c_dp] * 5 + [c_dp, C.c_int, c_dp, C.c_int, c_dp, c_dp,
                                                            c_dp, C.c_size_t, c_dp]),
    "pilco_gp_nlml_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "pilco_gp_nlml": (C.c_int, [C.c_int] * 4 + [c_dp, c_ll] * 5 + [c_dp] * 5 + [c_dp, C.c_size_t, c_dp]),
    "pilco_fitc_nlml_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "pilco_fitc_nlml": (C.c_int, [C.c_int] * 5 + [c_dp] * 6 + [c_dp] * 6 + [c_dp, C.c_size_t, c_dp]),
    "pilco_fitc_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "pilco_fitc_factorize": (C.c_int, [C.c_int] * 4 + [c_dp] * 6 + [c_dp, C.c_int, c_dp, c_dp, c_dp,
                                                                  C.c_size_t, c_dp]),
    "pilco_gp_predict_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "pilco_gp_predict": (C.c_int, [C.POINTER(GpModel), C.c_int] + [c_dp] * 5 + [C.c_size_t, c_dp]),
    "pilco_squash_sin":(C.c_int, [C.c_int, C.c_int] + [c_dp] * 7),
    "pilco_linear_action": (C.c_int, [C.c_int] * 3 + [c_dp, c_ll, c_dp, c_ll] + [c_dp] * 6),
    "pilco_exp_reward": (C.c_int, [C.c_int, C.c_int] + [c_dp] * 8),
    "pilco_box_risk": (C.c_int, [C.c_int, C.c_int] + [c_dp] * 7),
    "pilco_rollout_workspace_bytes": (C.c_size_t, [C.POINTER(Rollout)]),
    "pilco_rollout_tape_bytes": (C.c_size_t, [C.POINTER(Rollout)]),
    "pilco_mm_tape_bytes": (C.c_size_t, [C.c_int] * 4),
    "pilco_mm_tape_bwd_workspace_bytes": (C.c_size_t, [C.c_int] * 3),
    "pilco_mm_forward_taped": (C.c_int, [C.POINTER(GpModel), C.c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                         c_dp, C.c_size_t, c_dp, C.c_size_t, c_dp]),
    "pilco_mm_backward_taped": (C.c_int, [C.POINTER(GpModel), C.c_int] + [c_dp] * 6 + [c_dp, C.c_size_t, c_dp, c_dp,
                                                                                  c_dp, C.c_size_t, c_dp]),
    "pilco_rollout_forward": (C.c_int, [C.POINTER(Rollout), c_dp]),
    "pilco_mm_bwd_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "pilco_mm_backward": (C.c_int, [C.POINTER(GpModel), C.c_int] + [c_dp] * 11 + [c_dp, C.c_size_t, c_dp]),
    "pilco_rollout_bwd_workspace_bytes": (C.c_size_t, [C.POINTER(Rollout)]),
    "pilco_rollout_backward": (C.c_int, [C.POINTER(Rollout), C.POINTER(RolloutGrad), c_dp]),
    "pilco_mm_forward_profile": (C.c_int, [C.POINTER(GpModel), C.c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                           c_dp, C.c_size_t, C.POINTER(C.c_float), c_dp]),
    "pilco_mm_forward_taped_profile": (C.c_int, [C.POINTER(GpModel), C.c_int, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                                 c_dp, C.c_size_t, c_dp, C.c_size_t, C.POINTER(C.c_float), c_dp]),
    "pilco_microbench_fp64": (C.c_int, [C.c_int, C.c_int, C.c_int, c_dp, C.POINTER(C.c_float), c_dp]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "pilco_b200: %s is missing -- build it with `python -m pilco_b200.build` "
            "(there is no CPU fallback for the moment-matching path)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.pilco_version() != ABI_VERSION:
        raise RuntimeError("pilco_b200: ABI version mismatch")
    return lib


lib = _load()


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError("pilco_b200 %s failed: %s (status %d)" %
                           (what, lib.pilco_status_string(rc).decode(), rc))
