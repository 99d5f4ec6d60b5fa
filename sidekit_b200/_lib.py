"""ctypes binding of ``libsidekit_b200.so`` (C ABI declared in include/sidekit_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is
visible the ops raise.  ``build()`` compiles the library in-tree with nvcc for
sm_100a (``build.sh``); the built ``.so`` ships with the source tree.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("SKB_LIB_PATH") or os.path.join(_HERE, "libsidekit_b200.so")      # override: A/B builds
_lib = None

c_float_p = ctypes.c_void_p      # device / host pointers are passed as integers
c_i64_p = ctypes.POINTER(ctypes.c_int64)


def build(verbose=False):
    """Compile every CUDA source for sm_100a into ``libsidekit_b200.so`` (in-tree)."""
    out = subprocess.run(["bash", os.path.join(_ROOT, "build.sh")], cwd=_ROOT, capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout)
        print(out.stderr)
    if out.returncode != 0:
        raise RuntimeError("nvcc build of libsidekit_b200.so failed:\n" + out.stderr[-4000:])
    return LIB_PATH


def _declare(lib):
    vp, i32, i64, f32, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double
    sigs = {
        "skb_version": (i32, []),
        "skb_last_error": (ctypes.c_char_p, []),
        "skb_kernel_launches": (i64, []),
        "skb_profile_enable": (None, [i32]),
        "skb_profile_read": (i32, [ctypes.POINTER(ctypes.c_float), i32]),
        "skb_xtractor_create": (i32, [i32, i32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(vp),
                                      ctypes.POINTER(c_i64_p), ctypes.POINTER(i32), i32, f32, ctypes.POINTER(vp)]),
        "skb_xtractor_destroy": (None, [vp]),
        "skb_xtractor_embedding_size": (i32, [vp]),
        "skb_xtractor_speaker_number": (i32, [vp]),
        "skb_xtractor_num_frames": (i32, [vp, i64]),
        "skb_xtractor_forward": (i32, [vp, vp, c_i64_p, i32, i32, vp, vp, vp]),
        "skb_xtractor_forward_host": (i32, [vp, vp, c_i64_p, i32, i32, vp, vp, vp]),
        "skb_xtractor_frontend": (i32, [vp, vp, c_i64_p, i32, i32, vp, vp]),
        "skb_xtractor_debug_stage": (i32, [vp, vp, c_i64_p, i32, ctypes.c_char_p, i32, vp, c_i64_p, vp]),
        "skb_xtractor_pre_embedding": (i32, [vp, i32, vp, vp]),
        "skb_xtractor_reserve": (i32, [vp, i32, i64, vp]),
        "skb_xtractor_overflow_count": (i32, [vp, vp, c_i64_p]),
        "skb_xtractor_wait_tables": (i32, [vp, vp]),
        "skb_conv2d_bn_act": (i32, [vp, i32, i32, i32, i32, vp, vp, i32, i32, i32, vp, vp, f32, f32, vp, vp, i32, vp, vp]),
        "skb_ops_overflow_count": (i32, [vp, c_i64_p]),
        "skb_channel_mean": (i32, [vp, i32, i32, i64, vp, vp]),
        "skb_se_gate": (i32, [vp, vp, vp, i32, i32, i32, vp, vp]),
        "skb_scale_residual_act": (i32, [vp, vp, vp, i32, i32, i64, f32, vp, vp]),
        "skb_l2_normalize": (i32, [vp, i32, i32, f32, vp, vp]),
        "skb_attentive_pool": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp]),
        "skb_meanstd_pool": (i32, [vp, i32, i32, i32, vp, vp]),
        "skb_score_gemm": (i32, [vp, vp, i32, i32, i32, vp, vp, f64, f64, i32, i32, vp, i64, vp]),
        "skb_packed_create": (i32, [vp, i32, i32, ctypes.POINTER(vp), vp]),
        "skb_packed_destroy": (None, [vp]),
        "skb_score_gemm_packed": (i32, [vp, i32, vp, vp, vp, f64, f64, i32, i32, vp, i64, vp]),
        "skb_trial_index_create": (i32, [vp, i32, i32, i64, ctypes.POINTER(vp), c_i64_p, vp]),
        "skb_trial_index_destroy": (None, [vp]),
        "skb_score_gemm_trials": (i32, [vp, vp, i32, i32, i32, vp, vp, f64, f64, i32, vp, vp, vp]),
        "skb_score_gemm_trials_packed": (i32, [vp, i32, vp, vp, vp, f64, f64, i32, vp, vp, vp]),
        "skb_score_pairs": (i32, [vp, vp, i32, i32, i32, vp, vp, i64, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp]),
        "skb_score_gemm_topk": (i32, [vp, vp, i32, i32, i32, vp, vp, f64, f64, i32, i32, vp, vp, vp]),
        "skb_score_gemm_topk_packed": (i32, [vp, i32, vp, vp, vp, f64, f64, i32, i32, vp, vp, vp]),
        "skb_widen_f32_f64": (i32, [vp, vp, i64, vp]),
        "skb_quadratic_prepare": (i32, [vp, vp, vp, vp, i32, i32, vp, vp, vp]),
        "skb_asnorm_stats": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
        "skb_asnorm_apply": (i32, [vp, i32, i32, vp, vp, vp, vp]),
        "skb_asnorm_apply_panel": (i32, [vp, i32, i32, i32, i32, vp, vp, vp, i64, vp]),
        "skb_pavx": (i32, [vp, i64, vp, vp, vp, c_i64_p]),
        "skb_rocch": (i32, [vp, i64, vp, i64, vp, vp, c_i64_p]),
        "skb_eer": (i32, [vp, i64, vp, i64, ctypes.POINTER(f64)]),
        "skb_scoremat_stats": (i32, [vp, i32, i32, i64, i32, i32, i32, vp, vp, vp]),
        "skb_scoremat_normalise": (i32, [vp, i32, i32, i64, i32, vp, vp, vp, i64, vp]),
        "skb_plda_stats": (i32, [vp, i32, i32, vp, vp, i32, f64, vp, vp, vp, vp]),
        "skb_plda_em": (i32, [vp, vp, vp, i32, vp, vp, i32, vp, vp, i32, i32, i32, f64, vp, vp, vp]),
        "skb_gram_f64": (i32, [vp, i32, i64, i32, i64, vp, vp, vp, f64, vp, vp]),
        "skb_class_stats": (i32, [vp, i32, i64, i32, i64, vp, vp, i32, vp, vp, vp, vp]),
        "skb_affine_rows": (i32, [vp, i32, i64, i32, i64, vp, vp, vp, i32, i32, vp, i32, i64, vp]),
        "skb_resample":(i32, [vp, vp, i32, i64, i32, i32, i32, vp, vp, i32, vp, vp]),
        "skb_flac_workspace_bytes": (i64, [i64, i32, i64]),
        "skb_flac_decode": (i32, [vp, i64, vp, i32, i64, vp, i64, vp, vp, vp]),
        "skb_pcm_decode": (i32, [vp, vp, i32, i64, vp, vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)       # AttributeError here = header / library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    return sigs


def lib():
    """The loaded library; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("sidekit_b200: %s not found -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        _declare(l)
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError("sidekit_b200 native call failed (%d): %s" % (rc, lib().skb_last_error().decode()))


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def i64_array(values):
    arr = (ctypes.c_int64 * len(values))(*[int(v) for v in values])
    return arr
