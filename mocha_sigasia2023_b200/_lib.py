"""ctypes binding of libmocha_b200.so (include/mocha_b200.h).

The library is the product: if it is missing or the device is not an sm_100 GPU every compute call
raises — there is no CPU or PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# MOCHA_LIB selects another build of the same library (e.g. the --trace debug build)
LIB_PATH = os.environ.get("MOCHA_LIB") or os.path.join(_HERE, "libmocha_b200.so")

MOCHA_FP32 = 0
MOCHA_BF16 = 1
MOCHA_TF32X3 = 2


@contextlib.contextmanager
def workspace_precision(prec: int):
    """The mocha_*_workspace_bytes queries inside the block answer for precision mode `prec` (MOCHA_TF32X3 needs room for
    its split operands); the library default is restored afterwards."""
    lib = load()
    check(lib.mocha_workspace_precision(int(prec)), "mocha_workspace_precision")
    try:
        yield
    finally:
        lib.mocha_workspace_precision(MOCHA_BF16)


def precision_code(precision: str) -> int:
    """"fp32" (FFMA parity mode), "bf16" (tcgen05 throughput mode) or "tf32x3" (parity mode on tcgen05: split-fp32 GEMMs)."""
    try:
        return {"fp32": MOCHA_FP32, "bf16": MOCHA_BF16, "tf32x3": MOCHA_TF32X3}[precision]
    except KeyError:
        raise ValueError(f"unknown precision {precision!r} (fp32 | bf16 | tf32x3)") from None
MAX_DEPTH = 4

c_float_p = C.c_void_p  # device pointers travel as integers


class MochaError(RuntimeError):
    pass


class Dims(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "T", "V", "Cin", "C0", "D", "P", "tp", "Kj", "Kb", "taps_j", "taps_b", "heads", "enc_dh", "dec_dh",
        "mlp", "enc_depth", "dec_depth")]


class EncLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("wqkv", "wo", "bo", "w1", "b1", "w2", "b2")]


class DecLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "sw1", "sb1", "sw2", "sb2", "wq", "wk", "wv", "wo", "bo", "w1", "b1", "w2", "b2")]


class GeneratorWeights(C.Structure):
    _fields_ = (
        [("dims", Dims)]
        + [(n, C.c_void_p) for n in (
            "emb_w", "emb_b", "A_j", "jb_gcn_w", "jb_gcn_bias2d", "jb_tcn_w", "jb_tcn_b", "pool_w", "A_b",
            "bb_gcn_w", "bb_gcn_bias2d", "bb_tcn_w", "bb_tcn_b", "pos_emb", "tok_bias_pos")]
        + [("enc", EncLayer * MAX_DEPTH), ("dec", DecLayer * MAX_DEPTH)]
        + [(n, C.c_void_p) for n in (
            "tm_A_b", "tm_bb_gcn_w", "tm_bb_gcn_bias2d", "tm_bb_tcn_w", "tm_bb_tcn_b", "tm_jb_gcn_w",
            "tm_jb_gcn_b", "tm_A2", "tm_jb_tcn_w", "tm_jb_tcn_b", "tm_out_w", "tm_out_b")]
        + [("jb_gcn_w_aug", C.c_void_p), ("jb_gcn_kaug", C.c_int)]
    )


class CvaeEncLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "in_w", "in_b", "out_w", "out_b", "l1_w", "l1_b", "l2_w", "l2_b", "n1_g", "n1_b", "n2_g", "n2_b")]


class CvaeDecLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "sa_in_w", "sa_in_b", "sa_out_w", "sa_out_b", "ca_in_w", "ca_in_b", "ca_out_w", "ca_out_b",
        "l1_w", "l1_b", "l2_w", "l2_b", "n1_g", "n1_b", "n2_g", "n2_b", "n3_g", "n3_b")]


class CvaeWeights(C.Structure):
    _fields_ = [
        ("D", C.c_int), ("heads", C.c_int), ("dff", C.c_int), ("depth", C.c_int), ("out_seq", C.c_int),
        ("ln_eps", C.c_float),
        ("mu_token", C.c_void_p), ("logvar_token", C.c_void_p), ("pe", C.c_void_p),
        ("prior", CvaeEncLayer * MAX_DEPTH), ("dec", CvaeDecLayer * MAX_DEPTH),
        ("dec0_sa", C.c_void_p),
        ("dec0_q16", C.c_void_p),
    ]


class ClipState(C.Structure):
    _fields_ = [
        ("root_pos", C.c_double * 3), ("root_rot", C.c_double * 4),
        ("src_root_pos", C.c_double * 3), ("src_root_rot", C.c_double * 4),
        ("prev_pos", (C.c_double * 3) * 25), ("prev_ik_pos", (C.c_double * 3) * 25),
        ("contact_state", C.c_int32 * 2), ("contact_lock", C.c_int32 * 2),
        ("contact_position", (C.c_double * 3) * 2), ("contact_velocity", (C.c_double * 3) * 2),
        ("contact_point", (C.c_double * 3) * 2), ("contact_target", (C.c_double * 3) * 2),
        ("contact_offset_position", (C.c_double * 3) * 2), ("contact_offset_velocity", (C.c_double * 3) * 2),
    ]


class PostParams(C.Structure):
    _fields_ = [
        ("J", C.c_int), ("parents", C.c_int32 * 32), ("contact_bones", C.c_int32 * 2), ("dt", C.c_double),
        ("ik_max_length_buffer", C.c_double), ("ik_foot_height", C.c_double), ("ik_unlock_radius", C.c_double),
        ("ik_blending_halflife", C.c_double), ("ik_enabled", C.c_int),
    ]


class FrameOut(C.Structure):
    _fields_ = [
        ("pos", (C.c_double * 3) * 25), ("rot", (C.c_double * 4) * 25), ("vel", (C.c_double * 3) * 25),
        ("ang", (C.c_double * 3) * 25), ("blend_pos", (C.c_double * 3) * 25), ("ik_pos", (C.c_double * 3) * 25),
        ("ik_rot", (C.c_double * 4) * 25),
        ("src_root_pos", C.c_double * 3), ("src_root_rot", C.c_double * 4), ("src_root_vel", C.c_double * 3),
        ("src_root_ang", C.c_double * 3),
    ]


_STRUCTS = [Dims, EncLayer, DecLayer, GeneratorWeights, CvaeEncLayer, CvaeDecLayer, CvaeWeights, ClipState,
            PostParams, FrameOut]

# name -> (restype, argtypes); every symbol include/mocha_b200.h declares
_P, _I, _L, _D, _F, _S = C.c_void_p, C.c_int, C.c_longlong, C.c_double, C.c_float, C.c_size_t
SIGNATURES = {
    "mocha_last_error": (C.c_char_p, []),
    "mocha_version": (_I, []),
    "mocha_check_device": (_I, []),
    "mocha_launch_count": (_L, []),
    "mocha_reset_launch_count": (None, []),
    "mocha_struct_sizes": (_I, [C.POINTER(C.c_size_t), _I]),
    "mocha_register_bf16_blob": (_I, [_P, _P, _S]),
    "mocha_workspace_precision": (_I, [_I]),
    "mocha_embed_workspace_bytes": (_S, [C.POINTER(Dims), _I]),
    "mocha_embed_fwd": (_I, [C.POINTER(GeneratorWeights), _P, _I, _P, _I, _I, _P, _S, _P]),
    "mocha_bench_tconv": (_I, [C.POINTER(GeneratorWeights), _P, _I, _P, _I, _I, _P, _S, _P]),
    "mocha_bench_hbm_kernel": (_I, [C.POINTER(GeneratorWeights), _I, _I, _I, _P, _S, C.POINTER(C.c_double), _P]),
    "mocha_encoder_workspace_bytes": (_S, [C.POINTER(Dims), _I]),
    "mocha_encoder_fwd": (_I, [C.POINTER(GeneratorWeights), _P, _I, _P, _I, _P, _S, _P]),
    "mocha_cnt_features": (_I, [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _P]),
    "mocha_attention_core": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P, _I, _P]),
    "mocha_block_tail": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _F, _P, _P, _I, _P]),
    "mocha_decoder_workspace_bytes": (_S, [C.POINTER(Dims), _I]),
    "mocha_decoder_fwd": (_I, [C.POINTER(GeneratorWeights), _P, _P, _I, _P, _I, _P, _S, _P]),
    "mocha_to_mot_workspace_bytes": (_S, [C.POINTER(Dims), _I]),
    "mocha_to_mot_fwd": (_I, [C.POINTER(GeneratorWeights), _P, _I, _P, _P, _P, _P, _I, _P, _S, _P]),
    "mocha_cvae_workspace_bytes": (_S, [C.POINTER(CvaeWeights), _I, _I]),
    "mocha_cvae_sample": (_I, [C.POINTER(CvaeWeights), _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P, _S, _P]),
    "mocha_cvae_precompute_dec0": (_I, [C.POINTER(CvaeWeights), _P, _P, _S, _P]),
    "mocha_cvae_condition": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "mocha_match_exact_workspace_bytes": (_S, [_I, _L, _I]),
    "mocha_match_exact": (_I, [_P, _I, _P, _L, _I, _I, _L, _P, _P, _P, _S, _P]),
    "mocha_match_tc_workspace_bytes": (_S, [_I, _L, _I, _I]),
    "mocha_match_tc": (_I, [_P, _P, _I, _P, _P, _P, _L, _I, _I, _I, _L, _P, _P, _P, _S, _P]),
    "mocha_db_norms_f32": (_I, [_P, _L, _I, _P, _P]),
    "mocha_db_pack_bf16": (_I, [_P, _L, _I, _P, _P, _P]),
    "mocha_topk_merge": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "mocha_topk_exchange_bytes": (_S, [_I, _I, _I]),
    "mocha_peer_alloc": (_I, [_S, C.POINTER(C.c_void_p), C.c_char_p]),
    "mocha_peer_open": (_I, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "mocha_peer_close": (_I, [_P]),
    "mocha_peer_free": (_I, [_P]),
    "mocha_topk_exchange_merge": (_I, [_P, _P, _I, _I, _I, _I, _P, C.c_uint, _P, _P, _P]),
    "mocha_linear": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _S, _P]),
    "mocha_linear_workspace_bytes": (_S, [_I, _I, _I, _I]),
    "mocha_xy_to_quat": (_I, [_P, _L, _P, _P]),
    "mocha_quat_to_xy": (_I, [_P, _L, _P, _P]),
    "mocha_fk": (_I, [_P, _P, _P, _L, _I, _P, _P, _P]),
    "mocha_fk_vel": (_I, [_P, _P, _P, _P, _P, _L, _I, _P, _P, _P, _P, _P]),
    "mocha_ik": (_I, [_P, _P, _P, _L, _I, _P, _P, _P]),
    "mocha_fk_f64": (_I, [_P, _P, _P, _L, _I, _P, _P, _P]),
    "mocha_fk_vel_f64": (_I, [_P, _P, _P, _P, _P, _L, _I, _P, _P, _P, _P, _P]),
    "mocha_ik_f64": (_I, [_P, _P, _P, _L, _I, _P, _P, _P]),
    "mocha_post_frame": (_I, [C.POINTER(PostParams), _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "mocha_window_features": (_I, [_P, _P, _P, _P, _L, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mocha_source_windows": (_I, [_P, _P, _P, _P, _P, _L, _P, _P, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P, _I, _P, _P, _I,
                                  _P, _P]),
    "mocha_record_frames": (_I, [_P, _P, _I, _P, _P, _P, _I, _P, _P, _I, _I, _P, _L, _P, _P, _P]),
    "mocha_clip_payload": (_I, [_P, _L, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P, _I, _I, _P, _P, _P, _P, _P, _P]),
    "mocha_quat_op": (_I, [_I, _I, _P, _P, _L, C.c_double, _P, _P]),
    "mocha_fk_chain": (_I, [_I, _P, _P, _P, _P, _L, _I, _P, _P, _P]),
    "mocha_post_frame_packed": (_I, [C.POINTER(PostParams), _P, _P, _I, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "mocha_post_frame_packed_masked": (_I, [C.POINTER(PostParams), _P, _P, _I, _P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "mocha_seed_rows": (_I, [_P, _P, _I, _P, _L, _L, _P, _I, _P]),
    "mocha_contact_update": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _D, _D, _D, _D, _P]),
    "mocha_ik_two_bone": (_I, [_P] * 10 + [_D, _L, _P, _P, _P]),
    "mocha_pose_transition": (_I, [_P] * 16 + [_L, _I, _P, _P, _P, _P, _P]),
    "mocha_pose_update": (_I, [_P] * 16 + [_D, _D, _L, _I, _P]),
}

_lib = None


def load():
    """Load the shared library (once) and bind every declared symbol. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MochaError(
            f"{LIB_PATH} is missing: build it with `python -m mocha_sigasia2023_b200.build` "
            "(there is no CPU / PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    sizes = (C.c_size_t * 10)()
    if lib.mocha_struct_sizes(sizes, 10) != 0:
        raise MochaError("mocha_struct_sizes failed")
    for st, sz in zip(_STRUCTS, sizes):
        if C.sizeof(st) != sz:
            raise MochaError(f"ABI mismatch: {st.__name__} is {C.sizeof(st)} B in Python, {sz} B in C")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mocha_last_error()
        raise MochaError(f"{what or 'mocha call'} failed ({rc}): {msg.decode() if msg else ''}")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require_cuda(*tensors):
    import torch
    for t in tensors:
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise MochaError("mocha_sigasia2023_b200 kernels need CUDA tensors (no CPU fallback)")
        if not t.is_contiguous():
            raise MochaError("tensor must be contiguous")
