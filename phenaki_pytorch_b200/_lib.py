"""ctypes binding of libphk.so (include/phk.h).  There is NO fallback: if the CUDA library is
missing or a call fails, the product raises -- it never routes through PyTorch ops or the oracle."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PHK_LIB") or os.path.join(_HERE, "libphk.so")  # PHK_LIB: an A/B build of the same ABI (tools/ only)

PREC_F32, PREC_BF16, PREC_BF16X3 = 0, 1, 2
LN_STAT_BYTES, LN_COUNTERS = 2 * 148 * 128 * 8, 160   # phk_gemm_bf16_ln_ws scratch (include/phk.h)


def default_precision():
    """Precision mode new modules start in: `PHK_PREC` = f32 | bf16 | bf16x3 (unset: the module default below).
    f32    fp32 FFMA products -- the reference's fp32 arithmetic, token ids identical (slowest)
    bf16x3 split-bf16 products on tcgen05 -- ids identical at the same bars, 4.3x faster than f32
    bf16   bf16 products on tcgen05 -- the reference's autocast(bfloat16) dtype flow, 3x faster again (benchmarked mode)
    `model.precision = _lib.PREC_*` switches a module at any time."""
    name = os.environ.get("PHK_PREC", DEFAULT_PRECISION_NAME).lower()
    return {"f32": PREC_F32, "fp32": PREC_F32, "bf16": PREC_BF16, "bf16x3": PREC_BF16X3}.get(name, PREC_BF16X3)


DEFAULT_PRECISION_NAME = "bf16x3"  # exact token ids on the tensor cores (round 2; the whole CPU and GPU suites pass under it)

c_f = C.c_void_p  # device pointers travel as void*


class AttnT(C.Structure):
    _fields_ = [("norm_g", c_f), ("norm_b", c_f), ("ctx_g", c_f), ("ctx_b", c_f), ("null_kv", c_f),
                ("q_scale", c_f), ("k_scale", c_f), ("wq", c_f), ("wkv", c_f), ("wo", c_f),
                ("wq_h", c_f), ("wkv_h", c_f), ("wo_h", c_f),
                ("num_null_kv", C.c_int32), ("dim_context", C.c_int32)]


class FFT(C.Structure):
    _fields_ = [("ln_g", c_f), ("ln_b", c_f), ("w1", c_f), ("w2", c_f), ("w1_h", c_f), ("w2_h", c_f),
                ("inner", C.c_int32), ("inner_pad", C.c_int32)]


class PegT(C.Structure):
    _fields_ = [("w", c_f), ("b", c_f), ("causal", C.c_int32), ("_pad", C.c_int32)]


class LayerT(C.Structure):
    _fields_ = [("has_peg", C.c_int32), ("has_cross", C.c_int32), ("peg", PegT), ("self_attn", AttnT),
                ("cross_attn", AttnT), ("ff", FFT)]


class TransformerT(C.Structure):
    _fields_ = [("dim", C.c_int32), ("heads", C.c_int32), ("dim_head", C.c_int32), ("depth", C.c_int32),
                ("causal", C.c_int32), ("_pad", C.c_int32), ("layers", C.POINTER(LayerT)),
                ("out_g", c_f), ("out_b", c_f), ("alibi_slopes", c_f)]


class CpbT(C.Structure):
    _fields_ = [("w0", c_f), ("b0", c_f), ("w1", c_f), ("b1", c_f), ("w2", c_f), ("b2", c_f),
                ("num_dims", C.c_int32), ("hidden", C.c_int32), ("heads", C.c_int32), ("_pad", C.c_int32)]


class CvivitT(C.Structure):
    _fields_ = [("dim", C.c_int32), ("heads", C.c_int32), ("dim_head", C.c_int32), ("channels", C.c_int32),
                ("image_h", C.c_int32), ("image_w", C.c_int32), ("patch_h", C.c_int32), ("patch_w", C.c_int32),
                ("patch_t", C.c_int32), ("codebook_bits", C.c_int32), ("_pad0", C.c_int32), ("_pad1", C.c_int32),
                ("pf_ln1_g", c_f), ("pf_ln1_b", c_f), ("pf_w", c_f), ("pf_b", c_f), ("pf_ln2_g", c_f),
                ("pf_ln2_b", c_f), ("pf_w_h", c_f),
                ("pr_ln1_g", c_f), ("pr_ln1_b", c_f), ("pr_w", c_f), ("pr_b", c_f), ("pr_ln2_g", c_f),
                ("pr_ln2_b", c_f), ("pr_w_h", c_f),
                ("spatial_bias", CpbT), ("spatial", TransformerT), ("temporal", TransformerT),
                ("vq_w", c_f), ("vq_b", c_f),
                ("codebook", c_f), ("codebook_h", c_f), ("codebook_size", C.c_int32), ("_pad2", C.c_int32)]


class CvivitDecT(C.Structure):
    _fields_ = [("dim", C.c_int32), ("heads", C.c_int32), ("dim_head", C.c_int32), ("channels", C.c_int32),
                ("image_h", C.c_int32), ("image_w", C.c_int32), ("patch_h", C.c_int32), ("patch_w", C.c_int32),
                ("patch_t", C.c_int32), ("codebook_bits", C.c_int32),
                ("vq_out_w", c_f), ("vq_out_b", c_f),
                ("spatial_bias", CpbT), ("temporal", TransformerT), ("spatial", TransformerT),
                ("px_first_w", c_f), ("px_first_b", c_f), ("px_first_w_h", c_f),
                ("px_w", c_f), ("px_b", c_f), ("px_w_h", c_f)]


class MaskgitT(C.Structure):
    _fields_ = [("dim", C.c_int32), ("heads", C.c_int32), ("dim_head", C.c_int32), ("num_tokens", C.c_int32),
                ("max_seq_len", C.c_int32), ("is_critic", C.c_int32), ("has_bias", C.c_int32), ("_pad", C.c_int32),
                ("shrink_alpha", C.c_float), ("_padf", C.c_float),
                ("token_emb", c_f), ("pos_emb", c_f), ("pos_bias", CpbT), ("transformer", TransformerT),
                ("head_w", c_f), ("head_b", c_f), ("head_w_h", c_f)]


class AttnGeomT(C.Structure):
    _fields_ = [("n_outer", C.c_int32), ("n_inner", C.c_int32), ("n_q", C.c_int32), ("n_k", C.c_int32),
                ("heads", C.c_int32), ("dim_head", C.c_int32), ("num_null_kv", C.c_int32), ("causal", C.c_int32),
                ("q_outer", C.c_int64), ("q_inner", C.c_int64), ("q_tok", C.c_int64),
                ("k_outer", C.c_int64), ("k_inner", C.c_int64), ("k_tok", C.c_int64),
                ("o_outer", C.c_int64), ("o_inner", C.c_int64), ("o_tok", C.c_int64),
                ("kv_outer_mod", C.c_int32), ("mask_outer_mod", C.c_int32), ("mask_off_from", C.c_int32),
                ("out_bf16", C.c_int32), ("scale", C.c_float), ("_pad", C.c_int32)]


i32, i64, f32, u64, vp = C.c_int32, C.c_int64, C.c_float, C.c_uint64, C.c_void_p

# name -> argtypes (restype int unless listed in _RESTYPES); mirrors include/phk.h one to one
PROTOTYPES = {
    "phk_version": [],
    "phk_last_error": [],
    "phk_launch_count": [],
    "phk_prof_enable": [i32],
    "phk_prof_collect": [C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(C.c_double), i32],
    "phk_layernorm": [vp, vp, vp, vp, vp, i64, i32, i32, i64, i64, i64, vp],
    "phk_patchify_ln": [vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, i32, vp],
    "phk_gemm_f32": [vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp, i64, i64, i64, vp],
    "phk_gemm_bf16": [vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp, i64, i64, i64, i32, vp],
    "phk_gemm_bf16_x2": [vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp],
    "phk_debug_gemm_trace": [vp],
    "phk_debug_gemm_mode": [i32],
    "phk_debug_static_weights": [i32],
    "phk_debug_attention_tc_variant": [i32],
    "phk_geglu": [vp, vp, i64, i32, vp],
    "phk_attention": [vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(AttnGeomT), vp],
    "phk_attention_tc_scratch_bytes": [i32, i32, i32],
    "phk_attention_tc": [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, vp, i64, vp],
    "phk_attention_tc_bf16": [vp, i64, vp, i64, vp, vp, i32, i32, i32, vp],
    "phk_attention_small_bf16": [vp, vp, vp, vp, C.POINTER(AttnGeomT), vp],
    "phk_attention_mid_bf16": [vp, i64, vp, i64, vp, vp, i32, i32, i32, vp],
    "phk_gemm_bf16_ln": [vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp, vp, f32, vp, vp, i64, vp],
    "phk_gemm_bf16_ln_ws": [vp, i64, vp, i64, vp, i64, i64, i32, i32, vp, vp, vp, f32, vp, vp, i64, vp, vp, vp],
    "phk_train_set_progress_events": [vp, i32],
    "phk_split3": [vp, i64, vp, i64, i32, i32, vp],
    "phk_cross_kv_pack": [vp, vp, vp, i32, vp, i32, i32, i32, i32, vp, vp, vp],
    "phk_gemm_bf16_qnorm": [vp, i64, vp, i64, vp, i64, i32, i32, vp, f32, vp],
    "phk_attention_cross_packed": [vp, i64, vp, vp, vp, i64, i32, i32, i32, i32, i32, i32, vp],
    "phk_gemm_bf16_qkv": [vp, vp, i64, vp, vp, i64, vp, vp, i64, i32, i32, vp, vp, f32, vp],
    "phk_peg3d": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp],
    "phk_cpb_scratch_floats": [C.POINTER(CpbT), i32, i32, i32],
    "phk_cpb_bias": [C.POINTER(CpbT), i32, i32, i32, vp, vp, vp],
    "phk_lfq_ids": [vp, vp, vp, vp, vp, i64, i32, i32, vp],
    "phk_layernorm_lfq": [vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp],
    "phk_lfq_codes": [vp, vp, vp, vp, i64, i32, i32, vp],
    "phk_unpatchify": [vp, i64, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp],
    "phk_token_embed": [vp, vp, vp, vp, i32, i32, i32, i32, f32, i32, vp],
    "phk_sample_tokens": [vp, vp, i64, vp, u64, u64, f32, f32, vp, vp, vp, vp, i64, i32, i64, i64, i64, vp],
    "phk_topk_mask": [vp, i32, i32, i32, vp, vp, i64, vp],
    "phk_critic_scores": [vp, vp, vp, vp, vp, f32, f32, f32, vp, i64, i32, i64, i64, i64, vp],
    "phk_cfg_combine": [vp, vp, f32, vp, i64, vp],
    "phk_cvivit_workspace_bytes": [C.POINTER(CvivitT), i32, i32, i32],
    "phk_cvivit_encode": [C.POINTER(CvivitT), vp, i32, i32, vp, vp, i64, i32, vp, vp, vp, vp, vp, vp],
    "phk_cvivit_encode_host": [C.POINTER(CvivitT), vp, i32, i32, vp, vp, vp, vp, i64, i32, vp, vp],
    "phk_encode_pipe_create": [C.POINTER(vp), i32],
    "phk_encode_pipe_destroy": [vp],
    "phk_encode_pipe_submit": [vp, C.POINTER(CvivitT), vp, i32, i32, vp, vp, vp, vp, i64, i32, vp, vp, C.POINTER(i64)],
    "phk_encode_pipe_wait": [vp, i64],
    "phk_cvivit_decode_workspace_bytes": [C.POINTER(CvivitDecT), i32, i32, i32],
    "phk_cvivit_decode": [C.POINTER(CvivitDecT), vp, vp, i32, i32, vp, vp, i64, i32, vp, vp, vp, vp, vp],
    "phk_maskgit_context_kv": [C.POINTER(MaskgitT), vp, i32, i32, vp, vp, i32, vp],
    "phk_maskgit_workspace_bytes": [C.POINTER(MaskgitT), i32, i32, i32, i32, i32],
    "phk_head_sample_scratch_bytes": [i32],
    "phk_layernorm_cfg": [vp, vp, vp, vp, f32, vp, i64, i32, vp],
    "phk_head_sample": [vp, i64, i64, vp, i64, vp, i32, i32, i32, f32, u64, u64, vp, vp, vp, vp, vp, i64, vp],
    "phk_maskgit_sample_workspace_bytes": [C.POINTER(MaskgitT), i32, i32, i32],
    "phk_maskgit_demask_iteration_critic_workspace_bytes": [C.POINTER(MaskgitT), C.POINTER(MaskgitT), i32, i32, i32],
    "phk_maskgit_sample_step": [C.POINTER(MaskgitT), vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, vp, f32, f32, u64,
                                u64, vp, vp, vp, vp, i32, vp, i64, vp],
    "phk_sample_tail_scratch_bytes": [i32, i32, i32],
    "phk_sample_tail_rows": [vp, vp, vp, vp, f32, vp, i64, vp, i32, i32, i32, i32, i32, f32, u64, u64, vp, vp, vp, vp, vp, i32,
                             i32, vp, i64, vp],
    "phk_maskgit_sample_step_primed": [C.POINTER(MaskgitT), vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, f32, f32, u64, u64,
                                       vp, vp, vp, vp, i32, i32, vp, i64, vp],
    "phk_sample_tail": [vp, vp, vp, vp, f32, vp, i64, vp, i32, i32, i32, i32, i32, f32, u64, u64, vp, vp, vp, vp, vp, vp,
                        i64, vp],
    "phk_head_sample_rng": [vp, i64, i64, vp, i64, vp, i32, i32, i32, f32, u64, u64, vp, vp, vp, vp, vp, vp, i64, vp],
    "phk_rng_advance": [vp, u64, vp],
    "phk_noise_probe": [vp, u64, u64, i64, vp, vp, vp],
    "phk_debug_step_graph": [i32],
    "phk_vq_cosine_scratch_bytes": [i64, i32, i32],
    "phk_vq_cosine_ids": [vp, vp, vp, vp, i64, i32, i32, vp, i64, i32, vp],
    "phk_maskgit_demask_iteration": [C.POINTER(MaskgitT), vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, f32, f32,
                                     vp, i32, vp, i64, vp],
    "phk_maskgit_demask_iteration_critic": [C.POINTER(MaskgitT), C.POINTER(MaskgitT), vp, vp, vp, vp, vp, vp, vp, i32, i32, i32,
                                            i32, i32, i32, vp, vp, i32, vp, vp, f32, f32, vp, i32, vp, f32, f32, i32, vp, i64, vp],
    "phk_maskgit_forward": [C.POINTER(MaskgitT), vp, i32, i32, i32, i32, i32, vp, i32, vp, vp, i32, i32, vp, vp,
                            vp, i64, i32, vp],
    "phk_maskgit_train_workspace_bytes": [C.POINTER(MaskgitT), i32, i32, i32, i32, i32],
    "phk_maskgit_train_step": [C.POINTER(MaskgitT), C.POINTER(MaskgitT), vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, i32,
                               vp, vp, f32, vp, vp, vp, i64, i32, vp],
}
_RESTYPES = {"phk_attention_tc_scratch_bytes": i64, "phk_head_sample_scratch_bytes": i64,
             "phk_maskgit_sample_workspace_bytes": i64, "phk_maskgit_demask_iteration_critic_workspace_bytes": i64, "phk_sample_tail_scratch_bytes": i64, "phk_vq_cosine_scratch_bytes": i64, "phk_maskgit_train_workspace_bytes": i64, "phk_last_error": C.c_char_p, "phk_launch_count": i64, "phk_cpb_scratch_floats": i64,
             "phk_cvivit_workspace_bytes": i64, "phk_cvivit_decode_workspace_bytes": i64, "phk_maskgit_workspace_bytes": i64}

FAMILIES = ["patchify_ln", "layernorm", "gemm_f32", "gemm_bf16", "attention", "peg", "geglu", "lfq", "embed",
            "cpb", "sample_tokens", "topk_mask", "critic", "cfg_combine"]

_lib = None


class PhkError(RuntimeError):
    pass


def lib():
    """Loads libphk.so once.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PhkError(f"{LIB_PATH} is missing: build it with `python -m phenaki_pytorch_b200.build` "
                           "(there is no CPU / PyTorch fallback)")
        l = C.CDLL(LIB_PATH)
        for name, argtypes in PROTOTYPES.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, C.c_int)
        _lib = l
    return _lib


def check(rc, what=""):
    """Maps the C return convention to exceptions (shape contract -> AssertionError as in the reference)."""
    if rc == 0:
        return
    msg = lib().phk_last_error().decode() if rc < 0 else f"CUDA error {rc}"
    if rc == -2:
        raise AssertionError(f"{what}: {msg}")
    raise PhkError(f"{what}: {msg} (code {rc})")


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require_cuda(t, name, dtype=None):
    if not t.is_cuda:
        raise PhkError(f"{name} must live on a CUDA device: this framework has no CPU path")
    if dtype is not None and t.dtype != dtype:
        raise PhkError(f"{name} must be {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def profile_collect():
    """{family: (total_ms, calls, work)} recorded since phk_prof_enable(1)."""
    n = len(FAMILIES)
    ms, calls, work = (C.c_double * n)(), (i64 * n)(), (C.c_double * n)()
    check(lib().phk_prof_collect(ms, calls, work, n), "phk_prof_collect")
    return {FAMILIES[i]: (ms[i], calls[i], work[i]) for i in range(n) if calls[i]}
