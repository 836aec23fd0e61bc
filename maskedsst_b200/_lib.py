"""ctypes binding of libmsst.so (include/msst.h).  There is NO fallback: if the CUDA library is missing or
fails to load, every op raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmsst.so")

PREC_FP32, PREC_BF16 = 0, 1

u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p


RAW_I16, RAW_U16, RAW_F32 = 0, 1, 2


class RawInput(C.Structure):   # msst_raw_input
    _fields_ = [("tiles", vp), ("dtype", C.c_int), ("raw_bands", C.c_int), ("tile_h", C.c_int), ("tile_w", C.c_int),
                ("y0", C.c_int), ("x0", C.c_int), ("mean", vp), ("std", vp), ("clip", C.c_int), ("clip_lo", C.c_float),
                ("clip_hi", C.c_float), ("win_y", C.c_int), ("win_x", C.c_int), ("stride_y", C.c_int), ("stride_x", C.c_int),
                ("win_first", C.c_int)]


class EmbedDims(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("G", C.c_int), ("p0", C.c_int), ("p1", C.c_int), ("D", C.c_int),
                ("n_weight_blocks", C.c_int), ("drop_p", C.c_float), ("seed", C.c_uint64), ("seed_dev", vp),
                ("raw", C.POINTER(RawInput))]


class LinearDims(C.Structure):
    _fields_ = [("M", C.c_int64), ("N", C.c_int), ("K", C.c_int), ("act", C.c_int), ("drop_p", C.c_float),
                ("seed", C.c_uint64), ("site", C.c_uint32), ("prec", C.c_int), ("seed_dev", vp), ("y_fp32", C.c_int)]


class AttnDims(C.Structure):
    _fields_ = [("n_seq", C.c_int64), ("N", C.c_int), ("inner", C.c_int), ("H", C.c_int), ("dh", C.c_int),
                ("drop_p", C.c_float), ("seed", C.c_uint64), ("site", C.c_uint32), ("prec", C.c_int), ("seed_dev", vp)]


class LayerPtrs(C.Structure):   # msst_layer_params and msst_layer_grads share this layout
    _fields_ = [(n, vp) for n in ("ln1_w", "ln1_b", "w_qkv", "w_out", "b_out", "ln2_w", "ln2_b", "w1", "b1", "w2", "b2")]


class TfDims(C.Structure):
    _fields_ = [("n_seq", C.c_int64), ("N", C.c_int), ("inner", C.c_int), ("D", C.c_int), ("H", C.c_int), ("dh", C.c_int),
                ("M", C.c_int), ("L", C.c_int), ("drop_p", C.c_float), ("seed", C.c_uint64), ("site_base", C.c_uint32),
                ("prec", C.c_int), ("save_for_backward", C.c_int), ("seed_dev", vp)]


class HeadDims(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("G", C.c_int), ("p1", C.c_int), ("D", C.c_int), ("nc", C.c_int)]


class SceneDims(C.Structure):   # msst_scene_dims
    _fields_ = [(n, C.c_int) for n in ("B", "nc", "H", "W", "win", "stride_y", "stride_x", "win_y", "win_x", "win_first", "n")]


class SceneEmbedDims(C.Structure):   # msst_scene_embed_dims
    _fields_ = [(n, C.c_int) for n in ("B", "D", "H", "W", "win", "stride_y", "stride_x", "win_y", "win_x", "win_first", "n", "C", "p1")]


class SceneReconstructDims(C.Structure):   # msst_scene_reconstruct_dims
    _fields_ = [(n, C.c_int) for n in ("B", "D", "H", "W", "win", "stride_y", "stride_x", "win_y", "win_x", "win_first", "n", "C", "p0",
                                       "p1", "n_wb")]


class SceneAttributeDims(C.Structure):   # msst_scene_attribute_dims
    _fields_ = [(n, C.c_int) for n in ("B", "bands", "H", "W", "win", "stride_y", "stride_x", "win_y", "win_x", "win_first", "n", "steps")]


class KnnDims(C.Structure):   # msst_knn_dims
    _fields_ = [("n_ref", C.c_int64), ("n_query", C.c_int64), ("dim", C.c_int), ("k", C.c_int)]


class LinprobeDims(C.Structure):   # msst_linprobe_dims
    _fields_ = [("n", C.c_int64), ("dim", C.c_int), ("nc", C.c_int), ("heads", C.c_int), ("batch", C.c_int), ("step", C.c_int),
                ("lr", C.c_float * 16), ("wd", C.c_float * 16)]


class KmeansDims(C.Structure):   # msst_kmeans_dims
    _fields_ = [("n", C.c_int64), ("dim", C.c_int), ("k", C.c_int), ("restarts", C.c_int), ("normalize", C.c_int)]


class DecodeDims(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("G", C.c_int), ("p0", C.c_int), ("p1", C.c_int), ("D", C.c_int),
                ("nm", C.c_int), ("n_weight_blocks", C.c_int), ("raw", C.POINTER(RawInput))]


class MaskGenDims(C.Structure):
    _fields_ = [("B", C.c_int), ("C", C.c_int), ("rand_size", C.c_int), ("scale", C.c_int), ("mask_count", C.c_int), ("nm", C.c_int),
                ("tube", C.c_int), ("seed", C.c_uint64), ("seed_dev", vp)]


class AdamArgs(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("decoupled", C.c_int), ("clamp", C.c_float), ("grad_scale", C.c_float),
                ("step", C.c_int), ("step_dev", vp)]


# name -> (restype, argtypes); kept in sync with include/msst.h (tests/test_abi.py checks the export list)
SIGNATURES = {
    "msst_last_error": (C.c_char_p, []),
    "msst_version": (C.c_int, []),
    "msst_launch_count": (C.c_longlong, []),
    "msst_patch_embed_fwd": (C.c_int, [C.POINTER(EmbedDims)] + [vp] * 12 + [vp]),
    "msst_patch_embed_bwd": (C.c_int, [C.POINTER(EmbedDims)] + [vp] * 18 + [vp]),
    "msst_patch_embed_bwd_data": (C.c_int, [C.POINTER(EmbedDims)] + [vp] * 11 + [vp]),
    "msst_layernorm_fwd": (C.c_int, [vp, vp, vp, vp, C.c_int, vp, C.c_int64, C.c_int, C.c_float, vp]),
    "msst_layernorm_bwd": (C.c_int, [vp] * 8 + [C.c_int64, C.c_int, vp]),
    "msst_linear_fwd": (C.c_int, [C.POINTER(LinearDims)] + [vp] * 6 + [vp]),
    "msst_linear_bwd_data": (C.c_int, [C.POINTER(LinearDims)] + [vp] * 5 + [vp]),
    "msst_linear_bwd_weight": (C.c_int, [C.POINTER(LinearDims)] + [vp] * 4 + [vp]),
    "msst_dropout_apply": (C.c_int, [vp, vp, C.c_int64, C.c_float, C.c_uint64, C.c_uint32, vp, vp]),
    "msst_attention_fwd": (C.c_int, [C.POINTER(AttnDims), vp, vp, vp, vp]),
    "msst_attention_bwd": (C.c_int, [C.POINTER(AttnDims)] + [vp] * 5 + [vp]),
    "msst_attn_block_fwd": (C.c_int, [C.POINTER(AttnDims), C.c_int, vp, vp, vp, vp, vp]),
    "msst_attn_block_out_fwd": (C.c_int, [C.POINTER(AttnDims), C.c_int] + [vp] * 12 + [C.c_uint32, vp]),
    "msst_attn_block_bwd": (C.c_int, [C.POINTER(AttnDims), C.c_int] + [vp] * 7 + [vp]),
    "msst_mlp_block_fwd": (C.c_int, [vp] * 13 + [C.c_int64, C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint32, C.c_uint32, vp, vp]),
    "msst_mlp_block_bwd": (C.c_int, [vp] * 10 + [C.c_int64, C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint32, vp, vp]),
    "msst_transformer_workspace_bytes": (C.c_int64, [C.POINTER(TfDims)]),
    "msst_transformer_fwd": (C.c_int, [C.POINTER(TfDims), C.POINTER(LayerPtrs), vp, vp, vp, vp]),
    "msst_transformer_bwd": (C.c_int, [C.POINTER(TfDims), C.POINTER(LayerPtrs), C.POINTER(LayerPtrs), vp, vp, vp, vp, vp]),
    "msst_head_fwd": (C.c_int, [C.POINTER(HeadDims)] + [vp] * 6 + [vp]),
    "msst_head_bwd": (C.c_int, [C.POINTER(HeadDims)] + [vp] * 10 + [vp]),
    "msst_cross_entropy_fwd_bwd": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "msst_scene_blend": (C.c_int, [C.POINTER(SceneDims), vp, vp, vp, vp, vp]),
    "msst_scene_embed": (C.c_int, [C.POINTER(SceneEmbedDims), vp, vp, vp, vp, vp]),
    "msst_scene_reconstruct": (C.c_int, [C.POINTER(SceneReconstructDims)] + [vp] * 7 + [vp]),
    "msst_scene_attribute": (C.c_int, [C.POINTER(SceneAttributeDims)] + [vp] * 4 + [vp]),
    "msst_knn_prepare": (C.c_int, [vp, C.c_int64, C.c_int, vp, vp]),
    "msst_knn_topk": (C.c_int, [C.POINTER(KnnDims), vp, vp, vp, vp, vp]),
    "msst_knn_vote": (C.c_int, [C.c_int64, C.c_int, C.c_int64, vp, vp, vp, C.c_int, C.c_float, vp, vp, vp]),
    "msst_linprobe_workspace": (C.c_int64, [C.POINTER(LinprobeDims)]),
    "msst_linprobe_grad": (C.c_int, [C.POINTER(LinprobeDims), vp, vp, vp, vp, vp, vp]),
    "msst_linprobe_update": (C.c_int, [C.POINTER(LinprobeDims), vp, vp, vp, vp, vp, vp]),
    "msst_linprobe_predict": (C.c_int, [C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp, vp]),
    "msst_kmeans_workspace": (C.c_int64, [C.POINTER(KmeansDims)]),
    "msst_kmeans_seed": (C.c_int, [C.POINTER(KmeansDims), C.c_int, vp, vp, vp, vp, vp, vp, vp]),
    "msst_kmeans_assign": (C.c_int, [C.POINTER(KmeansDims), vp, vp, vp, vp, vp, vp]),
    "msst_kmeans_update": (C.c_int, [C.POINTER(KmeansDims), vp, vp, vp, vp, vp, vp]),
    "msst_moments_workspace": (C.c_int64, [C.c_int64, C.c_int]),
    "msst_moments_mean": (C.c_int, [C.c_int64, C.c_int, vp, vp, vp, vp]),
    "msst_moments_cov": (C.c_int, [C.c_int64, C.c_int, vp, vp, vp, vp, vp]),
    "msst_moments_project": (C.c_int, [C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    "msst_simmim_decode_l1_fwd": (C.c_int, [C.POINTER(DecodeDims)] + [vp] * 9 + [vp]),
    "msst_simmim_decode_l1_bwd": (C.c_int, [C.POINTER(DecodeDims)] + [vp] * 11 + [vp]),
    "msst_draw_masks": (C.c_int, [C.POINTER(MaskGenDims), vp, vp, vp]),
    "msst_adam_step": (C.c_int, [C.POINTER(AdamArgs), vp, vp, vp, vp, vp, C.c_int64, vp]),
}

_lib = None


def lib():
    """Loads libmsst.so once (building it first if nvcc is present and it is stale/missing)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("MSST_LIB", LIB_PATH)   # A/B runs of two builds of the library (profiling only)
    if path == LIB_PATH:
        from . import build as _build
        _build.build()   # no-op when the in-tree library is up to date (source digest) or nvcc is absent
    try:
        L = C.CDLL(path)
    except OSError as e:   # fail loudly: there is no CPU / eager fallback
        raise RuntimeError(f"maskedsst_b200: cannot load {LIB_PATH}: {e}. Run `python -m maskedsst_b200.build`.") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


class MsstError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = lib().msst_last_error()
        raise MsstError(f"libmsst error {rc}: {msg.decode() if msg else '?'}")
