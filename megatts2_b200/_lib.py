"""ctypes binding of libmegatts2_b200.so (see include/megatts2_b200.h).

The library is the product: if it is missing this module raises - there is no
CPU / PyTorch fallback anywhere in the package.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmegatts2_b200.so")

ABI_VERSION = 4
ACT_NONE, ACT_RELU, ACT_LEAKY, ACT_TANH = 0, 1, 2, 3
TC_BF16X3, TC_F16X2 = 0, 1
PAD_ZERO, PAD_REFLECT, PAD_REPLICATE = 0, 1, 2

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class ConvParams(C.Structure):
    _fields_ = [
        ("x", vp), ("x_batch_stride", i64), ("ldx", i32),
        ("w", vp), ("bias", vp),
        ("res", vp), ("res_batch_stride", i64), ("ldr", i32),
        ("y", vp), ("y_batch_stride", i64), ("ldy", i32),
        ("B", i32), ("Tin", i32), ("Tout", i32), ("Cin", i32), ("Cout", i32),
        ("k", i32), ("stride", i32), ("dil", i32), ("pad", i32),
        ("pad_mode", i32),
        ("pre_act", i32), ("pre_slope", f32),
        ("post_act", i32), ("post_slope", f32),
        ("out_scale", f32), ("accumulate", i32),
        ("out_shift", i64), ("y_batch_elems", i64),
        ("in_lens", vp),
        ("w_tc", vp), ("tc_scratch", vp), ("tc_scratch_bytes", i64), ("tc_rows_cap", i64),
        ("tc_presplit", i32), ("tc_out_planes", vp), ("tc_out_plane_stride", i64),
        ("tc_out_ld", i32), ("tc_out_tp", i32), ("tc_out_hl", i32), ("tc_out_act", i32), ("tc_out_slope", f32),
        ("tc_partial", vp), ("tc_partial_bytes", i64),
        ("tc_fmt", i32), ("tc_in_tp", i32), ("tc_in_row0", i32),
    ]


class AttnParams(C.Structure):
    _fields_ = [
        ("q", vp), ("q_sb", i64), ("q_st", i32),
        ("k", vp), ("k_sb", i64), ("k_st", i32),
        ("v", vp), ("v_sb", i64), ("v_st", i32),
        ("o", vp), ("o_sb", i64), ("o_st", i32),
        ("mask", vp), ("mask_sb", i64), ("mask_sh", i64), ("mask_sq", i64),
        ("B", i32), ("H", i32), ("Tq", i32), ("Tk", i32), ("dh", i32),
        ("scale", f32),
        ("o_planes", vp), ("o_plane_stride", i64), ("o_planes_ld", i32), ("o_planes_fmt", i32),
    ]


class EncoderLayer(C.Structure):
    _fields_ = [(n, vp) for n in (
        "ln1_g", "ln1_b", "ln2_g", "ln2_b", "w_qkv", "b_qkv", "w_o", "b_o",
        "w_ff1", "b_ff1", "w_ff2", "b_ff2", "w_qkv_tc", "w_o_tc", "w_ff1_tc", "w_ff2_tc")]


class Encoder(C.Structure):
    _fields_ = [("n_layers", i32), ("d_model", i32), ("n_heads", i32), ("ff_dim", i32), ("conv_ff", i32),
                ("engine", i32), ("layers", C.POINTER(EncoderLayer))]


class PLM(C.Structure):
    _fields_ = [("enc", Encoder), ("pc_embedding", vp), ("w_predict", vp), ("pe", vp), ("pe_alpha", f32),
                ("vq_bins", i32), ("vq_dim", i32), ("tc_dim", i32)]


class ADM(C.Structure):
    _fields_ = [("enc", Encoder), ("w_dt", vp), ("w_tc", vp), ("w_predict", vp), ("pe", vp), ("pe_alpha", f32),
                ("emb_dim", i32), ("tc_dim", i32), ("tc_emb_dim", i32)]


class ConvBlock(C.Structure):
    _fields_ = [("w", vp), ("b", vp), ("ln_g", vp), ("ln_b", vp), ("w_tc", vp)]


class ConvNet(C.Structure):
    _fields_ = [("in_channels", i32), ("out_channels", i32), ("hidden", i32), ("k", i32), ("n_stacks", i32),
                ("n_blocks", i32), ("engine", i32), ("w_first", vp), ("b_first", vp), ("w_last", vp), ("b_last", vp),
                ("blocks", C.POINTER(ConvBlock))]


class ConvNetDouble(C.Structure):
    _fields_ = [("in_channels", i32), ("out_channels", i32), ("hidden", i32), ("k", i32), ("n_layers", i32),
                ("n_stacks", i32), ("n_blocks", i32), ("engine", i32), ("middle_kind", i32), ("middle_k", i32),
                ("middle_stride", i32), ("middle_pad", i32), ("w_middle", vp), ("b_middle", vp),
                ("w_first", vp), ("b_first", vp), ("w_last", vp), ("b_last", vp),
                ("blocks", C.POINTER(ConvBlock))]


class HifiganResblock(C.Structure):
    _fields_ = [("w1", vp * 3), ("b1", vp * 3), ("w2", vp * 3), ("b2", vp * 3), ("k", i32), ("dil", i32 * 3),
                ("w1_tc", vp * 3), ("w2_tc", vp * 3)]


class Hifigan(C.Structure):
    _fields_ = [("in_channels", i32), ("ch0", i32), ("n_ups", i32), ("n_kernels", i32), ("inference_padding", i32),
                ("engine", i32), ("up_factor", i32 * 4), ("up_kernel", i32 * 4), ("w_pre", vp), ("b_pre", vp),
                ("w_up", vp * 4), ("b_up", vp * 4), ("w_up_tc", vp * 4), ("resblocks", C.POINTER(HifiganResblock)),
                ("w_post", vp), ("b_post", vp)]


# name -> (restype, argtypes); every symbol include/megatts2_b200.h declares
SIGNATURES = {
    "mtts_abi_version": (C.c_int, []),
    "mtts_last_error": (C.c_char_p, []),
    "mtts_launch_count": (i64, []),
    "mtts_profile_begin": (C.c_int, []),
    "mtts_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i64)]),
    "mtts_profile_split": (C.c_int, [C.POINTER(C.c_double)]),
    "mtts_trace_begin": (C.c_int, [vp]),
    "mtts_trace_end": (C.c_int, [C.c_char_p, i32]),
    "mtts_conv1d_f32": (C.c_int, [C.POINTER(ConvParams), vp]),
    "mtts_linear_tc_scratch_bytes": (i64, [i64, i32]),
    "mtts_linear_tc_f32": (C.c_int, [vp, i32, i64, i32, vp, i32, vp, vp, i32, vp, i32, i32, f32, i32, vp, i64, i64, i32, vp]),
    "mtts_split_planes_f32": (C.c_int, [vp, i32, i64, i32, vp, i32, vp]),
    "mtts_tc_overflow_bind": (C.c_int, [vp]),
    "mtts_tc_plan_query": (C.c_int, [i32, i32, i32, i32, i32, i32, i32, i32, i64, i32, C.POINTER(i32)]),
    "mtts_mask_tail_f32": (C.c_int, [vp, i32, i32, i32, vp, vp]),
    "mtts_resample_f32": (C.c_int, [vp, i64, i32, i32, vp, vp, i32, i32, i32, i32, vp, i64, i32, vp, vp]),
    "mtts_peak_normalize_f32": (C.c_int, [vp, i64, i32, i32, vp, vp, vp]),
    "mtts_pcm16_f32": (C.c_int, [vp, i64, vp, vp]),
    "mtts_bmm_f32": (C.c_int, [vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32, i32, i32, i32, i32,
                               f32, i32, vp]),
    "mtts_softmax_fwd_f32": (C.c_int, [vp, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp]),
    "mtts_softmax_bwd_f32": (C.c_int, [vp, vp, vp, vp, i32, i64, vp]),
    "mtts_layernorm_bwd_f32": (C.c_int, [vp, vp, vp, vp, vp, i64, i32, f32, vp]),
    "mtts_colsum_f32": (C.c_int, [vp, i64, i64, i32, vp, i32, vp]),
    "mtts_relu_bwd_f32": (C.c_int, [vp, vp, vp, i64, vp]),
    "mtts_embedding_bwd_f32": (C.c_int, [vp, vp, i64, i32, i32, vp, vp]),
    "mtts_rowdot_f32": (C.c_int, [vp, vp, i64, i32, i32, vp, vp]),
    "mtts_kmeans_assign_f32": (C.c_int, [vp, vp, i32, i32, i32, vp, vp]),
    "mtts_vq_cluster_sum_f32": (C.c_int, [vp, vp, i32, i32, i32, vp, vp, vp]),
    "mtts_kmeans_update_f32": (C.c_int, [vp, vp, vp, i32, i32, vp]),
    "mtts_vq_ema_update_f32": (C.c_int, [vp, vp, vp, vp, vp, i32, i32, f32, f32, vp, vp]),
    "mtts_vq_replace_rows_f32": (C.c_int, [vp, vp, vp, vp, f32, i32, i32, i32, vp]),
    "mtts_vq_ste_commit_f32": (C.c_int, [vp, vp, i64, vp, vp, vp, vp]),
    "mtts_vq_ste_commit_bwd_f32": (C.c_int, [vp, vp, vp, vp, f32, i64, vp, vp]),
    "mtts_layernorm_f32": (C.c_int, [vp, i32, vp, vp, vp, i32, vp, i32, i64, i32, f32, i32, i32, vp]),
    "mtts_attention_f32": (C.c_int, [C.POINTER(AttnParams), vp]),
    "mtts_vq_argmin_f32": (C.c_int, [vp, i32, vp, i64, i32, i32, vp, vp]),
    "mtts_vq_gather_f32": (C.c_int, [vp, i32, vp, i32, i32, i32, i32, i32, vp, i64, i32, vp]),
    "mtts_mel_spectrogram_f32": (C.c_int, [vp, i64, i32, i32, vp, vp, vp, vp, i32, f32, vp, i64, i64, i64, vp]),
    "mtts_mel_spectrogram_ragged_f32": (C.c_int, [vp, i64, i32, i32, vp, vp, vp, vp, vp, i32, f32, vp, i64, i64, i64, vp]),
    "mtts_maxpool_time_f32": (C.c_int, [vp, i64, i32, vp, i64, i32, i32, i32, i32, i32, vp]),
    "mtts_embed_pe_f32": (C.c_int, [vp, i32, vp, i32, i32, vp, f32, i32, i32, i32, vp, i64, i32, vp]),
    "mtts_add_pe_f32": (C.c_int, [vp, i64, i32, vp, f32, i32, i32, i32, vp, i64, i32, vp]),
    "mtts_length_regulate_f32": (C.c_int, [vp, i64, i32, vp, i32, i32, i32, i32, i32, vp, i64, i32, vp, vp]),
    "mtts_copy_strided_f32": (C.c_int, [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp]),
    "mtts_encoder_workspace_bytes": (i64, [C.POINTER(Encoder), i32, i32]),
    "mtts_encoder_forward_f32": (C.c_int, [C.POINTER(Encoder), vp, vp, i32, i32, vp, i64, i64, i64, i32, vp, i64, vp]),
    "mtts_plm_infer_workspace_bytes": (i64, [C.POINTER(PLM), i32, i32]),
    "mtts_plm_infer_f32": (C.c_int, [C.POINTER(PLM), vp, i64, i32, i32, i32, vp, vp, vp, i64, vp]),
    "mtts_adm_infer_workspace_bytes": (i64, [C.POINTER(ADM), i32, i32]),
    "mtts_adm_infer_f32": (C.c_int, [C.POINTER(ADM), vp, i64, i32, i32, i32, vp, vp, vp, i64, vp]),
    "mtts_plm_decode_causal_workspace_bytes": (i64, [C.POINTER(PLM), i32, i32]),
    "mtts_plm_decode_causal_f32": (C.c_int, [C.POINTER(PLM), vp, i64, i32, i32, i32, vp, vp, vp, i64, vp]),
    "mtts_adm_decode_causal_workspace_bytes": (i64, [C.POINTER(ADM), i32, i32]),
    "mtts_adm_decode_causal_f32": (C.c_int, [C.POINTER(ADM), vp, i64, i32, i32, i32, vp, vp, vp, i64, vp]),
    "mtts_convnet_workspace_bytes": (i64, [C.POINTER(ConvNet), i32, i32]),
    "mtts_convnet_forward_f32": (C.c_int, [C.POINTER(ConvNet), vp, i64, i32, vp, i64, i32, i32, i32, vp, i64, vp]),
    "mtts_convnet_double_out_len": (i32, [C.POINTER(ConvNetDouble), i32]),
    "mtts_convnet_double_workspace_bytes": (i64, [C.POINTER(ConvNetDouble), i32, i32]),
    "mtts_convnet_double_forward_f32": (C.c_int, [C.POINTER(ConvNetDouble), vp, i64, i32, vp, i64, i32, i32, i32, vp, i64, vp]),
    "mtts_hifigan_workspace_bytes": (i64, [C.POINTER(Hifigan), i32, i32]),
    "mtts_hifigan_forward_f32": (C.c_int, [C.POINTER(Hifigan), vp, i64, i32, i32, i32, vp, i64, vp, i64, vp]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C megatts2_b200/csrc` (there is no fallback path).")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)     # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        if handle.mtts_abi_version() != ABI_VERSION:
            raise RuntimeError("libmegatts2_b200.so ABI version mismatch")
        _lib = handle
    return _lib


class MttsError(RuntimeError):
    pass


def check(status):
    if status != 0:
        msg = lib().mtts_last_error()
        raise MttsError(f"libmegatts2_b200 error {status}: {msg.decode() if msg else ''}")
