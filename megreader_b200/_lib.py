"""ctypes binding of libmegreader_b200.so — the only way host code reaches the CUDA kernels.

Fails loudly: there is no CPU fallback and no alternative backend.  If the library is missing
or a symbol is absent the import of any op raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libmegreader_b200.so")

_lib = None

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_f32 = ctypes.c_float
c_p = ctypes.c_void_p

# name -> argtypes (restype is int status unless listed in _RESTYPES)
_SIGS = {
    "mr_status_string": [c_int],
    "mr_last_cuda_error": [],
    "mr_abi_version": [],
    "mr_launch_count": [],
    "mr_launch_count_reset": [],
    "mr_ctc2d_forward_f32": [c_p] * 4 + [c_i64] * 8 + [c_int, c_p, c_p, c_p],
    "mr_ctc2d_forward_f64": [c_p] * 4 + [c_i64] * 8 + [c_int, c_p, c_p, c_p],
    "mr_ctc2d_backward_f32": [c_p, c_i64] + [c_p] * 6 + [c_i64] * 8 + [c_int, c_p, c_p],
    "mr_ctc2d_backward_f64": [c_p, c_i64] + [c_p] * 6 + [c_i64] * 8 + [c_int, c_p, c_p],
    "mr_ctc2d_forward_train_f32": [c_p] * 4 + [c_i64] * 8 + [c_int, c_p, c_p, c_p],
    "mr_ctc2d_backward_apply_f32": [c_p, c_i64, c_p, c_p] + [c_i64] * 4 + [c_int, c_p, c_p],
    "mr_log_softmax_rows_f32": [c_p, c_i64, c_i64, c_p, c_p],
    "mr_ctc1d_forward_train_f32": [c_p] * 4 + [c_i64] * 7 + [c_int, c_int, c_p, c_p, c_p],
    "mr_ctc1d_backward_logits_f32": [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p],
    "mr_nchw_to_nhwc": [c_p] + [c_int] * 6 + [c_p, c_p],
    "mr_nhwc_to_nchw": [c_p] + [c_int] * 6 + [c_p, c_p],
    "mr_im2col_nhwc": [c_p] + [c_int] * 10 + [c_p, c_p],
    "mr_col2im_nhwc": [c_p] + [c_int] * 10 + [c_p, c_p],
    "mr_bias_relu_pool_fwd": [c_p, c_p] + [c_int] * 11 + [c_p, c_p, c_p],
    "mr_bias_relu_pool_bwd": [c_p, c_p, c_p] + [c_int] * 11 + [c_p, c_p, c_p, c_p],
    "mr_bias_act": [c_p, c_p, c_i64, c_int, c_int, c_int, c_p, c_p],
    "mr_bn_train_fwd": [c_p] * 6 + [c_f32, c_f32, c_i64, c_int, c_int] + [c_p] * 5,
    "mr_bn_apply": [c_p] * 6 + [c_i64, c_int, c_int, c_p, c_p],
    "mr_bn_train_bwd": [c_p] * 6 + [c_i64, c_int, c_int] + [c_p] * 6,
    "mr_colsum": [c_p, c_i64, c_int, c_int, c_p, c_int, c_p, c_p],
    "mr_lstm_cell_fwd": [c_p] * 6 + [c_i64, c_p, c_int, c_int, c_int, c_int, c_p],
    "mr_lstm_cell_bwd": [c_p] * 4 + [c_i64, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_p],
    "mr_adam_step": [c_p] * 4 + [c_i64] + [c_f32] * 4 + [c_i64, c_f32, c_p, c_p],
    "mr_cast": [c_p, c_int, c_i64, c_int, c_p, c_p],
    "mr_gemm": [c_p] * 3 + [c_i64] * 6 + [c_int] * 4 + [c_f32, c_f32, c_p],
    "mr_gemm_batched": [c_p] * 3 + [c_i64] * 9 + [c_int] * 5 + [c_f32, c_f32, c_p],
    "mr_gemm_tcgen05": [c_p] * 3 + [c_i64] * 6 + [c_int] * 3 + [c_p, c_int, c_f32, c_int, c_p],
    "mr_conv_fprop_tcgen05": [c_p] * 3 + [c_int] * 10 + [c_p, c_int, c_p],
    "mr_conv_wgrad_tcgen05": [c_p] * 3 + [c_int] * 10 + [c_p],
    "mr_conv2d_fprop_tcgen05": [c_p] * 3 + [c_int] * 14 + [c_p, c_int, c_p],
    "mr_conv2d_wgrad_tcgen05": [c_p] * 3 + [c_int] * 14 + [c_p],
    "mr_lstm_step_fwd_tcgen05": [c_p] * 7 + [c_i64, c_p, c_int, c_int, c_int, c_p],
    "mr_lstm_step_bwd_tcgen05": [c_p] * 6 + [c_i64, c_p, c_p, c_int, c_int, c_int, c_p],
    "mr_lstm_seq_fwd_tcgen05": [c_p] * 6 + [c_int] * 3 + [c_p],
    "mr_lstm_seq_bwd_tcgen05": [c_p] * 6 + [c_int] * 3 + [c_p],
    "mr_lstm_seq_set_trace": [c_p],
    "mr_ctc2d_head_fwd_f32": [c_p, c_p] + [c_int] * 4 + [c_f32, c_p, c_p],
    "mr_ctc2d_head_bwd_f32": [c_p] * 5 + [c_i64] + [c_int] * 4 + [c_f32, c_p, c_p, c_p],
    "mr_deform_psroi_pool_forward_f32": [c_p] * 3 + [c_int] * 7 + [c_f32] + [c_int] * 5 + [c_f32, c_p, c_p, c_p],
    "mr_deform_psroi_pool_backward_f32": [c_p] * 5 + [c_int] * 7 + [c_f32] + [c_int] * 5 + [c_f32, c_p, c_p, c_p],
    "mr_resize_normalize_f32": [c_p, c_int, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p, c_p],
    "mr_pack_labels": [c_p, c_p, c_int, c_p, c_int, c_p, c_p, c_p],
    "mr_conv_weight_pack": [c_p] + [c_int] * 8 + [c_p, c_p],
    "mr_gate_rows_permute": [c_p, c_p] + [c_int] * 4 + [c_p, c_p],
    "mr_ctc_greedy_decode": [c_p, c_p] + [c_int] * 4 + [c_i64] * 7 + [c_int, c_int, c_p, c_p],
    "mr_blank_after_first_blank": [c_p, c_int, c_int, c_int, c_p],
    "mr_dcn_workspace_bytes": [c_i64] * 6,
    "mr_dcn_fused_workspace_bytes": [c_i64] * 7,
    "mr_dcn_forward_fused_f32": [c_p, c_p, c_p, c_p, c_i64, c_p, c_i64, c_p, c_p, c_i64] + [c_int] * 15 + [c_p],
    "mr_dcn_forward_f32": [c_p, c_p, c_p, c_p, c_i64, c_p, c_i64, c_p, c_p, c_i64] + [c_int] * 15 + [c_p],
    "mr_attn_decode_workspace_bytes": [c_i64] * 3,
    "mr_attn_decode_f32": [c_p] * 3 + [c_i64] + [c_p] * 11 + [c_i64] + [c_int] * 7 + [c_p],
    "mr_attn_decode_status": [c_p, c_i64, c_i64, c_i64, c_p, c_p],
    "mr_attn_train_fwd_f32": [c_p] * 3 + [c_i64] + [c_p] * 22 + [c_int] * 7 + [c_p],
    "mr_attn_train_bwd_f32": [c_p] * 3 + [c_i64] + [c_p] * 24 + [c_int] * 6 + [c_p],
    "mr_attn_sync_status": [c_p, c_p, c_p],
    "mr_dcn_fused_wgrad_workspace_bytes": [c_i64] * 7,
    "mr_dcn_fused_backward_workspace_bytes": [c_i64] * 9,
    "mr_dcn_backward_fused_f32": [c_p, c_p, c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_i64, c_p, c_i64, c_f32,
                                  c_p, c_i64] + [c_int] * 15 + [c_p],
    "mr_dcn_wgrad_fused_f32": [c_p, c_p, c_i64, c_p, c_i64, c_p, c_p, c_f32, c_p, c_i64] + [c_int] * 15 + [c_p],
    "mr_dcn_backward_f32": [c_p, c_p, c_p, c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_i64, c_p, c_i64, c_f32,
                            c_p, c_i64] + [c_int] * 15 + [c_p],
    "mr_db_maps_fwd_f32": [c_p, c_p, c_i64, c_f32, c_p, c_p, c_p, c_p],
    "mr_db_maps_bwd_f32": [c_p] * 6 + [c_i64, c_f32, c_p, c_p, c_p],
    "mr_db_loss_workspace_bytes": [c_i64, c_i64],
    "mr_db_loss_fwd_f32": [c_p] * 7 + [c_i64, c_i64] + [c_f32] * 5 + [c_p, c_i64, c_p, c_p],
    "mr_db_loss_bwd_f32": [c_p] * 7 + [c_i64, c_i64, c_f32, c_f32, c_p, c_i64, c_p, c_p, c_p, c_p],
}
_RESTYPES = {
    "mr_dcn_workspace_bytes": c_i64,
    "mr_dcn_fused_workspace_bytes": c_i64,
    "mr_dcn_fused_wgrad_workspace_bytes": c_i64,
    "mr_attn_decode_workspace_bytes": c_i64,
    "mr_dcn_fused_backward_workspace_bytes": c_i64,
    "mr_db_loss_workspace_bytes": c_i64,
    "mr_status_string": ctypes.c_char_p,
    "mr_last_cuda_error": ctypes.c_char_p,
    "mr_launch_count": c_i64,
    "mr_launch_count_reset": None,
}


class MegReaderB200Error(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise MegReaderB200Error(
                "megreader_b200: %s is missing - build it with `python -m megreader_b200.build` "
                "(there is no CPU or library fallback)" % SO_PATH)
        L = ctypes.CDLL(SO_PATH)
        for name, args in _SIGS.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported: fail loudly
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, c_int)
        _lib = L
    return _lib


MR_ERR_UNSUPPORTED = 5      # include/megreader_b200.h


def check(status, what=""):
    if status != 0:
        L = lib()
        msg = L.mr_status_string(status).decode()
        if status == 6:
            msg += ": " + L.mr_last_cuda_error().decode()
        raise MegReaderB200Error("%s%s" % (what + ": " if what else "", msg))


def launch_count():
    return int(lib().mr_launch_count())


def reset_launch_count():
    lib().mr_launch_count_reset()
