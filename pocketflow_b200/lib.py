"""ctypes binding of libpf_b200.so (the C ABI declared in include/pf_b200.h).

There is NO fallback: if the shared library is missing or fails to load, importing any
compute entry point raises immediately (north star: "no CPU fallback").  Build it with
``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C pocketflow_b200/csrc``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libpf_b200.so')

c_i32, c_i64, c_f32, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p

# name -> (restype, argtypes); mirrors include/pf_b200.h one to one
SIGNATURES = {
    'pf_abi_version': (c_i32, []),
    'pf_last_error': (ctypes.c_char_p, []),
    'pf_launch_count': (c_i64, []),
    'pf_launch_count_reset': (None, []),
    'pf_sm_count': (c_i32, [ctypes.POINTER(c_i32)]),
    'pf_fill_u32': (c_i32, [c_vp, c_i64, ctypes.c_uint32, c_vp]),
    'pf_minmax_reset': (c_i32, [c_vp, c_i64, c_vp]),
    'pf_uq_weight_minmax': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_uq_weight_scales': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_uq_weight_quant': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp]),
    'pf_uq_weight_ste_bwd': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp]),
    'pf_uq_act_minmax': (c_i32, [c_vp, c_i64, c_vp, c_vp]),
    'pf_uq_act_quant': (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i32, c_vp]),
    'pf_uq_act_quant_planes': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp]),
    'pf_ws_mask_build': (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'pf_select_desc': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'pf_momentum_step': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_f32, c_f32, c_f32, c_vp]),
    'pf_adam_step': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_f32, c_f32, c_f32, c_f32, c_f32, c_vp]),
    'pf_softmax_ce_fwd_bwd': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp]),
    'pf_l2_loss': (c_i32, [c_vp, c_i64, c_f32, c_i32, c_vp, c_vp, c_vp]),
    'pf_nuq_weight_quant': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'pf_nuq_weight_quant_ex': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_nuq_cluster_grad': (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_nuq_bucket_weight_quant': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_nuq_bucket_quantile_init': (c_i32, [c_vp, c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_nuq_bucket_cluster_grad': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                           c_vp]),
    'pf_im2col': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_s2d_planes': (c_i32, [c_vp] + [c_i32] * 9 + [c_vp, c_vp, c_vp]),
    'pf_preprocess_images': (c_i32, [c_vp, c_vp, c_i32, c_i32, c_i32, c_f32, c_f32, c_f32, c_vp, c_vp]),
    'pf_gather_rows': (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp]),
    'pf_im2col_planes': (c_i32, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_conv2d_fwd': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_conv2d_dgrad': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_conv2d_wgrad_workspace_bytes': (c_i64, [c_vp]),
    'pf_conv2d_wgrad': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_supported': (c_i32, [c_vp]),
    'pf_conv2d_tc_weight_elems': (c_i64, [c_vp, c_i32]),
    'pf_conv2d_tc_prep_weight': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_fwd': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_dgrad': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_conv2d_tc_wgrad_supported': (c_i32, [c_vp]),
    'pf_conv2d_tc_wgrad_workspace_bytes': (c_i64, [c_vp]),
    'pf_conv2d_tc_wgrad': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_prep_weights_multi': (c_i32, [c_vp, c_vp, c_i32, c_vp]),
    'pf_conv2d_tc_wgrad_splits': (c_i32, [c_vp]),
    'pf_conv2d_tc_wgrad_reduce_multi': (c_i32, [c_vp, c_vp, c_i32, c_vp]),
    'pf_split_bf16': (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    'pf_conv2d_tc_wgrad_planes_workspace_bytes': (c_i64, [c_vp]),
    'pf_conv2d_tc_fwd_planes': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_dgrad_planes': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_conv2d_tc_wgrad_planes': (c_i32, [c_vp] * 8),
    'pf_conv2d_tc_tma_supported': (c_i32, [c_vp, c_i32]),
    'pf_conv2d_tc_set_feed': (c_i32, [c_i32]),
    'pf_conv2d_tc_fwd_ex': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_conv2d_tc_dgrad_ex': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_conv2d_tc_wgrad_ex': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_tc_probe': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32] + [ctypes.c_uint32] * 6 + [c_vp]),
    'pf_dwconv_fwd': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_dwconv_dgrad': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_dwconv_wgrad_workspace_bytes': (c_i64, [c_vp]),
    'pf_dwconv_wgrad': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_bn_train_stats': (c_i32, [c_vp, c_i64, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_bn_eval_prepare': (c_i32, [c_vp, c_i32, c_f32, c_vp, c_vp]),
    'pf_bn_apply': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    'pf_bn_bwd': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32,
                          c_vp, c_vp]),
    'pf_bn_train_stats_range': (c_i32, [c_vp, c_i64, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32,
                                        c_vp, c_vp, c_vp]),
    'pf_bn_apply_eval': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_f32, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_bn_apply_quant': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp]),
    'pf_bn_apply_quant_levels': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp,
                                         c_vp, c_vp]),
    'pf_bn_apply_planes': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_bn_bwd_planes': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32,
                                 c_vp, c_vp, c_vp, c_vp]),
    'pf_add': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp]),
    'pf_fold_diag_blocks': (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'pf_relu_bwd': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    'pf_colsum': (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    'pf_maxpool_fwd': (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp]),
    'pf_maxpool_bwd': (c_i32, [c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    'pf_global_avgpool_fwd': (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'pf_global_avgpool_bwd': (c_i32, [c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'pf_softmax_fwd': (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp]),
    'pf_softmax_bwd': (c_i32, [c_vp, c_vp, c_i32, c_i32, c_vp, c_vp]),
    'pf_comm_nccl_version': (c_i32, [ctypes.POINTER(c_i32)]),
    'pf_comm_unique_id': (c_i32, [c_vp]),
    'pf_comm_init': (c_i32, [c_vp, c_i32, c_i32, ctypes.POINTER(c_vp)]),
    'pf_comm_destroy': (c_i32, [c_vp]),
    'pf_allreduce_flat': (c_i32, [c_vp, c_vp, c_i64, c_vp]),
    'pf_broadcast_flat': (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp]),
    'pf_cpg_diff_l2': (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    'pf_cpg_group_norms': (c_i32, [c_vp, c_vp, c_f32, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'pf_cpg_prox_apply': (c_i32, [c_vp, c_vp, c_f32, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    'pf_cpg_channel_mask': (c_i32, [c_vp, c_i32, c_i32, c_i32, c_vp, c_vp]),
    'pf_mul': (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp]),
}


class ConvDesc(ctypes.Structure):
    """pf_conv_desc (host struct)."""
    _fields_ = [(n, c_i32) for n in ('n', 'h', 'w', 'c', 'k', 'r', 's', 'p', 'q',
                                     'stride_h', 'stride_w', 'pad_t', 'pad_l')]



class TcAct(ctypes.Structure):
    """pf_tc_act: activation / gradient operand of the tensor-core kernels (host struct of device pointers)."""
    _fields_ = [('plane0', c_vp), ('plane1', c_vp), ('hdr', c_vp), ('csum', c_vp), ('nseg', c_i32), ('reserved', c_i32)]


class TcWt(ctypes.Structure):
    """pf_tc_wt: weight operand (split-bf16 planes, or integer levels + the quantizer's bucket scales)."""
    _fields_ = [('plane0', c_vp), ('plane1', c_vp), ('alpha', c_vp), ('beta', c_vp), ('per_channel', c_i32),
                ('bits', c_i32)]


_lib = None


class PFLibraryMissing(RuntimeError):
    pass


def load():
    """Load libpf_b200.so once; raise loudly when it is absent (no CPU path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PFLibraryMissing(
            'libpf_b200.so not found at %s — build it first (__graft_entry__.build()); '
            'pocketflow_b200 has no CPU fallback' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.pf_abi_version() != 1:
        raise RuntimeError('libpf_b200.so ABI version mismatch')
    _lib = lib
    return lib


def check(status, what):
    """0 = ok; <0 argument errors -> ValueError (the run scripts' `except ValueError` contract,
    nets/resnet_at_cifar10_run.py:64-66); >0 cudaError_t -> RuntimeError."""
    if status == 0:
        return
    msg = load().pf_last_error().decode('utf-8', 'replace')
    if status in (-1, -2):       # argument errors
        raise ValueError('%s: %s' % (what, msg))
    raise RuntimeError('%s failed with status %d: %s' % (what, status, msg))
