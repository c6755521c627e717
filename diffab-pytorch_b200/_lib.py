"""ctypes binding of ``csrc/libdiffab_b200.so`` (the C ABI declared in ``include/diffab_b200.h``).

No fallback of any kind: ``lib()`` raises if the shared library has not been built, and every
wrapper raises on CPU tensors, wrong dtypes or a non-zero return code (with ``dab_last_error``).
PyTorch is used only for device memory and the current stream.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# DAB_DEBUG_LIB=1 loads the debug build (make -C csrc debug: adds the process-global dab_debug_* hooks used by tools/)
LIB_PATH = os.path.join(_HERE, "csrc", "libdiffab_b200_dbg.so" if os.environ.get("DAB_DEBUG_LIB") == "1"
                        else os.environ.get("DAB_LIB_VARIANT", "libdiffab_b200.so"))   # DAB_LIB_VARIANT: an experiment build in csrc/ (tools only)
_lib = None


class DabSchedule(Structure):
    _fields_ = [("T", c_int), ("alpha", c_void_p), ("alpha_bar", c_void_p), ("alpha_bar_sqrt", c_void_p),
                ("one_minus_alpha_bar_sqrt", c_void_p), ("beta", c_void_p)]


class DabIpaDims(Structure):
    _fields_ = [(n, c_int) for n in ("B", "L", "D", "C", "H", "ds", "Pq", "Pv")]


_W_FIELDS = ("w_q_scalar", "w_k_scalar", "w_v_scalar", "w_q_point", "w_k_point", "w_v_point",
             "w_pair_bias", "gamma", "w_out", "b_out")


class DabIpaWeights(Structure):
    _fields_ = [(n, c_void_p) for n in _W_FIELDS]


class DabIpaGrads(Structure):
    _fields_ = [(n, c_void_p) for n in _W_FIELDS]


class DabHeadWeights(Structure):
    _fields_ = [(f"{h}_{n}", c_void_p) for h in ("c", "o", "s") for n in ("w1", "b1", "w2", "b2", "w3", "b3")]


class DabPairEmbedWeights(Structure):
    _fields_ = [(n, c_void_p) for n in ("type_emb", "relpos_emb", "pair2distcoef", "d_w1", "d_b1", "d_w2", "d_b2",
                                        "m_w1", "m_b1", "m_w2", "m_b2", "m_w3", "m_b3")]


EXPORTS = {
    # name: (restype, argtypes)
    "dab_version": (c_int, []),
    "dab_last_error": (c_char_p, []),
    "dab_launch_count": (ctypes.c_longlong, []),
    "dab_so3_exp": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dab_so3_log": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dab_so3_log_skew": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dab_so3_exp_skew": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dab_so3_scale_rot": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "dab_igso3_table": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dab_igso3_sample": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "dab_forward_noise": (c_int, [POINTER(DabSchedule), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                  c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p]),
    "dab_seq_probs": (c_int, [POINTER(DabSchedule), c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                              c_void_p, c_void_p]),
    "dab_reverse_step": (c_int, [POINTER(DabSchedule)] + [c_void_p] * 8 + [c_int, c_int] + [c_void_p] * 3 + [c_int] +
                         [c_void_p] * 5),
    "dab_reverse_step_weighted": (c_int, [POINTER(DabSchedule)] + [c_void_p] * 8 + [c_int, c_int] + [c_void_p] * 4 +
                                  [c_int] + [c_void_p] * 5),
    "dab_ipa_f32_workspace_bytes": (c_size_t, [POINTER(DabIpaDims), c_int]),
    "dab_ipa_fwd_f32": (c_int, [POINTER(DabIpaDims), POINTER(DabIpaWeights), c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "dab_ipa_bwd_f32": (c_int, [POINTER(DabIpaDims), POINTER(DabIpaWeights), c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, POINTER(DabIpaGrads), c_void_p, c_size_t, c_void_p]),
    "dab_ipa_packed_bytes": (c_size_t, [POINTER(DabIpaDims)]),
    "dab_ipa_pack_weights": (c_int, [POINTER(DabIpaDims), POINTER(DabIpaWeights), c_void_p, c_void_p]),
    "dab_ipa_packed_layout": (c_int, [POINTER(DabIpaDims), POINTER(c_size_t)]),
    "dab_ipa_sm100_workspace_bytes": (c_size_t, [POINTER(DabIpaDims)]),
    "dab_ipa_pair_bias_multi": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "dab_ipa_mid_sm100": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dab_ipa_fwd_sm100_stages": (c_int, [POINTER(DabIpaDims)] + [c_void_p] * 10 + [c_size_t, c_int, c_void_p]),
    "dab_ipa_core_sm100_live": (c_int, [POINTER(DabIpaDims)] + [c_void_p] * 6 + [c_size_t, c_void_p, c_void_p, c_void_p]),
    "dab_ipa_fwd_sm100_train": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_size_t, c_void_p]),
    "dab_ipa_sm100_workspace_layout": (c_int, [POINTER(DabIpaDims), POINTER(c_size_t)]),
    "dab_ipa_bwd_sm100_workspace_bytes": (c_size_t, [POINTER(DabIpaDims)]),
    "dab_ipa_bwd_sm100_main": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dab_ipa_bwd_sm100_finish": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dab_heads_packed_bytes": (c_size_t, []),
    "dab_heads_pack_weights": (c_int, [POINTER(DabHeadWeights), c_void_p, c_void_p]),
    "dab_heads_fwd_sm100": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dab_front_fwd_sm100": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p]),
    "dab_pair_embed_packed_bytes": (c_size_t, []),
    "dab_pair_embed_pack_weights": (c_int, [POINTER(DabPairEmbedWeights), c_void_p, c_void_p]),
    "dab_pair_embed_fwd_sm100": (c_int, [c_void_p] * 7 + [c_int, c_int, c_int, c_void_p, c_void_p]),
    "dab_rbf_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dab_rbf_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t,
                            c_void_p]),
    "dab_rbf_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                            c_size_t, c_void_p]),
    "dab_pair_base_fwd": (c_int, [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dab_pair_table_grad_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dab_pair_table_grad": (c_int, [c_void_p] * 4 + [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dab_sum_bf16": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p]),
    "dab_relu_bwd_colsum": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dab_pair_zero_masked": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "dab_pair_table_grad_sm100": (c_int, [c_void_p] * 4 + [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dab_pair_mlp_fwd_train_sm100": (c_int, [c_void_p] * 10 + [c_int, c_int, c_int] + [c_void_p] * 6),
    "dab_pair_mlp_bwd_layer_sm100": (c_int, [c_void_p] * 4 + [c_int, c_int] + [c_void_p] * 5),
    "dab_losses_fwd": (c_int, [c_void_p] * 7 + [c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "dab_losses_bwd": (c_int, [c_void_p] * 7 + [c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dab_adam_flat": (c_int, [c_void_p] * 5 + [c_float] * 5 + [c_int64, c_void_p]),
    "dab_cast_f32_to_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "dab_out_heads_fwd_sm100": (c_int, [c_void_p] * 5 + [c_int, c_int] + [c_void_p] * 6),
    "dab_ipa_front_proj_sm100": (c_int, [c_void_p] * 10 + [c_size_t, c_void_p]),
    "dab_gemm_bf16_tn": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    "dab_gemm_bf16_tn_acc": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int, c_void_p]),
    "dab_linear_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dab_bias_grad": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "dab_colsum_f32": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
}

# present only in the debug build (libdiffab_b200_dbg.so)
DEBUG_EXPORTS = {
    "dab_debug_set_timeline": (c_int, [c_void_p]),
    "dab_debug_set_bwd_timeline": (c_int, [c_void_p]),
    "dab_debug_bwd_keep_qkv": (c_int, [c_int]),
    "dab_debug_bwd_sm100_buffers": (c_int, [POINTER(DabIpaDims), c_void_p, c_void_p]),
}


_weight_generation = 0
repack_when_capturing = False   # set by distributed.GraphedTrainStep around its captures (see _packed_weights)


def weight_generation():
    """Counter that is part of every weight-derived cache key (packed weights, captured sampling graphs)."""
    return _weight_generation


def bump_weight_generation():
    """Declare that parameters may have changed behind PyTorch's back (updates replayed from a CUDA graph, raw
    ``.data`` writes)."""
    global _weight_generation
    _weight_generation += 1


def weight_key(tensors):
    """The key every weight-derived cache (packed weights, glue constants, captured sampling graphs) is checked against:
    it changes when any of ``tensors`` may have changed.  Noticed on their own: eager in-place updates of a tensor (its
    version counter) and eager in-place updates of the flat parameter a tensor is a view of
    (``distributed.GradientBucket.flatten_parameters`` records it on the view as ``_dab_flat_param``: a view made with
    ``p.data = ...`` keeps its own version counter, so an optimizer step on the flat parameter moves no per-tensor
    version).  Everything else - raw ``.data`` writes, updates replayed from a CUDA graph - must be declared with
    ``bump_weight_generation``."""
    key = []
    for t in tensors:
        flat = getattr(t, "_dab_flat_param", None)
        key.append((t.data_ptr(), t._version, -1 if flat is None else flat._version))
    key.append(_weight_generation)
    return tuple(key)


def lib():
    """Load the shared library once; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C diffab-pytorch_b200/csrc`). There is no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        for name, (res, args) in DEBUG_EXPORTS.items():
            if hasattr(handle, name):
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().dab_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed with code {rc}: {msg}")


def stream_ptr():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def dev(t, dtype, name):
    """Validate a tensor argument and return it contiguous (never copies to another device)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor - diffab_pytorch_b200 has no CPU path")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if t.device.index != torch.cuda.current_device():
        # kernels are launched on the current device's stream (stream_ptr): a tensor that lives elsewhere would be
        # dereferenced on the wrong GPU
        raise RuntimeError(f"{name}: tensor is on cuda:{t.device.index} but the current device is "
                           f"cuda:{torch.cuda.current_device()} - wrap the call in torch.cuda.device(...)")
    return t.contiguous()


def aligned_empty(nbytes, device, align=1024):
    """uint8 buffer whose data pointer is `align`-byte aligned (TMA / tcgen05 operands want 1024)."""
    buf = torch.empty(nbytes + align, device=device, dtype=torch.uint8)
    off = (-buf.data_ptr()) % align
    return buf[off: off + nbytes]


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def mask_u8(mask, name="mask"):
    if not mask.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor - diffab_pytorch_b200 has no CPU path")
    if mask.dtype == torch.bool:      # one byte per element, values 0 / 1: reinterpret, no kernel
        return mask.contiguous().view(torch.uint8)
    return mask.to(torch.uint8).contiguous() if mask.dtype != torch.uint8 else mask.contiguous()


class Schedule:
    """Device copy of the five schedule tables plus the ctypes struct that points at them."""

    def __init__(self, sched_cpu, device):
        self.T = sched_cpu["beta"].numel() - 1
        self.device = torch.device(device)
        self.tensors = {k: v.to(device=self.device, dtype=torch.float32).contiguous() for k, v in sched_cpu.items()}
        self.struct = DabSchedule(self.T, *(self.tensors[k].data_ptr() for k in
                                            ("alpha", "alpha_bar", "alpha_bar_sqrt", "one_minus_alpha_bar_sqrt",
                                             "beta")))

    def ref(self):
        return ctypes.byref(self.struct)
