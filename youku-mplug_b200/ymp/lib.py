"""ctypes binding of libymp_b200.so (the C ABI declared in include/ymp.h).

There is deliberately NO fallback: if the shared library is missing the import raises, and every
op raises ``YmpError`` when a kernel call fails.  PyTorch is used only as the owner of device
memory and streams; tensors cross this boundary as raw pointers.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libymp_b200.so")


class YmpError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `make -C youku-mplug_b200/csrc` "
        "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback."
    )

lib = C.CDLL(LIB_PATH)

ACT_NONE, ACT_GELU_ERF, ACT_GELU_TANH = 0, 1, 2
MASK_NONE, MASK_CAUSAL, MASK_BLOCK = 0, 1, 2
DT_BF16, DT_F32 = 0, 1

c_i32 = C.c_int32
c_vp = C.c_void_p


class DropoutSpec(C.Structure):
    _fields_ = [("rng", c_vp), ("site", C.c_uint32), ("p", C.c_float)]


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", c_vp), ("B", c_vp), ("D", c_vp),
        ("M", c_i32), ("N", c_i32), ("K", c_i32),
        ("lda", c_i32), ("ldb", c_i32), ("ldd", c_i32),
        ("a_mn_major", c_i32), ("b_mn_major", c_i32),
        ("bias", c_vp), ("residual", c_vp), ("ldr", c_i32),
        ("act", c_i32), ("aux_out", c_vp), ("aux_in", c_vp),
        ("out_dtype", c_i32), ("accumulate", c_i32), ("split_k", c_i32),
        ("alpha", C.c_float), ("tile_n", c_i32),
        ("res_row_mod", c_i32), ("d_row_block", c_i32), ("d_row_stride", c_i32), ("residual_dtype", c_i32),
        ("drop", DropoutSpec),
        ("im2col_P", c_i32), ("im2col_B", c_i32), ("im2col_C", c_i32), ("im2col_T", c_i32), ("im2col_H", c_i32), ("im2col_W", c_i32),
    ]


class LayerNormArgs(C.Structure):
    _fields_ = [
        ("x", c_vp), ("gamma", c_vp), ("beta", c_vp), ("y", c_vp), ("mean", c_vp), ("rstd", c_vp),
        ("in_rows", c_vp), ("rows", c_i32), ("D", c_i32), ("ldx", c_i32), ("ldy", c_i32),
        ("eps", C.c_float), ("x_dtype", c_i32), ("y_dtype", c_i32),
    ]


class LayerNormBwdArgs(C.Structure):
    _fields_ = [
        ("dy", c_vp), ("x", c_vp), ("gamma", c_vp), ("mean", c_vp), ("rstd", c_vp), ("add", c_vp),
        ("dx", c_vp), ("dgamma", c_vp), ("dbeta", c_vp), ("in_rows", c_vp),
        ("rows", c_i32), ("D", c_i32), ("ldx", c_i32), ("lddy", c_i32), ("ldadd", c_i32), ("x_dtype", c_i32),
        ("dx_drop", c_vp), ("drop", DropoutSpec),
    ]


class SeqMap(C.Structure):
    _fields_ = [
        ("seq_div", c_i32), ("n_prefix", c_i32), ("prefix_per_seq", c_i32), ("_pad", c_i32),
        ("outer_stride", C.c_int64), ("inner_stride", C.c_int64), ("pos_stride", C.c_int64),
        ("prefix_base", C.c_int64), ("prefix_stride", C.c_int64),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", c_vp), ("k", c_vp), ("v", c_vp), ("o", c_vp), ("lse", c_vp),
        ("ldq", c_i32), ("ldk", c_i32), ("ldv", c_i32), ("ldo", c_i32),
        ("q_head_stride", c_i32), ("k_head_stride", c_i32), ("v_head_stride", c_i32), ("o_head_stride", c_i32),
        ("map_q", SeqMap), ("map_kv", SeqMap), ("map_o", SeqMap),
        ("n_seq", c_i32), ("n_heads", c_i32), ("head_dim", c_i32), ("s_q", c_i32), ("s_kv", c_i32),
        ("mask", c_i32), ("mask_block", c_i32), ("total_rows", C.c_int64), ("scale", C.c_float),
        ("drop", DropoutSpec), ("s_kv_dev", c_vp), ("kv_rows", c_vp), ("ld_kv_rows", c_i32),
    ]


class GemmSkinnyArgs(C.Structure):
    _fields_ = [("x", c_vp), ("w", c_vp), ("bias", c_vp), ("residual", c_vp), ("y", c_vp),
                ("M", c_i32), ("N", c_i32), ("K", c_i32), ("ldx", c_i32), ("ldw", c_i32), ("ldr", c_i32), ("ldy", c_i32),
                ("act", c_i32), ("residual_dtype", c_i32), ("out_dtype", c_i32),
                ("y2", c_vp), ("y2_off_dev", c_vp), ("ldy2", C.c_int64), ("y2_off_stride", C.c_int64),
                ("ln_gamma", c_vp), ("ln_beta", c_vp), ("ln_out", c_vp), ("ln_counter", c_vp), ("ld_ln", c_i32),
                ("ln_eps", C.c_float)]


class AttnBwdArgs(C.Structure):
    _fields_ = [
        ("fwd", AttnArgs), ("dout", c_vp), ("dq", c_vp), ("dk", c_vp), ("dv", c_vp), ("delta_ws", c_vp),
        ("lddo", c_i32), ("lddq", c_i32), ("lddk", c_i32), ("lddv", c_i32),
        ("do_head_stride", c_i32), ("dq_head_stride", c_i32), ("dk_head_stride", c_i32), ("dv_head_stride", c_i32),
        ("map_do", SeqMap), ("map_dq", SeqMap), ("map_dkv", SeqMap),
    ]


class DropoutArgs(C.Structure):
    _fields_ = [("x", c_vp), ("y", c_vp), ("rows", c_i32), ("cols", c_i32), ("ldx", c_i32), ("ldy", c_i32),
                ("dtype", c_i32), ("row0", C.c_int64), ("drop", DropoutSpec)]


class Im2colArgs(C.Structure):
    _fields_ = [("video", c_vp), ("out", c_vp), ("B", c_i32), ("C", c_i32), ("T", c_i32), ("H", c_i32),
                ("W", c_i32), ("P", c_i32), ("ldo", c_i32)]


class ClipArgs(C.Structure):
    _fields_ = [("frames", c_vp), ("out", c_vp), ("lut", c_vp), ("B", c_i32), ("T", c_i32), ("H", c_i32), ("W", c_i32),
                ("C", c_i32)]


class EmbedArgs(C.Structure):
    _fields_ = [("ids", c_vp), ("table", c_vp), ("pos", c_vp), ("out", c_vp), ("B", c_i32), ("L", c_i32),
                ("S", c_i32), ("row_offset", c_i32), ("hidden", c_i32), ("vocab", c_i32), ("ldo", c_i32),
                ("out_dtype", c_i32)]


class CeArgs(C.Structure):
    _fields_ = [("logits", c_vp), ("labels", c_vp), ("loss", c_vp), ("lse", c_vp), ("grad_rows", c_vp),
                ("dlogits", c_vp), ("rows", c_i32), ("V", c_i32), ("ld", c_i32)]


class ColsumArgs(C.Structure):
    _fields_ = [("in_", c_vp), ("out", c_vp), ("R", c_i32), ("C", c_i32), ("ld", c_i32)]


class GroupArgs(C.Structure):
    _fields_ = [("in_", c_vp), ("out", c_vp), ("G", c_i32), ("T", c_i32), ("C", c_i32), ("ld_in", c_i32),
                ("ld_out", c_i32), ("broadcast", c_i32), ("scale", C.c_float)]


class AdamwArgs(C.Structure):
    _fields_ = [("master", c_vp), ("param", c_vp), ("grad", c_vp), ("m", c_vp), ("v", c_vp), ("sumsq", c_vp),
                ("n", C.c_int64), ("step", c_i32), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("weight_decay", C.c_float), ("grad_scale", C.c_float),
                ("max_grad_norm", C.c_float), ("hyper", c_vp), ("zero_grad", c_i32)]


lib.ymp_last_error.restype = C.c_char_p
lib.ymp_abi_version.restype = C.c_int
lib.ymp_launch_count.restype = C.c_uint64
lib.ymp_attn_last_path.restype = C.c_int
lib.ymp_set_pdl.restype = C.c_int
lib.ymp_set_pdl.argtypes = [C.c_int]
ATTN_PATH_MMA_SYNC, ATTN_PATH_TCGEN05, ATTN_PATH_SMALL, ATTN_PATH_DECODE = 0, 1, 2, 3


def _declare(name, argstruct):
    fn = getattr(lib, name)
    fn.restype = C.c_int
    fn.argtypes = [C.POINTER(argstruct), c_vp]
    return fn


_gemm = _declare("ymp_gemm", GemmArgs)
_gemm_skinny = _declare("ymp_gemm_skinny", GemmSkinnyArgs)
_gemm_skinny_batch = _declare("ymp_gemm_skinny_batch", GemmSkinnyArgs)
_ln_fwd = _declare("ymp_layernorm_fwd", LayerNormArgs)
_ln_bwd = _declare("ymp_layernorm_bwd", LayerNormBwdArgs)
_attn_fwd = _declare("ymp_attn_fwd", AttnArgs)
_attn_bwd = _declare("ymp_attn_bwd", AttnBwdArgs)
_im2col = _declare("ymp_im2col", Im2colArgs)
_clip = _declare("ymp_clip_normalize", ClipArgs)
_embed = _declare("ymp_embed_gather", EmbedArgs)
_ce_fwd = _declare("ymp_ce_fwd", CeArgs)
_ce_bwd = _declare("ymp_ce_bwd", CeArgs)
_colsum = _declare("ymp_colsum", ColsumArgs)
_group = _declare("ymp_group_reduce", GroupArgs)
_adamw = _declare("ymp_adamw", AdamwArgs)
_dropout = _declare("ymp_dropout", DropoutArgs)
_sumsq = lib.ymp_sumsq
_sumsq.restype = C.c_int
_sumsq.argtypes = [c_vp, C.c_int64, c_vp, c_vp]


def check(rc, what):
    if rc != 0:
        raise YmpError(f"{what} failed ({rc}): {lib.ymp_last_error().decode()}")


def launch_count():
    return int(lib.ymp_launch_count())


def set_pdl(on):
    """Programmatic dependent launch for this thread's next skinny-GEMM / LayerNorm / mma.sync attention launches
    (the decoding step).  Returns the previous setting."""
    return int(lib.ymp_set_pdl(int(bool(on))))


def attn_last_path():
    """Kernel family of the last attention call on this thread (ATTN_PATH_*)."""
    return int(lib.ymp_attn_last_path())


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def cur_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def call(fn, args, what):
    check(fn(C.byref(args), cur_stream()), what)
