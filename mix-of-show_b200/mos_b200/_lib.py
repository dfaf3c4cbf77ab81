"""ctypes binding of libmos_sm100.so (C ABI declared in include/mos_sm100.h).

The product path has no CPU fallback: if the shared library is missing or a call fails, we raise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), 'lib', 'libmos_sm100.so')

MOS_OUT_BF16, MOS_OUT_HEADS, MOS_OUT_F32 = 0, 1, 2
MOS_DT_BF16, MOS_DT_F16 = 0, 1
MOS_SEG_ROWS, MOS_SEG_TRANSPOSED = 0, 1
MOS_ACT_NONE, MOS_ACT_RELU = 0, 1

c_i32, c_i64, c_f32, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p


class GemmArgs(ctypes.Structure):
    _fields_ = [
        ('A', c_vp), ('W', c_vp),
        ('M', c_i64), ('N', c_i64), ('K', c_i64), ('lda', c_i64),
        ('conv', c_i32), ('B', c_i32), ('H', c_i32), ('Wd', c_i32), ('C', c_i32),
        ('splits', c_i32), ('stages', c_i32),
        ('partial', c_vp), ('bias', c_vp), ('bias_batch', c_vp), ('rows_per_batch', c_i64), ('bias_batch_ld', c_i64),
        ('residual', c_vp), ('ldr', c_i64),
        ('geglu', c_i32),
        ('lora_down', c_vp), ('lora_up', c_vp), ('lora_seg', c_i64),
        ('out_mode', c_i32), ('out', c_vp), ('ldc', c_i64),
        ('seg_ptr', c_vp * 3), ('seg_kind', c_i32 * 3), ('seg_rows_pad', c_i64 * 3),
        ('heads', c_i32), ('head_dim', c_i32), ('dpad', c_i32), ('dv_pad', c_i32),
        ('tokens_per_batch', c_i64), ('accumulate', c_i32), ('w_static', c_i32),
        ('a_dtype', c_i32), ('w_dtype', c_i32), ('pair_mode', c_i32),
        ('tile_counters', c_vp), ('tile_counters_len', c_i32),
        ('prefetch_ptr', c_vp), ('prefetch_bytes', c_i64),
        ('act', c_i32),
    ]


class LbfgsProblem(ctypes.Structure):
    """mos_lbfgs_problem (include/mos_sm100.h)"""
    _fields_ = [('G', c_vp), ('R', c_vp), ('out_f', c_i32), ('in_f', c_i32), ('s', ctypes.c_double), ('f0', ctypes.c_double),
                ('max_iter', c_i32), ('history', c_i32), ('best_D', c_vp), ('best_loss', ctypes.POINTER(ctypes.c_double)),
                ('n_evals', ctypes.POINTER(c_i32))]


class MosError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the CUDA library; fail loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MosError(f'{LIB_PATH} not found: run `python -c "import __graft_entry__ as g; g.build()"` '
                           f'(or `make -C mix-of-show_b200/csrc`) first; there is no CPU fallback')
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.mos_last_error.restype = ctypes.c_char_p
        _lib.mos_version.restype = ctypes.c_int
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = lib().mos_last_error().decode('utf-8', 'replace')
        if rc == -1:
            raise ValueError(f'{what}: {msg}')
        raise MosError(f'{what}: rc={rc}: {msg}')


def act_dtype(*tensors):
    """MOS_DT_* of the 16-bit activation tensors of one call (they must agree): bf16 (training) or fp16 (inference)."""
    import torch
    dts = {t.dtype for t in tensors if t is not None}
    if dts == {torch.float16}:
        return MOS_DT_F16
    if dts == {torch.bfloat16}:
        return MOS_DT_BF16
    raise TypeError(f'16-bit activation tensors must all be bf16 or all fp16, got {sorted(str(d) for d in dts)}')


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
