"""ctypes binding of libre2nn_b200.so (the C-ABI declared in include/re2nn_b200.h).

The library is built in-tree by re2nn_seq_b200/build.py (nvcc, sm_100a).  There is no CPU or
PyTorch fallback: if the shared object is missing, import fails; if a kernel fails, a
RuntimeError carrying re2nn_last_error() is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libre2nn_b200.so')

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "re2nn_seq_b200: %s not found. Build it with `python -m re2nn_seq_b200.build` "
        "(or __graft_entry__.build()); there is no fallback path." % LIB_PATH)

lib = C.CDLL(LIB_PATH)

# TORCH_LIBRARY(re2nn, ...) registration of the hot-path ops (csrc/torch_ops.cpp): torch.ops.re2nn.*
TORCH_LIB_PATH = os.path.join(_HERE, 'libre2nn_torch.so')
if not os.path.exists(TORCH_LIB_PATH):
    raise ImportError(
        "re2nn_seq_b200: %s not found. Build it with `python re2nn_seq_b200/build.py` (or __graft_entry__.build()); "
        "there is no fallback path." % TORCH_LIB_PATH)
import torch as _torch  # noqa: E402

_torch.ops.load_library(TORCH_LIB_PATH)
tops = _torch.ops.re2nn

vp, i32, i64, f32, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

NL = {'none': 0, 'relu': 1, 'tanh': 2, 'relutanh': 3, 'sigmoid': 4}
PREC = {'fp32': 0, 'bf16': 1, 'tf32x3': 2, 'fp16x3': 3}
V_TOKEN, V_DENSE = 0, 1


class RecurrenceArgs(C.Structure):
    _fields_ = [
        ('B', i32), ('Lpad', i32), ('L', i32), ('S', i32), ('R', i32), ('farnn', i32),
        ('update_nonlinear', i32), ('precision', i32), ('v_mode', i32), ('full_pad', i32),
        ('save_for_backward', i32), ('sigmoid_exponent', f32),
        ('x', vp), ('lengths', vp), ('vtab', vp), ('gtab', vp), ('S1', vp), ('S2', vp), ('W', vp),
        ('o', vp), ('h0', vp), ('hT', vp), ('Wss1', vp), ('Wss2', vp), ('alpha', vp), ('beta', vp),
        ('hbar_save', vp), ('hst_save', vp), ('u_save', vp), ('a_save', vp), ('zsave', vp), ('rsave', vp),
        ('ws', vp), ('ws_bytes', sz), ('ab_out', vp), ('wprep', vp),
    ]


class BackwardArgs(C.Structure):
    _fields_ = [
        ('B', i32), ('Lpad', i32), ('L', i32), ('S', i32), ('R', i32), ('C', i32),
        ('farnn', i32), ('update_nonlinear', i32), ('v_mode', i32), ('full_pad', i32), ('ce1', i32),
        ('table_rows', i32), ('sigmoid_exponent', f32),
        ('x', vp), ('lengths', vp), ('dscores', vp), ('priority_mat', vp),
        ('vtab', vp), ('S1', vp), ('S2', vp), ('W', vp), ('o', vp), ('h0', vp), ('hT', vp), ('Wss1', vp),
        ('Wss2', vp), ('Wrs1', vp), ('Wrs2', vp), ('C_mat', vp),
        ('alpha', vp), ('beta', vp), ('hbar_save', vp), ('hst_save', vp), ('u_save', vp), ('a_save', vp),
        ('zsave', vp), ('rsave', vp),
        ('dS1', vp), ('dS2', vp), ('dW', vp), ('dC', vp), ('d_o', vp), ('dh0', vp), ('dhT', vp), ('dWss1', vp),
        ('dWss2', vp), ('dWrs1', vp), ('dWrs2', vp), ('dbs1', vp), ('dbs2', vp), ('dvtab', vp),
        ('ws', vp), ('ws_bytes', sz), ('dalpha_in', vp), ('dbeta_in', vp),
    ]


class OnehotBackwardArgs(C.Structure):
    _fields_ = [
        ('B', i32), ('Lpad', i32), ('L', i32), ('S', i32), ('update_nonlinear', i32), ('full_pad', i32),
        ('x', vp), ('lengths', vp), ('language', vp), ('W', vp), ('o', vp), ('h0', vp), ('hT', vp),
        ('alpha', vp), ('beta', vp), ('dalpha', vp), ('dbeta', vp), ('dlanguage', vp),
    ]


class OnehotArgs(C.Structure):
    _fields_ = [
        ('B', i32), ('Lpad', i32), ('L', i32), ('S', i32), ('update_nonlinear', i32),
        ('max_semiring', i32), ('full_pad', i32),
        ('x', vp), ('lengths', vp), ('language', vp), ('W', vp), ('o', vp), ('h0', vp), ('hT', vp),
        ('alpha', vp), ('beta', vp),
    ]


def _sig(name, restype, argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = argtypes
    return fn


# every symbol declared in include/re2nn_b200.h (tests/test_abi.py checks this list against the header)
SYMBOLS = {
    're2nn_abi_version': (C.c_int, []),
    're2nn_last_error': (C.c_char_p, []),
    're2nn_has_tcgen05': (C.c_int, []),
    're2nn_profile_enable': (C.c_int, [C.c_int]),
    're2nn_debug_set_tc_trace': (C.c_int, [vp]),
    're2nn_debug_set_tc_timeline': (C.c_int, [vp]),
    're2nn_debug_set_tc_cta_group': (C.c_int, [C.c_int]),
    're2nn_debug_set_resident': (C.c_int, [C.c_int]),
    're2nn_debug_set_tn_tc': (C.c_int, [C.c_int]),
    're2nn_debug_set_crf_backward_split': (C.c_int, [C.c_int]),
    're2nn_debug_set_backward_tc': (C.c_int, [C.c_int]),
    're2nn_debug_set_viterbi_seqs': (C.c_int, [C.c_int]),
    're2nn_profile_read': (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    're2nn_profile_intervals': (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_int]),
    're2nn_profile_count': (C.c_int, [C.c_int]),
    're2nn_profile_enabled': (C.c_int, []),
    're2nn_gemm_nt_workspace': (sz, [C.c_int, C.c_int, C.c_int, C.c_int]),
    're2nn_gemm_nt': (C.c_int, [C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, sz, vp]),
    're2nn_gemm_tn_path': (C.c_int, [C.c_int, C.c_int, i64, C.c_int]),
    're2nn_gemm_tn_workspace': (sz, [C.c_int, C.c_int]),
    're2nn_gemm_tn': (C.c_int, [C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, i64, vp, vp, C.c_int, C.c_int, i64,
                                vp, vp, C.c_int, vp, vp, sz, vp]),
    're2nn_token_table': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    're2nn_gate_table': (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp]),
    're2nn_output_vector_sum': (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp]),
    're2nn_decompose_recurrence_workspace': (sz, [C.POINTER(RecurrenceArgs)]),
    're2nn_decompose_recurrence_launches': (C.c_int, [C.POINTER(RecurrenceArgs)]),
    're2nn_decompose_recurrence_resident': (C.c_int, [C.POINTER(RecurrenceArgs)]),
    're2nn_decompose_recurrence_fuses': (C.c_int, [C.POINTER(RecurrenceArgs)]),
    're2nn_decompose_weight_prep_bytes': (sz, [C.POINTER(RecurrenceArgs)]),
    're2nn_decompose_weight_prep': (C.c_int, [C.POINTER(RecurrenceArgs), vp, vp]),
    're2nn_label_scores_ab_bytes': (sz, [C.c_int, C.c_int, C.c_int, C.c_int]),
    're2nn_label_scores_ab': (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, vp, vp, sz, vp]),
    're2nn_decompose_recurrence': (C.c_int, [C.POINTER(RecurrenceArgs), vp]),
    're2nn_decompose_backward_workspace': (sz, [C.POINTER(BackwardArgs)]),
    're2nn_decompose_backward': (C.c_int, [C.POINTER(BackwardArgs), vp]),
    're2nn_token_table_backward_workspace': (sz, [C.c_int, C.c_int, C.c_int]),
    're2nn_token_table_backward': (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, sz, vp]),
    're2nn_decompose_max_workspace': (sz, [C.c_int, C.c_int]),
    're2nn_decompose_max_recurrence': (C.c_int, [C.POINTER(RecurrenceArgs), vp]),
    're2nn_batched_vecmat': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    're2nn_onehot_recurrence': (C.c_int, [C.POINTER(OnehotArgs), vp]),
    're2nn_debug_set_onehot_cluster': (C.c_int, [C.c_int]),
    're2nn_onehot_backward': (C.c_int, [C.POINTER(OnehotBackwardArgs), vp]),
    're2nn_onehot_sum_tensor': (C.c_int, [vp, vp, C.c_int, C.c_int, vp, vp]),
    're2nn_label_scores_backward': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, C.c_int, vp, vp, vp, vp]),
    're2nn_label_scores_workspace': (sz, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    're2nn_label_scores': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.c_int, vp, vp, sz,
                                     vp]),
    're2nn_argmax_decode': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, f32, i64, vp, vp, vp]),
    're2nn_length_order_supported': (C.c_int, [C.c_int, C.c_int]),
    're2nn_length_order': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    're2nn_flatten_i64': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp]),
    're2nn_crf_viterbi': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, f32, i64, vp, vp, vp, vp]),
    're2nn_crf_nll': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]),
    're2nn_crf_nll_backward': (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    're2nn_ce_loss': (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, i64, vp, vp, vp]),
    're2nn_ce_loss_backward': (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, i64, vp, vp]),
}

fn = {name: _sig(name, r, a) for name, (r, a) in SYMBOLS.items()}


def check(rc, what):
    if rc != 0:
        msg = fn['re2nn_last_error']()
        raise RuntimeError("re2nn_b200 %s failed: %s" % (what, msg.decode() if msg else '?'))
