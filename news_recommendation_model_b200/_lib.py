"""ctypes binding of libnrm_b200.so (include/nrm_b200.h).

There is no CPU fallback: if the library is missing or a call fails, the caller gets
an exception.  `build()` compiles the library in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, 'csrc')
LIB_PATH = os.path.join(CSRC, 'libnrm_b200.so')

_lock = threading.Lock()
_lib = None

vp, ll, i32, f32, sz = C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/nrm_b200.h one to one
SIGNATURES = {
    'nrm_version': (i32, []),
    'nrm_last_error': (C.c_char_p, []),
    'nrm_launch_count': (C.c_ulonglong, []),
    'nrm_timing_enable': (None, [i32]),
    'nrm_timing_report': (i32, [C.c_char_p, sz]),
    'nrm_debug_umma_selftest': (i32, [vp, vp, vp, vp, vp, i32, i32, vp]),
    'nrm_debug_mma_microbench': (i32, [vp, i32, i32, i32, vp]),
    'nrm_debug_rsprof': (i32, [vp]),
    'nrm_debug_headprof': (i32, [vp]),
    'nrm_debug_ws_field': (ll, [i32, i32, i32, i32, C.c_char_p, vp]),
    'nrm_layout_entries': (i32, []),
    'nrm_layout_name': (C.c_char_p, [i32]),
    'nrm_layout_offset': (ll, [i32]),
    'nrm_layout_numel': (ll, [i32]),
    'nrm_layout_fixed_floats': (ll, []),
    'nrm_workspace_bytes': (sz, [i32, i32, i32, i32]),
    'nrm_workspace_e_offset': (sz, [i32, i32, i32, i32]),
    'nrm_forward': (i32, [vp, vp, ll, vp, ll, i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp, sz, vp]),
    'nrm_forward_encoder': (i32, [vp, vp, ll, vp, ll, i32, i32, i32, vp, i32, i32, vp, vp, sz, vp]),
    'nrm_forward_head': (i32, [i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, ll, vp, vp, sz, vp]),
    'nrm_backward': (i32, [vp, vp, ll, vp, ll, i32, i32, i32, vp, i32, i32, vp, vp, vp, sz, vp]),
    'nrm_forward_compact': (i32, [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp, sz, vp]),
    'nrm_forward_encoder_compact': (i32, [vp, i32, i32, i32, vp, i32, i32, vp, vp, sz, vp]),
    'nrm_backward_compact': (i32, [vp, i32, i32, i32, vp, i32, i32, vp, vp, vp, sz, vp]),
    'nrm_backward_encoder_compact': (i32, [vp, i32, i32, i32, vp, i32, i32, vp, ll, vp, vp, sz, vp]),
    'nrm_backward_head': (i32, [i32, i32, i32, vp, i32, vp, vp, vp, vp, sz, vp]),
    'nrm_backward_head_deferred': (i32, [i32, i32, i32, vp, i32, vp, vp, vp, vp, sz, vp]),
    'nrm_backward_encoder': (i32, [vp, vp, ll, vp, ll, i32, i32, i32, vp, i32, i32, vp, ll, vp, vp, sz, vp]),
    'nrm_loss_scratch_bytes': (sz, [i32, i32]),
    'nrm_loss_forward': (i32, [vp, vp, ll, vp, vp, i32, i32, f32, vp, vp, sz, vp]),
    'nrm_loss_backward': (i32, [vp, i32, i32, vp, vp, vp, ll, vp, sz, vp]),
    'nrm_adam_step': (i32, [vp, vp, vp, vp, ll, f32, f32, f32, f32, f32, ll, f32, vp]),
    'nrm_adam_step_device': (i32, [vp, vp, vp, vp, ll, vp, vp]),
    'nrm_peer_ctx_bytes': (sz, []),
    'nrm_peer_stats_bytes': (sz, []),
    'nrm_peer_flag_words': (i32, []),
    'nrm_peer_preload': (i32, []),
    'nrm_adam_step_allreduce': (i32, [vp, vp, vp, ll, vp, vp, vp, vp]),
    'nrm_peer_wait_consumed': (i32, [vp, vp, vp]),
    'nrm_loss_backward_sparse': (i32, [vp, i32, i32, vp, vp, ll, vp, vp, vp, sz, vp]),
    'nrm_peer_allsum_stats': (i32, [vp, i32, vp, vp, vp, vp]),
    'nrm_batch_metrics': (i32, [vp, ll, vp, ll, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
    'nrm_score_epilogue': (i32, [vp, i32, ll, ll, i32, i32, vp, vp, vp, vp]),
    'nrm_rank_strings_capacity': (sz, [i32, i32]),
    'nrm_rank_strings': (i32, [vp, vp, vp, i32, i32, vp, vp, ll, vp]),
    'nrm_expand_compact': (i32, [vp, i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
    'nrm_forward_scores': (i32, [vp, vp, ll, vp, ll, i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]),
    'nrm_forward_scores_compact': (i32, [vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, vp, vp, vp, sz, vp]),
    'nrm_history_topk': (i32, [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp]),
    'nrm_pool_workspace_bytes': (sz, [i32, i32, i32, i32]),
    'nrm_forward_pool': (i32, [vp, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp]),
    'nrm_pool_topk': (i32, [vp, i32, ll, i32, i32, i32, vp, i32, vp, i32, vp, vp, vp]),
    'nrm_pool_rank': (i32, [vp, i32, ll, i32, i32, vp, i32, vp, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp]),
    'nrm_pool_diversify': (i32, [vp, vp, i32, i32, i32, f32, i32, vp, i32, vp, i32, vp, vp, vp, vp]),
    'nrm_sample_negatives': (i32, [vp, i32, vp, vp, vp, i32, i32, i32, vp, vp, i32, i32, C.c_ulonglong, vp, i32, vp]),
}


class NrmError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu -> csrc/libnrm_b200.so with nvcc for sm_100a (cross-compiles
    without a GPU)."""
    out = subprocess.run(['make', '-C', CSRC, '-j8'], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise NrmError('building libnrm_b200.so failed (see make output above)')
    return LIB_PATH


def load():
    """Load the shared library (once) and attach the prototypes."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NrmError(f'{LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                           f'(or `make -C {CSRC}`); there is no CPU fallback')
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().nrm_last_error().decode('utf-8', 'replace')
        raise NrmError(f'{what} failed with code {rc}: {msg}')


def layout():
    """[(state_dict key, offset in floats, numel or -1 for delta)], fixed float count."""
    lib = load()
    entries = [(lib.nrm_layout_name(i).decode(), int(lib.nrm_layout_offset(i)), int(lib.nrm_layout_numel(i)))
               for i in range(lib.nrm_layout_entries())]
    return entries, int(lib.nrm_layout_fixed_floats())


class CompactBatchStruct(C.Structure):
    """`nrm_compact_batch` of include/nrm_b200.h: the compact wire format as a direct input of the row kernels."""
    _fields_ = [('articles', C.c_void_p), ('n_articles', C.c_int), ('hist_article', C.c_void_p), ('hist_time', C.c_void_p),
                ('hist_click', C.c_void_p), ('cand_article', C.c_void_p), ('cand_time', C.c_void_p), ('label32', C.c_void_p),
                ('label64', C.c_void_p)]
