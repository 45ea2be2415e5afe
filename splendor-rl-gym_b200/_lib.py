"""ctypes binding of libsplendor_b200.so (C ABI: include/splendor_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is
no Python or CPU fallback: if the library is missing, importing this module raises.
"""
import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get('SPLENDOR_B200_LIB', _HERE / 'libsplendor_b200.so'))  # override: kernel A/B experiments

SPL_OK = 0
SPL_E_CAPACITY = -6  # caller buffer too small; the call reports the size it needs
ERRORS = {-1: 'SPL_E_INVALID', -2: 'SPL_E_NODEVICE', -3: 'SPL_E_CUDA', -4: 'SPL_E_NOMEM',
          -5: 'SPL_E_TABLE_FULL', -6: 'SPL_E_CAPACITY', -7: 'SPL_E_STATE'}


class SplendorB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'{ERRORS.get(code, code)}: {msg}')
        self.code = code


class Key(C.Structure):
    _fields_ = [('lo', C.c_uint64), ('hi', C.c_uint64)]


class Config(C.Structure):
    _fields_ = [('device', C.c_int32), ('reserved0', C.c_int32), ('table_slots', C.c_uint64),
                ('max_table_bytes', C.c_uint64), ('chunk_parents', C.c_uint64), ('node_slots', C.c_uint64),
                ('max_node_bytes', C.c_uint64)]


class LevelInfo(C.Structure):
    _fields_ = [('level', C.c_int32), ('ended', C.c_int32), ('frontier', C.c_int64), ('expanded', C.c_int64),
                ('generated', C.c_int64), ('unique', C.c_int64), ('kept', C.c_int64), ('goal_rank', C.c_int64),
                ('visited', C.c_int64), ('table_slots', C.c_uint64), ('ms_count', C.c_float), ('ms_expand', C.c_float),
                ('ms_resolve', C.c_float), ('ms_select', C.c_float), ('ms_sort', C.c_float), ('ms_warp', C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RGameInfo(C.Structure):
    _fields_ = [('level', C.c_int64), ('frontier', C.c_int64), ('generated', C.c_int64), ('unique', C.c_int64),
                ('kept', C.c_int64), ('visited', C.c_int64), ('goal_rank', C.c_int64), ('ended', C.c_int32),
                ('pad', C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != 'pad'}


def _load():
    if not LIB_PATH.exists():
        raise ImportError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback for this path.')
    L = C.CDLL(str(LIB_PATH), mode=getattr(os, 'RTLD_LOCAL', 0))
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    sig = {
        'spl_abi_version': (i32, []),
        'spl_last_error': (C.c_char_p, [vp]),
        'spl_deck_table': (C.POINTER(C.c_uint32), [C.POINTER(i32)]),
        'spl_host_takes': (i32, [vp, vp]),
        'spl_host_buys': (i32, [vp, vp]),
        'spl_create': (i32, [C.POINTER(Config), C.POINTER(vp)]),
        'spl_destroy': (i32, [vp]),
        'spl_reset_visited': (i32, [vp, vp]),
        'spl_set_identity': (i32, [vp, i32]),
        'spl_set_link_budget': (i32, [vp, u64]),
        'spl_spilled_bytes': (i32, [vp, C.POINTER(i64)]),
        'spl_pyhash': (i32, [vp, vp, i64, vp, vp]),
        'spl_visited_count': (i32, [vp, C.POINTER(i64)]),
        'spl_launch_count': (i32, [vp, C.POINTER(i64)]),
        'spl_transfer_bytes': (i32, [vp, C.POINTER(i64), C.POINTER(i64)]),
        'spl_expand': (i32, [vp, vp, vp, i64, vp, vp, vp, i64, C.POINTER(i64), vp]),
        'spl_dedup': (i32, [vp, vp, vp, i64, vp, vp, vp, C.POINTER(i64), vp]),
        'spl_score': (i32, [vp, i32, i32, vp, vp, i64, vp, vp]),
        'spl_topk': (i32, [vp, vp, vp, i64, i64, i32, vp, C.POINTER(i64), vp]),
        'spl_owner_partition': (i32, [vp, vp, i64, i32, vp, vp, vp]),
        'spl_expand_rows': (i32, [vp, vp, i64, i64, vp, i64, C.POINTER(i64), vp]),
        'spl_route_keys': (i32, [vp, vp, i64, i32, vp, vp, vp]),
        'spl_dedup_flags': (i32, [vp, vp, i64, vp, vp]),
        'spl_compact_winners': (i32, [vp, vp, i64, vp, vp, C.POINTER(i64), vp]),
        'spl_score_rows': (i32, [vp, i32, i32, vp, i64, vp, vp, vp]),
        'spl_move_rows': (i32, [vp, vp, vp, i64, vp, i32, vp]),
        'spl_dtopk_begin': (i32, [vp, vp, vp, i64, C.POINTER(u64), C.POINTER(u64), vp]),
        'spl_dtopk_hist': (i32, [vp, i32, i32, i32, i32, u64, C.POINTER(vp), vp]),
        'spl_dtopk_pick': (i32, [vp, i32, i32, i32, i32, i64, vp]),
        'spl_dtopk_get': (i32, [vp, vp, vp]),
        'spl_dtopk_set': (i32, [vp, vp, vp]),
        'spl_dtopk_cut': (i32, [vp, i32, i32, i32, u64, u64, vp, vp, vp, vp, C.POINTER(i64), vp]),
        'spl_count_less': (i32, [vp, i32, i32, vp, vp, vp, i64, vp, vp, vp, i64, vp, i32, i32, vp]),
        'spl_rexpand': (i32, [vp, vp, vp, i64, vp, i64, C.POINTER(i64), vp]),
        'spl_rscore': (i32, [vp, vp, vp, i64, vp, vp]),
        'spl_rmaxpts': (i32, [vp, vp, vp, i64, vp, vp]),
        'spl_rpack': (i32, [vp, vp, vp, i64, vp, vp]),
        'spl_rsolver_create': (i32, [vp, vp, vp, i64, i32, C.POINTER(vp)]),
        'spl_rsolver_frontier': (i32, [vp, C.POINTER(vp), C.POINTER(i64)]),
        'spl_rbatch_create': (i32, [vp, vp, vp, vp, i32, i32, C.POINTER(vp)]),
        'spl_rbatch_games': (i32, [vp, vp, i32]),
        'spl_rbatch_frontier': (i32, [vp, i32, C.POINTER(vp), C.POINTER(i64)]),
        'spl_rbatch_lines': (i32, [vp, vp, i64, vp]),
        'spl_sbatch_create': (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, C.POINTER(vp)]),
        'spl_sbatch_games': (i32, [vp, vp, i32]),
        'spl_sbatch_frontier': (i32, [vp, i32, C.POINTER(vp), C.POINTER(i64)]),
        'spl_sbatch_lines': (i32, [vp, vp, i64, vp]),
        'spl_rexpand_rows': (i32, [vp, vp, vp, i64, i64, vp, i64, C.POINTER(i64), vp]),
        'spl_rroute_keys': (i32, [vp, vp, vp, i64, i32, vp, vp, vp]),
        'spl_rdedup_flags': (i32, [vp, vp, i64, vp, vp]),
        'spl_rcompact_winners': (i32, [vp, vp, i64, vp, vp, C.POINTER(i64), vp]),
        'spl_rmove_rows': (i32, [vp, vp, vp, i64, vp, i32, vp]),
        'spl_rfirst_goal': (i32, [vp, vp, vp, i64, C.POINTER(i64), vp]),
        'spl_rreset_visited': (i32, [vp, vp]),
        'spl_rvisited_count': (i32, [vp, C.POINTER(i64)]),
        'spl_solver_create': (i32, [vp, C.POINTER(Key), u64, i32, i32, i32, i64, i32, i32, i32, C.POINTER(vp)]),
        'spl_solver_create_queue': (i32, [vp, vp, i64, i32, i32, i32, i64, i32, i32, i32, C.POINTER(vp)]),
        'spl_solver_destroy': (i32, [vp]),
        'spl_solver_step': (i32, [vp, C.POINTER(LevelInfo), vp]),
        'spl_solver_cut': (i32, [vp, vp, i64, C.POINTER(LevelInfo), vp]),
        'spl_solver_frontier': (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(i64)]),
        'spl_solver_path': (i32, [vp, vp, vp, i32, C.POINTER(i32)]),
        'spl_gs_create': (i32, [vp, i32, i32, C.POINTER(Key), u64, i32, i32, i64, i32, i32, C.POINTER(vp)]),
        'spl_gs_destroy': (i32, [vp]),
        'spl_gs_goal': (i32, [vp, C.POINTER(i64), C.POINTER(i64), vp]),
        'spl_gs_round_begin': (i32, [vp, i64, i64, vp, C.POINTER(i64), vp]),
        'spl_gs_round_buys': (i32, [vp, vp, vp]),
        'spl_gs_round_buys_peer': (i32, [vp, vp, vp, vp]),
        'spl_ipc_alloc': (i32, [vp, u64, C.POINTER(vp), vp]),
        'spl_ipc_open': (i32, [vp, vp, C.POINTER(vp)]),
        'spl_ipc_close': (i32, [vp, vp]),
        'spl_ipc_free': (i32, [vp, vp]),
        'spl_gs_round_group': (i32, [vp, vp, i64, C.POINTER(i64), vp]),
        'spl_gs_counters': (i32, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        'spl_gs_stage_ms': (i32, [vp, vp]),
        'spl_gs_dict': (i32, [vp, C.POINTER(vp), C.POINTER(i64), vp]),
        'spl_gs_threshold': (i32, [vp, vp, i64, i64, C.POINTER(i32), vp]),
        'spl_gs_tie_begin': (i32, [vp, C.POINTER(i32), vp]),
        'spl_gs_tie_hist': (i32, [vp, i32, i32, i32, C.POINTER(vp), vp]),
        'spl_gs_tie_pick': (i32, [vp, i32, i32, vp]),
        'spl_gs_cut': (i32, [vp, i32, C.POINTER(i64), C.POINTER(vp), C.POINTER(i32), vp]),
        'spl_gs_partition': (i32, [vp, vp, i32, vp, vp]),
        'spl_gs_rank_sort': (i32, [vp, vp, i64, i32, i64, vp, vp]),
        'spl_gs_adopt': (i32, [vp, vp, i64, vp]),
        'spl_gs_frontier': (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i64)]),
        'spl_gs_link_at': (i32, [vp, i32, i64, C.POINTER(i32), C.POINTER(u64)]),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)  # AttributeError here == the library does not export the ABI
        f.restype, f.argtypes = res, args
    return L, tuple(sig)


lib, EXPORTS = _load()


def check(code, ctx=None):
    if code != SPL_OK:
        msg = lib.spl_last_error(ctx)
        raise SplendorB200Error(code, msg.decode() if msg else '')
