"""ctypes binding of the C ABI in include/azalea_b200.h.

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc,
sm_100a).  There is no CPU fallback: if the library is missing or cannot be
loaded this module raises, loudly.
"""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
# AZALEA_B200_LIB: a probe build of the same sources (tools/probe), for A/B measurements only
LIB_PATH = os.environ.get('AZALEA_B200_LIB') or os.path.join(_HERE, 'lib', 'libazalea_b200.so')
HEADER_PATH = os.path.join(os.path.dirname(_HERE), 'include', 'azalea_b200.h')

AZ_OK = 0
AZ_ST_POOL_FULL, AZ_ST_TREE_FULL, AZ_ST_ILLEGAL, AZ_ST_DISABLED = 1, 2, 4, 8
AZ_LEAF_TERMINAL_KNOWN, AZ_LEAF_TERMINAL_NEW = 1, 2
AZ_LEAF_REFLECTED_BIT = 9       # leaf_info[..][1]: the leaf's network row is rotated
AZ_PRIOR_PROBS, AZ_PRIOR_LOGITS = 0, 1
AZ_CFG_SOFT_POOL_FULL, AZ_CFG_PACK_LEAVES = 1, 2
AZ_ABI_VERSION = 3
(AZ_BUF_LEAF_BOARD, AZ_BUF_LEAF_INFO, AZ_BUF_VALUE, AZ_BUF_PRIOR, AZ_BUF_META,
 AZ_BUF_REPLAY, AZ_BUF_COUNTERS, AZ_BUF_LEAF_MOVES, AZ_BUF_GLOBALS,
 AZ_BUF_LEAF_ROWS, AZ_BUF_RESIGN) = range(11)
# AZ_BUF_RESIGN columns: lowest r of colours 1 / 2 (f32 bits), resigned games, calibration games,
# false positives, then the 65-bin histogram of the winner's lowest r
AZ_RS_MIN, AZ_RS_RESIGNED, AZ_RS_CALIB, AZ_RS_FALSE_POS, AZ_RS_HIST, AZ_RS_BINS = 0, 2, 3, 4, 5, 65
COUNTER_NAMES = ('simulations', 'sum_children', 'sum_depth', 'unique_leaves',
                 'expanded_children', 'plies', 'games', 'replay_rows',
                 'replay_dropped', 'games_failed', 'compacted_nodes',
                 'nn_rows', 'pool_skipped_expansions', 'terminal_leaves',
                 'reflected_rows', 'fast_plies')
ROW_HEADER_BYTES = 48


class AzConfig(C.Structure):
    _fields_ = [('num_games', C.c_int32), ('board_size', C.c_int32),
                ('max_batch', C.c_int32), ('nodes_per_game', C.c_int32),
                ('max_nodes_ref', C.c_int64), ('replay_rows', C.c_int32),
                ('max_plies', C.c_int32), ('seed', C.c_uint64),
                ('first_game_id', C.c_int64), ('game_id_stride', C.c_int64),
                ('flags', C.c_int32), ('reserved', C.c_int32)]


class AzBufferDesc(C.Structure):
    _fields_ = [('offset', C.c_size_t), ('bytes', C.c_size_t),
                ('elem_bytes', C.c_int32), ('ndim', C.c_int32),
                ('shape', C.c_int64 * 4)]


class AzSearchParams(C.Structure):
    _fields_ = [('batch_size', C.c_int32), ('exploration_coef', C.c_float),
                ('noise_scale', C.c_double), ('noise_alpha', C.c_double)]


class AzPlayParams(C.Structure):
    _fields_ = [('temperature', C.c_float), ('exploration_depth', C.c_int32),
                ('move_sampling', C.c_int32), ('collect_replay', C.c_int32),
                ('auto_reset', C.c_int32)]


def declared_symbols():
    """Entry points declared in include/azalea_b200.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(az_[a-z_0-9]+)\s*\(', text)))


_lib = None


def lib():
    """Load libazalea_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} is missing: build the CUDA engine first '
            '(python -c "import __graft_entry__ as g; g.build()"). '
            'azalea_b200 has no CPU fallback.')
    L = C.CDLL(LIB_PATH)
    vp, i32p, f32p = C.c_void_p, C.c_void_p, C.c_void_p  # device pointers
    eng = C.c_void_p
    L.az_abi_version.restype = C.c_int
    L.az_strerror.restype = C.c_char_p
    L.az_strerror.argtypes = [C.c_int]
    L.az_last_cuda_error.restype = C.c_char_p
    L.az_engine_device_bytes.restype = C.c_size_t
    L.az_engine_device_bytes.argtypes = [C.POINTER(AzConfig)]
    L.az_engine_create.argtypes = [C.POINTER(eng), C.POINTER(AzConfig), vp,
                                   C.c_size_t, C.c_int]
    L.az_engine_destroy.argtypes = [eng]
    L.az_engine_destroy.restype = None
    L.az_engine_buffer.argtypes = [eng, C.c_int, C.POINTER(AzBufferDesc)]
    L.az_replay_row_bytes.argtypes = [eng]
    L.az_games_reset.argtypes = [eng, vp, vp]
    L.az_hex_step.argtypes = [eng, i32p, i32p, vp]
    L.az_hex_state.argtypes = [eng, vp, i32p, i32p, i32p, vp]
    L.az_hex_legal_moves.argtypes = [eng, i32p, i32p, vp]
    L.az_hex_set_state.argtypes = [eng, vp, i32p, i32p, C.c_int, vp]
    L.az_mcts_select_root.argtypes = [eng, vp]
    L.az_mcts_select.argtypes = [eng, C.POINTER(AzSearchParams), vp]
    L.az_leaf_moves.argtypes = [eng, vp]
    L.az_mcts_expand_backup.argtypes = [eng, f32p, f32p, C.c_int, vp]
    L.az_mcts_expand_root.argtypes = [eng, f32p, C.c_int, vp]
    L.az_root_stats.argtypes = [eng, f32p, f32p, f32p, i32p, f32p, vp, vp]
    L.az_tree_move.argtypes = [eng, i32p, vp]
    L.az_mcts_root_uniform.argtypes = [eng, vp]
    L.az_engine_set_window.argtypes = [eng, C.c_int, C.c_int]
    L.az_engine_set_reflect.argtypes = [eng, C.c_int]
    L.az_engine_set_playout_cap.argtypes = [eng, C.c_float, C.c_int]
    L.az_engine_set_resign.argtypes = [eng, C.c_float, C.c_float]
    L.az_engine_set_forced_playouts.argtypes = [eng, C.c_float, C.c_float]
    L.az_status.argtypes = [eng, i32p, vp]
    L.az_stub_eval.argtypes = [eng, C.c_int, vp]
    L.az_replay_collate.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, i32p, i32p,
                                    f32p, f32p, vp, vp, i32p, vp]
    L.az_batch_reflect.argtypes = [i32p, i32p, f32p, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]
    L.az_nn_stem.argtypes = [vp, C.c_int, C.c_int, C.c_int64, vp, f32p, vp, C.c_int,
                             C.c_int, vp]
    L.az_nn_heads.argtypes = [vp, C.c_int64, f32p, f32p, vp, C.c_int64, C.c_int, C.c_int, C.c_int, vp]
    L.az_nn_tail.argtypes = [vp, C.c_int64, C.c_int, C.c_int, C.c_int, f32p, f32p, f32p,
                             f32p, C.c_int64, f32p, C.c_int64, vp]
    L.az_nn_stem_live.argtypes = L.az_nn_stem.argtypes[:-1] + [i32p, vp]
    L.az_nn_heads_live.argtypes = L.az_nn_heads.argtypes[:-1] + [i32p, vp]
    L.az_nn_tail_live.argtypes = L.az_nn_tail.argtypes[:-1] + [i32p, vp]
    L.az_nn_tower_group.argtypes = [C.c_int]
    L.az_nn_tower_halo.argtypes = [C.c_int]
    L.az_nn_tower_rows.argtypes = [C.c_int, C.c_int64]
    L.az_nn_tower_rows.restype = C.c_int64
    L.az_nn_conv3x3.argtypes = [vp, vp, f32p, vp, vp, C.c_int, C.c_int64, vp]
    L.az_nn_resblock.argtypes = [vp, vp, f32p, vp, C.c_int, C.c_int64, vp]
    L.az_nn_resblocks.argtypes = [vp, vp, f32p, vp, C.c_int, C.c_int64, C.c_int, vp]
    L.az_nn_resblocks_live.argtypes = L.az_nn_resblocks.argtypes[:-1] + [i32p, vp]
    L.az_nn_resblock_scratch_bytes.restype = C.c_size_t
    L.az_noise_sample.argtypes = [eng, C.c_float, C.c_int, C.c_int, f32p, vp]
    L.az_play_commit.argtypes = [eng, C.POINTER(AzPlayParams), i32p, vp]
    L.az_replay_clear.argtypes = [eng, vp]
    for name in declared_symbols():
        fn = getattr(L, name)       # AttributeError if a symbol is missing
        if fn.restype is C.c_int and name not in ('az_abi_version',):
            fn.restype = C.c_int
    _lib = L
    return L


def check(code):
    if code != AZ_OK:
        L = lib()
        msg = L.az_strerror(code).decode()
        if code == -2:
            msg += ': ' + L.az_last_cuda_error().decode()
        raise RuntimeError(f'azalea_b200 engine call failed: {msg}')
