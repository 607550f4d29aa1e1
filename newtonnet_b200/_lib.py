"""ctypes binding of libnewtonnet_b200.so (declared in include/newtonnet_b200.h).

There is no CPU fallback and no pure-PyTorch fallback: if the CUDA library is missing the import of
anything that needs it raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libnewtonnet_b200.so')

NN_F = 128
NN_NB = 20
NN_MAX_LAYERS = 8
NN_STATUS_WORDS = 8
NN_B_IMAGE_FLOATS = 2 * 128 * 128
NN_WE_IMAGE_FLOATS = 2 * 128 * 32
ST_EDGE_OVERFLOW, ST_ROW_OVERFLOW, ST_BATCH_UNSORTED, ST_SINGULAR_CELL, ST_N_EDGES, ST_N_PAIRS, ST_N_CELLS = range(7)
STAGES = ['nbr', 'geom', 'node_gemm', 'pair_gemm', 'message', 'aggregate', 'head', 'bwd_gather', 'bwd_message',
          'bwd_aggregate', 'force', 'other']
(PH_BEGIN, PH_FWD_NODE, PH_FWD_PAIR, PH_HEAD, PH_BWD_SEED, PH_BWD_NODE, PH_BWD_PAIR, PH_FINISH, PH_FWD_PAIR_A, PH_FWD_PAIR_B,
 PH_BWD_NORM, PH_BWD_NODE_B, PH_BWD_PAIR_A, PH_BWD_PAIR_B) = range(14)
DD_MAX_RANKS, DD_CHANNELS, DD_MAX_WIDTH, DD_PARTIAL, DD_STATUS_WORDS = 16, 2, 384, 32, 8
DD_ST_STALE, DD_ST_TIMEOUT, DD_ST_OVERFLOW, DD_ST_BAD_INPUT, DD_ST_STEP, DD_ST_EDGES = range(6)
BUF_MN, BUF_F_OUT, BUF_DFB, BUF_ABAR = range(4)
PRO_NONE, PRO_SILU, PRO_ROWSCALE3, PRO_SILU_SAVE = 0, 1, 2, 3
EPI_BIAS, EPI_DSILU, EPI_ADD, EPI_EQUIV_BWD, EPI_MUL = 0, 1, 2, 3, 4

_fp = C.c_void_p   # device pointers travel as integers


class Mat(C.Structure):
    _fields_ = [('w', _fp), ('wt', _fp), ('w_img', _fp), ('wt_img', _fp)]


class LayerWeights(C.Structure):
    _fields_ = [('W1', Mat), ('b1', _fp), ('W2', Mat), ('b2', _fp), ('We', _fp), ('Wet', _fp), ('We_img', _fp),
                ('U1', Mat), ('U2', Mat), ('V1', Mat), ('V2', Mat), ('Wu', Mat), ('ln_gamma', _fp), ('ln_beta', _fp)]


class Weights(C.Structure):
    _fields_ = [('n_layers', C.c_int32), ('cutoff', C.c_float), ('embedding', _fp), ('frequencies', _fp),
                ('layer', LayerWeights * NN_MAX_LAYERS), ('H1', Mat), ('hb1', _fp), ('H2', Mat), ('hb2', _fp),
                ('w3', _fp), ('hb3', _fp), ('scale', _fp), ('shift', _fp),
                ('D1', Mat), ('db1', _fp), ('D2', Mat), ('db2', _fp), ('D3', Mat), ('db3', _fp), ('dscale', _fp)]


class Nbr(C.Structure):
    _fields_ = [('n_atoms', C.c_int32), ('n_systems', C.c_int32), ('cap_edges', C.c_int32),
                ('cap_pairs', C.c_int32), ('cap_cells', C.c_int32), ('n_owned', C.c_int32)] + [(n, _fp) for n in (
                    'pos', 'cell', 'batch', 'sys_ptr', 'row_ptr', 'col', 'edge_pair', 'pair_ptr', 'pair_i',
                    'pair_j', 'pair_disp', 'status', 'workspace')] + [('workspace_bytes', C.c_size_t)]


class GemmArgs(C.Structure):
    _fields_ = [('X', _fp), ('B', _fp), ('Y', _fp), ('B_img', _fp), ('bias', _fp), ('aux1', _fp), ('aux2', _fp), ('aux3', _fp), ('aux_out', _fp),
                ('m_dev', _fp), ('m_dev_mul', C.c_int32), ('m', C.c_int32), ('prologue', C.c_int32),
                ('epilogue', C.c_int32), ('aux_tiled', C.c_int32)]


class GemmChainArgs(C.Structure):
    _fields_ = [('X', _fp), ('B1_img', _fp), ('B2_img', _fp), ('bias1', _fp), ('bias2', _fp), ('aux1', _fp), ('aux2', _fp),
                ('aux_out', _fp), ('Y', _fp), ('m_dev', _fp), ('m_dev_mul', C.c_int32), ('m', C.c_int32), ('mid', C.c_int32),
                ('out', C.c_int32), ('B1_img_b', _fp), ('B2_img_b', _fp), ('aux_out_b', _fp), ('Y_b', _fp),
                ('pad_', C.c_int32)]


class DDComm(C.Structure):
    _R = DD_MAX_RANKS
    _fields_ = [('world', C.c_int32), ('rank', C.c_int32), ('n_atoms_total', C.c_int32), ('n_owned', C.c_int32),
                ('n_ghost', C.c_int32), ('pad_', C.c_int32), ('stride', C.c_int32 * DD_CHANNELS),
                ('landing', (_fp * 2) * DD_CHANNELS), ('flags', _fp * DD_CHANNELS), ('forces_full', _fp), ('partials', _fp),
                ('peer_landing', ((_fp * DD_MAX_RANKS) * 2) * DD_CHANNELS), ('peer_flags', (_fp * DD_MAX_RANKS) * DD_CHANNELS),
                ('peer_forces_full', _fp * DD_MAX_RANKS), ('peer_partials', _fp * DD_MAX_RANKS),
                ('send_idx', _fp), ('send_begin', C.c_int32 * DD_MAX_RANKS), ('send_end', C.c_int32 * DD_MAX_RANKS),
                ('row_offset', C.c_int32 * DD_MAX_RANKS), ('step', _fp), ('done', _fp), ('status', _fp)]


class EvalArgs(C.Structure):
    _fields_ = [('nbr', C.POINTER(Nbr)), ('w', C.POINTER(Weights)), ('z', _fp), ('want_forces', C.c_int32),
                ('want_virial', C.c_int32), ('n_owned', C.c_int32), ('pad_', C.c_int32), ('energy', _fp), ('forces', _fp), ('virial', _fp), ('stress', _fp),
                ('atom_node', _fp), ('force_node', _fp), ('direct_force', _fp), ('workspace', _fp), ('workspace_bytes', C.c_size_t)]


# every symbol include/newtonnet_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    'nn_last_error': (C.c_char_p, []),
    'nn_version': (C.c_int, []),
    'nn_launch_count': (C.c_longlong, [C.c_int]),
    'nn_profile_enable': (C.c_int, [C.c_int]),
    'nn_profile_collect': (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int), C.c_int]),
    'nn_nbr_workspace_bytes': (C.c_size_t, [C.c_int32, C.c_int32]),
    'nn_nbr_count': (C.c_int, [C.POINTER(Nbr), C.c_float, _fp]),
    'nn_nbr_fill': (C.c_int, [C.POINTER(Nbr), C.c_float, _fp]),
    'nn_nbr_edge_reverse': (C.c_int, [C.POINTER(Nbr), _fp, _fp]),
    'nn_nbr_edge_index': (C.c_int, [C.POINTER(Nbr), _fp, C.c_int64, _fp]),
    'nn_gemm128': (C.c_int, [C.POINTER(GemmArgs), _fp]),
    'nn_gemm128_prepare_b': (C.c_int, [_fp, _fp, _fp]),
    'nn_gemm128_prepare_b_batch': (C.c_int, [_fp, _fp, _fp, C.c_int32, _fp]),
    'nn_set_gemm_backend': (C.c_int, [C.c_int]),
    'nn_get_gemm_backend': (C.c_int, []),
    'nn_eval_workspace_bytes': (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    'nn_eval': (C.c_int, [C.POINTER(EvalArgs), _fp]),
    'nn_eval_phase': (C.c_int, [C.POINTER(EvalArgs), C.c_int32, C.c_int32, _fp]),
    'nn_eval_buffer': (C.c_void_p, [C.POINTER(EvalArgs), C.c_int32, C.c_int32]),
    'nn_halo_pack': (C.c_int, [_fp, _fp, C.c_int32, C.c_int32, _fp, _fp]),
    'nn_p2p_alloc': (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    'nn_p2p_free': (C.c_int, [_fp]),
    'nn_p2p_get_handle': (C.c_int, [_fp, _fp]),
    'nn_p2p_open_handle': (C.c_int, [_fp, C.POINTER(C.c_void_p)]),
    'nn_p2p_close_handle': (C.c_int, [_fp]),
    'nn_dd_begin': (C.c_int, [C.POINTER(DDComm), _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, C.c_float, _fp, _fp, _fp]),
    'nn_dd_halo_push': (C.c_int, [C.POINTER(DDComm), C.c_int32, C.c_int32, _fp, C.c_int32, _fp]),
    'nn_dd_halo_wait': (C.c_int, [C.POINTER(DDComm), C.c_int32, C.c_int32, _fp, C.c_int32, _fp]),
    'nn_dd_finish': (C.c_int, [C.POINTER(DDComm), C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_segment_sum': (C.c_int, [_fp, _fp, _fp, C.c_int32, C.c_int32, _fp, _fp]),
    'nn_gemm128_tn_workspace_bytes': (C.c_size_t, [C.c_int32]),
    'nn_gemm128_tn': (C.c_int, [_fp, _fp, C.c_int32, _fp, _fp, _fp]),
    'nn_gemm128_tn_acc': (C.c_int, [_fp, _fp, C.c_int32, _fp, _fp, C.c_int32, _fp]),
    'nn_ew_mul3': (C.c_int, [_fp, _fp, _fp, _fp, C.c_int64, _fp]),
    'nn_ew_rows': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_ew_gmul': (C.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_seg_prod': (C.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp, _fp]),
    'nn_ew_g3': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_ew_silu': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, C.c_int64, _fp]),
    'nn_ew_rbf': (C.c_int, [C.c_int32, C.c_int32, _fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_gemm128_chain': (C.c_int, [C.POINTER(GemmChainArgs), _fp]),
    'nn_mlp_mid_tiled': (C.c_int, [C.c_int32, C.c_int32]),
    'nn_mlp_fwd': (C.c_int, [_fp, C.POINTER(Mat), _fp, _fp, C.POINTER(Mat), _fp, _fp, C.c_int32, _fp, C.c_int32, _fp]),
    'nn_mlp_bwd': (C.c_int, [_fp, C.POINTER(Mat), _fp, _fp, C.POINTER(Mat), _fp, C.c_int32, _fp, C.c_int32, _fp]),
    'nn_energy_head_bwd': (C.c_int, [_fp, _fp, _fp, _fp, C.c_int32, _fp, _fp]),
    'nn_pair_gather_bwd': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_edge_message_bwd': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_node_aggregate_bwd': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_md_advance': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_double, C.c_double, C.c_double, C.c_uint64, _fp, _fp]),
    'nn_md_finish': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, C.c_double, _fp, _fp, C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    'nn_wrap_positions': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    'nn_fire_step': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_double, C.c_double, C.c_double,
                               C.c_double, C.c_double, C.c_double, C.c_int32, _fp]),
    'nn_fire_check': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    'nn_neb_forces': (C.c_int, [C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_double, _fp, _fp,
                                _fp, _fp]),
    'nn_edge_geom_fwd': (C.c_int, [_fp, _fp, C.c_float, _fp, C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    'nn_edge_geom_bwd': (C.c_int, [_fp, C.c_int32, _fp, _fp, _fp, C.c_float, _fp, C.c_int32, _fp, _fp]),
    'nn_message_prepare_b': (C.c_int, [_fp, _fp, _fp]),
    'nn_edge_message_fwd': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_node_aggregate_fwd': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_equiv_update_fwd': (C.c_int, [_fp, _fp, _fp, _fp, C.c_int32, _fp]),
    'nn_energy_head_fwd': (C.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, C.c_int32, _fp, _fp, _fp]),
    'nn_force_virial_reduce': (C.c_int, [C.POINTER(Nbr), _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_hessian_expand': (C.c_int, [_fp, _fp, C.c_int32, C.c_int32, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    'nn_hessian_scatter': (C.c_int, [_fp, _fp, C.c_int32, C.c_int32, _fp, _fp, _fp, C.c_int64, _fp, _fp]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raises NativeLibraryError (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` or '
            f'newtonnet_b200/csrc/build.sh.  newtonnet_b200 has no CPU or PyTorch fallback.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    # dense contractions: tcgen05 3xTF32 kernel with the A operand in tensor memory by default;
    # NN_GEMM_BACKEND=tc selects the shared-memory-operand variant, =simt the fp32 SIMT kernel (all are
    # CUDA kernels of this library - there is no non-CUDA path)
    lib.nn_set_gemm_backend({'simt': 0, 'tc': 1}.get(os.environ.get('NN_GEMM_BACKEND', 'ts'), 2))
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().nn_last_error().decode()
        raise RuntimeError(f'{what} failed (rc={rc}): {msg}')


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
