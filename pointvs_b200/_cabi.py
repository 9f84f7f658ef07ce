"""ctypes binding of include/pvs_b200.h.

The CUDA library is the product path: if it is missing this module raises on
first use (there is no CPU or PyTorch fallback).
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# PVS_B200_LIB selects another build of the same sources (profiling variants)
LIB_PATH = os.environ.get('PVS_B200_LIB') or os.path.join(
    _HERE, '_C', 'libpvs_b200.so')

# flags / enums (mirror include/pvs_b200.h)
F_RESIDUAL = 0x001
F_EDGE_RESIDUAL = 0x002
F_EDGE_ATTENTION = 0x004
F_NORMALIZE = 0x008
F_TANH = 0x010
F_GRAPHNORM = 0x020
F_UPDATE_COORDS = 0x040
F_PERM_INVARIANT = 0x080
F_NODE_ATTENTION = 0x100
F_GATED_RESIDUAL = 0x200
F_REZERO = 0x400
F_SOFTMAX_ATTENTION = 0x800

ACT = {'none': 0, 'sigmoid': 1, 'tanh': 2, 'relu': 3, 'silu': 4, 'softplus': 5}
MATH = {'fp32': 0, 'bf16x3': 1, 'bf16': 2, 'fp16x2': 3}
MAX_K = 64            # every path, training included
MAX_K_TC_FWD = 128    # forward (scoring) in the tensor-core math modes
TILE_EDGES = 128

CAP_FWD_FP32 = 1
CAP_FWD_TCGEN05 = 2
CAP_BWD_FP32 = 4
CAP_FWD_WIDE_K = 32
CAP_POCKET = 64

POCKET_MAX_LIG_ATOMS = 256     # emitted ligand atoms per pose (K1p)
POCKET_MAX_REC_ATOMS = 65536   # atoms per receptor of a pocket (K1p)

_fp = C.c_void_p


class Graph(C.Structure):
    _fields_ = [('n_nodes', C.c_int32), ('n_edges', C.c_int32),
                ('row_ptr', _fp), ('col', _fp), ('attr', _fp),
                ('tile_ptr', _fp), ('n_tiles', _fp), ('n_tiles_cap', C.c_int32),
                ('ptile_last', _fp), ('n_ptiles', _fp),
                ('n_ptiles_cap', C.c_int32)]


class LayerConfig(C.Structure):
    _fields_ = [('k', C.c_int32), ('n_edge_classes', C.c_int32),
                ('flags', C.c_uint32), ('att_act', C.c_int32),
                ('math', C.c_int32), ('stages', C.c_int32),
                ('ev_edge_begin', C.c_void_p), ('ev_edge_end', C.c_void_p),
                ('saved_fwd_workspace', C.c_void_p)]


PARAM_FIELDS = ('edge_w1', 'edge_b1', 'edge_w2', 'edge_b2', 'coord_w1',
                'coord_b1', 'coord_w2', 'att_w', 'att_b', 'node_w1', 'node_b1',
                'gn_weight', 'gn_bias', 'gn_mean_scale', 'node_w2', 'node_b2',
                'natt_w', 'natt_b', 'edge_gate', 'node_gate')
GRAD_FIELDS = PARAM_FIELDS


class LayerParams(C.Structure):
    _fields_ = [(n, _fp) for n in PARAM_FIELDS]


class LayerGrads(C.Structure):
    _fields_ = [(n, _fp) for n in GRAD_FIELDS]


class HeadLayer(C.Structure):
    _fields_ = [('w', _fp), ('b', _fp), ('ki', C.c_int32), ('ko', C.c_int32),
                ('act', C.c_int32)]


class ModelDesc(C.Structure):
    _fields_ = [('n_layers', C.c_int32), ('k', C.c_int32),
                ('dim_input', C.c_int32), ('n_head', C.c_int32),
                ('embed_w', _fp), ('embed_b', _fp),
                ('layer_cfg', C.POINTER(LayerConfig)),
                ('layer_params', C.POINTER(LayerParams)),
                ('head', C.POINTER(HeadLayer))]


class PocketDesc(C.Structure):
    """struct pvs_pocket"""
    _fields_ = [('n_receptors', C.c_int32), ('n_atoms', C.c_int32),
                ('max_atoms', C.c_int32), ('inter_radius', C.c_double),
                ('intra_radius', C.c_double), ('xyz', _fp), ('emit', _fp),
                ('rec_ptr', _fp), ('cells', _fp), ('rr_ptr', _fp),
                ('rr_col', _fp)]


class PvsError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the CUDA library; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PvsError(
                f'{LIB_PATH} not found: build it with '
                '`python -m pointvs_b200.build` (or __graft_entry__.build()). '
                'There is no CPU fallback.')
        handle = C.CDLL(LIB_PATH)
        handle.pvs_status_string.restype = C.c_char_p
        handle.pvs_capabilities.restype = C.c_uint32
        handle.pvs_launch_count.restype = C.c_int64
        for name in ('pvs_scan_scratch_bytes', 'pvs_tiles_scratch_bytes',
                     'pvs_egnn_layer_workspace_bytes',
                     'pvs_egnn_model_workspace_bytes',
                     'pvs_radius_graph_mask_bytes',
                     'pvs_linear_bwd_workspace_bytes',
                     'pvs_egnn_layer_bwd_workspace_bytes',
                     'pvs_egnn_stack_layer_ws_stride',
                     'pvs_egnn_stack_bwd_workspace_bytes',
                     'pvs_pocket_cells_bytes',
                     'pvs_pocket_build_scratch_bytes'):
            if hasattr(handle, name):
                getattr(handle, name).restype = C.c_int64
        _lib = handle
    return _lib


def check(rc, what=''):
    if rc != 0:
        h = lib()
        msg = h.pvs_status_string(int(rc)).decode()
        if rc == 4:
            msg += f' [cudaError {h.pvs_last_cuda_error()}]'
        raise PvsError(f'{what or "pvs call"} failed: {msg} (status {rc})')


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream():
    """Raw handle of torch's current stream on the current device (the private
    accessor is ~10x cheaper than building a torch.cuda.Stream object, and this
    is called once per library call)."""
    try:
        return C.c_void_p(torch._C._cuda_getCurrentRawStream(
            torch._C._cuda_getDevice()))
    except AttributeError:      # other torch builds
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise PvsError('pointvs_b200 kernels need CUDA tensors; there is '
                           'no CPU fallback')


_SCRATCH = {}


def scratch(name, nbytes, device):
    """Grow-only device scratch buffer, reused across calls on the same
    stream.  Reuse is safe because every kernel that touches it is ordered on
    that stream; it keeps a run-ahead host from growing the allocator (a
    cudaMalloc is a device-wide sync) and saves an allocator call per use.
    Only for memory that never escapes to the caller."""
    key = (name, str(device), torch.cuda.current_stream(device).cuda_stream)
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes * 1.25), 256), dtype=torch.uint8,
                          device=device)
        _SCRATCH[key] = buf
    return buf
