"""ctypes mirror of the reference's tree-likelihood interface over the C ABI (include/physher_b200.h).

Method names follow the reference so that the parity tests read like its own tests:
`calculate()` is `tlk->calculate(tlk)` (treelikelihood.c:1552), `update_all_nodes()` is
`SingleTreeLikelihood_update_all_nodes` (:1737), `use_rescaling()` is
`SingleTreeLikelihood_use_rescaling` (:164 of the header), `initialize_gradient(flags)` /
`gradient()` are `TreeLikelihood_initialize_gradient` / `TreeLikelihood_gradient` (:237, :320).
Every call goes through the shared library; a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libphysher_b200.so")

FLAG_TREE_MODEL = 1 << 0
OPT_INCLUDE_ROOT_FREQS = 1
OPT_COMPAT_SCALED_GRADIENT = 2
OPT_UNROOTED = 3
OPT_KERNELS = 4
OPT_SCALING_THRESHOLD_EXP = 5
OPT_TIMING = 6
OPT_HOST_EXPONENTIALS = 8
OPT_INCREMENTAL = 7
OPT_TUNE = 9
KERNELS_AUTO, KERNELS_GENERIC, KERNELS_FUSED = 0, 1, 2
RAN_GENERIC, RAN_WALK, RAN_TENSOR = 1, 2, 3

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_bp = C.POINTER(C.c_uint8)

# every symbol include/physher_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("phb_last_error", C.c_char_p, []),
    ("phb_device_count", C.c_int, []),
    ("phb_version", C.c_char_p, []),
    ("phb_tlk_create", C.c_void_p, [C.c_int, C.c_int, C.c_int, C.c_int, _ip, _ip, C.c_int, C.c_int, C.c_int]),
    ("phb_tlk_free", None, [C.c_void_p]),
    ("phb_tlk_clone", C.c_void_p, [C.c_void_p, C.c_int]),
    ("phb_tlk_set_topology", C.c_int, [C.c_void_p, _ip, _ip, C.c_int]),
    ("phb_tlk_set_tip_states", C.c_int, [C.c_void_p, _bp]),
    ("phb_tlk_set_tip_partials", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_set_pattern_weights", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_set_eigen", C.c_int, [C.c_void_p, _dp, _dp, _dp]),
    ("phb_tlk_set_matrices", C.c_int, [C.c_void_p, _dp, _dp]),
    ("phb_tlk_set_frequencies", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_set_site_model", C.c_int, [C.c_void_p, _dp, _dp]),
    ("phb_tlk_set_branch_lengths", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_set_branch_length", C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    ("phb_tlk_update_all_nodes", None, [C.c_void_p]),
    ("phb_tlk_update_one_node", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_tlk_update_three_nodes", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_tlk_store", C.c_int, [C.c_void_p]),
    ("phb_tlk_restore", C.c_int, [C.c_void_p]),
    ("phb_tlk_use_rescaling", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_tlk_rescaling", C.c_int, [C.c_void_p]),
    ("phb_tlk_set_option", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("phb_tlk_calculate", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_pattern_log_likelihoods", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_initialize_gradient", C.c_size_t, [C.c_void_p, C.c_int]),
    ("phb_tlk_gradient", C.c_int, [C.c_void_p, C.POINTER(_dp)]),
    ("phb_tlk_cat_branch_gradient", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_matrix_gradient", C.c_int, [C.c_void_p, C.c_int, _dp, _dp]),
    ("phb_tlk_root_frequency_gradient", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_category_gradient", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_update_uppers", C.c_int, [C.c_void_p]),
    ("phb_tlk_calculate_branch", C.c_int, [C.c_void_p, C.c_int, C.c_int, _dp, _dp, _dp, _dp]),
    ("phb_tlk_branch_hessian_diagonal", C.c_int, [C.c_void_p, _dp, _dp, _dp]),
    ("phb_tlk_nni_moves", C.c_int, [C.c_void_p, _ip]),
    ("phb_tlk_nni_scores", C.c_int, [C.c_void_p, C.c_int, _ip, _dp, _dp, _dp]),
    ("phb_tlk_spr_targets", C.c_int, [C.c_void_p, C.c_int, _ip]),
    ("phb_tlk_spr_scores", C.c_int, [C.c_void_p, C.c_int, C.c_int, _ip, _dp, _dp, _dp]),
    ("phb_tlk_update_partials", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _dp]),
    ("phb_tlk_get_partials", C.c_int, [C.c_void_p, C.c_int, _dp]),
    ("phb_tlk_get_matrices", C.c_int, [C.c_void_p, _dp, _dp]),
    ("phb_tlk_gradient_device", C.c_int, [C.c_void_p, C.c_void_p]),
    ("phb_tlk_evaluate_launch", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_tlk_evaluate_collect", C.c_int, [C.c_void_p, _dp, _dp]),
    ("phb_group_create", C.c_void_p, [C.c_int, _ip, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _ip, C.c_int, C.c_int]),
    ("phb_group_free", None, [C.c_void_p]),
    ("phb_group_size", C.c_int, [C.c_void_p]),
    ("phb_group_shard", C.c_void_p, [C.c_void_p, C.c_int]),
    ("phb_group_shard_range", C.c_int, [C.c_void_p, C.c_int, _ip, _ip]),
    ("phb_group_set_tip_states", C.c_int, [C.c_void_p, _bp]),
    ("phb_group_set_tip_partials", C.c_int, [C.c_void_p, _dp]),
    ("phb_group_set_pattern_weights", C.c_int, [C.c_void_p, _dp]),
    ("phb_group_set_eigen", C.c_int, [C.c_void_p, _dp, _dp, _dp]),
    ("phb_group_set_frequencies", C.c_int, [C.c_void_p, _dp]),
    ("phb_group_set_site_model", C.c_int, [C.c_void_p, _dp, _dp]),
    ("phb_group_set_branch_lengths", C.c_int, [C.c_void_p, _dp]),
    ("phb_group_set_option", C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ("phb_group_use_rescaling", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_group_rescaling", C.c_int, [C.c_void_p]),
    ("phb_group_set_reduction", C.c_int, [C.c_void_p, C.c_int]),
    ("phb_group_reduction", C.c_int, [C.c_void_p]),
    ("phb_nccl_version", C.c_int, []),
    ("phb_comm_unique_id", C.c_int, [C.c_void_p]),
    ("phb_comm_init_rank", C.c_void_p, [C.c_int, C.c_int, C.c_void_p, C.c_int]),
    ("phb_comm_free", None, [C.c_void_p]),
    ("phb_comm_size", C.c_int, [C.c_void_p]),
    ("phb_comm_rank", C.c_int, [C.c_void_p]),
    ("phb_tlk_gradient_allreduce_device", C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("phb_tlk_gradient_allreduce", C.c_int, [C.c_void_p, C.c_void_p, _dp, C.POINTER(_dp)]),
    ("phb_group_calculate", C.c_int, [C.c_void_p, _dp]),
    ("phb_group_gradient", C.c_int, [C.c_void_p, _dp, C.POINTER(_dp)]),
    ("phb_tlk_stream", C.c_void_p, [C.c_void_p]),
    ("phb_tlk_synchronize", C.c_int, [C.c_void_p]),
    ("phb_tlk_gradient_batch", C.c_int, [C.c_void_p, C.c_int, _dp, _dp, _dp]),
    ("phb_tlk_set_time_tree", C.c_int, [C.c_void_p, _dp]),
    ("phb_tlk_gradient_batch_time", C.c_int, [C.c_void_p, C.c_int, _dp, _dp, C.c_int, C.c_int, _dp, _dp, _dp, _dp]),
    ("phb_compress_patterns", C.c_int, [C.c_int, C.c_int, C.c_size_t, _bp, C.c_int, C.POINTER(C.c_size_t), C.POINTER(_bp), C.POINTER(_dp),
                                        C.POINTER(_ip)]),
    ("phb_free", None, [C.c_void_p]),
    ("phb_patterns_last_error", C.c_char_p, []),
    ("phb_tlk_kernel_time", C.c_int, [C.c_void_p, _dp, C.POINTER(C.c_longlong)]),
    ("phb_tlk_launch_count", C.c_longlong, [C.c_void_p]),
    ("phb_tlk_last_kernels", C.c_int, [C.c_void_p]),
]


class PhysherB200Error(RuntimeError):
    pass


_lib = None


def load_library() -> C.CDLL:
    """Load the in-tree shared library; fail loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PhysherB200Error(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). The tree-likelihood path has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def device_count() -> int:
    return int(load_library().phb_device_count())


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def compress_patterns(alignment, device=0, hashtable_size=100, want_site_map=True):
    """SitePattern construction (new_SitePattern2, sitepattern.c:186-251) on the device.
    alignment: uint8 [ntaxa][nsites] encoded states.  Returns (patterns uint8 [ntaxa][P], weights float64 [P], site_to_pattern int32 [nsites])
    with the patterns in the reference's own order."""
    lib = load_library()
    a = np.ascontiguousarray(alignment, dtype=np.uint8)
    assert a.ndim == 2
    T, n = a.shape
    npat = C.c_size_t(0)
    pat, w, smap = _bp(), _dp(), _ip()
    rc = lib.phb_compress_patterns(int(device), T, n, a.ctypes.data_as(_bp), int(hashtable_size), C.byref(npat), C.byref(pat), C.byref(w),
                                   C.byref(smap) if want_site_map else None)
    if rc != 0:
        raise PhysherB200Error(f"[{rc}] {(lib.phb_patterns_last_error() or b'').decode()}")
    try:
        P = npat.value
        patterns = np.ctypeslib.as_array(pat, shape=(T, P)).copy()
        weights = np.ctypeslib.as_array(w, shape=(P,)).copy()
        site_map = np.ctypeslib.as_array(smap, shape=(n,)).copy() if want_site_map else None
    finally:
        lib.phb_free(pat)
        lib.phb_free(w)
        if want_site_map:
            lib.phb_free(smap)
    return patterns, weights, site_map


NCCL_ID_BYTES = 128
GROUP_REDUCE_HOST, GROUP_REDUCE_NCCL = 0, 1


_nccl_preloaded = False


def _preload_nccl():
    """The C layer binds NCCL at run time by soname (dlopen "libnccl.so.2").  A Python process that also imports torch must end up with
    ONE NCCL: torch's wheels bring their own copy (nvidia/nccl/lib/libnccl.so.2, newer than a system package and linked against by
    libtorch_cuda), so that copy is loaded first when it exists -- the dynamic linker then resolves the soname to it for the C layer
    and for torch alike, whichever of the two asks first.  Pure C hosts (physher itself) use the system library."""
    global _nccl_preloaded
    if _nccl_preloaded:
        return
    _nccl_preloaded = True
    try:
        import importlib.util

        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
            path = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(path):
                C.CDLL(path, mode=C.RTLD_GLOBAL)
                return
    except Exception:
        pass


def nccl_version() -> int:
    """NCCL_VERSION_CODE of the library the C layer bound at run time (0: not loadable)."""
    _preload_nccl()
    return int(load_library().phb_nccl_version())


class Comm:
    """NCCL communicator owned by the C library (csrc/phb_nccl.c): one rank per process, one GPU per rank.  Rank 0 makes the unique
    id (`Comm.unique_id()`), the launcher carries its 128 bytes to the other ranks, every rank builds `Comm(nranks, rank, id, device)`."""

    @staticmethod
    def unique_id() -> bytes:
        _preload_nccl()
        lib = load_library()
        buf = C.create_string_buffer(NCCL_ID_BYTES)
        rc = lib.phb_comm_unique_id(buf)
        if rc != 0:
            raise PhysherB200Error(f"[{rc}] {(lib.phb_last_error() or b'').decode()}")
        return buf.raw

    def __init__(self, nranks: int, rank: int, unique_id: bytes, device: int):
        _preload_nccl()
        self.lib = load_library()
        assert len(unique_id) == NCCL_ID_BYTES
        self._id = C.create_string_buffer(unique_id, NCCL_ID_BYTES)
        self.h = self.lib.phb_comm_init_rank(int(nranks), int(rank), self._id, int(device))
        if not self.h:
            raise PhysherB200Error((self.lib.phb_last_error() or b"").decode() or "phb_comm_init_rank failed")

    def size(self) -> int:
        return int(self.lib.phb_comm_size(self.h))

    def rank(self) -> int:
        return int(self.lib.phb_comm_rank(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.phb_comm_free(self.h)
            self.h = None


class SingleTreeLikelihood:
    """One tree likelihood on one GPU (mirrors `struct _SingleTreeLikelihood`, treelikelihood.h:46-124)."""

    def __init__(self, left, right, root, nstate, ncat, npatterns, use_tip_states=True, device=0):
        self.lib = load_library()
        self.left = np.ascontiguousarray(left, dtype=np.int32)
        self.right = np.ascontiguousarray(right, dtype=np.int32)
        self.N = int(self.left.shape[0])
        self.T = (self.N + 1) // 2
        self.S, self.C, self.P = int(nstate), int(ncat), int(npatterns)
        self.root = int(root)
        self.device = int(device)
        self.h = self.lib.phb_tlk_create(self.T, self.S, self.C, self.P, self.left.ctypes.data_as(_ip),
                                         self.right.ctypes.data_as(_ip), self.root, int(bool(use_tip_states)), int(device))
        if not self.h:
            raise PhysherB200Error(self._err())

    # -- plumbing ---------------------------------------------------------------------------
    def _err(self) -> str:
        return (self.lib.phb_last_error() or b"").decode()

    def _check(self, rc: int):
        if rc != 0:
            raise PhysherB200Error(f"[{rc}] {self._err()}")

    def clone(self, device=None):
        """clone_SingleTreeLikelihood (treelikelihood.c:1241-1395): an independent object, optionally on another device."""
        h = self.lib.phb_tlk_clone(self.h, int(self.device if device is None else device))
        if not h:
            raise PhysherB200Error(self._err())
        other = object.__new__(type(self))
        other.__dict__.update({k: v for k, v in self.__dict__.items() if k != "h"})
        other.left, other.right = self.left.copy(), self.right.copy()
        other.device = int(self.device if device is None else device)
        other.h = h
        return other

    def set_topology(self, left, right, root):
        """A topology move (NNI / SPR): same taxa and node-id convention, new child arrays; everything else is kept."""
        left = np.ascontiguousarray(left, dtype=np.int32)
        right = np.ascontiguousarray(right, dtype=np.int32)
        assert left.shape == (self.N,) and right.shape == (self.N,)
        self._check(self.lib.phb_tlk_set_topology(self.h, left.ctypes.data_as(_ip), right.ctypes.data_as(_ip), int(root)))
        self.left, self.right, self.root = left, right, int(root)

    def close(self):
        if getattr(self, "h", None):
            self.lib.phb_tlk_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @classmethod
    def from_problem(cls, pb, device=0, kernels=KERNELS_AUTO):
        """Build from a plain-array problem description (attributes left, right, root, nstate, ...) and push every input."""
        tlk = cls(pb.left, pb.right, pb.root, pb.nstate, pb.ncat, pb.npatterns, use_tip_states=pb.use_tip_states, device=device)
        if pb.use_tip_states:
            tlk.set_tip_states(pb.tip_states)
        else:
            tlk.set_tip_partials(pb.tip_partials)
        tlk.set_pattern_weights(pb.weights)
        if pb.evec is not None:
            tlk.set_eigen(pb.evec, pb.eval, pb.ivec)
        else:
            tlk.set_matrices(pb.P_override, pb.dP_override)
        tlk.set_frequencies(pb.freqs)
        tlk.set_site_model(pb.rates, pb.props)
        tlk.set_branch_lengths(pb.bl)
        tlk.set_option(OPT_UNROOTED, int(pb.unrooted))
        tlk.set_option(OPT_INCLUDE_ROOT_FREQS, int(pb.include_root_freqs))
        tlk.set_option(OPT_COMPAT_SCALED_GRADIENT, int(pb.compat_scaled_gradient))
        tlk.set_option(OPT_KERNELS, kernels)
        if pb.scale:
            tlk.use_rescaling(True)
        return tlk

    # -- inputs -----------------------------------------------------------------------------
    def set_tip_states(self, states):
        a = np.ascontiguousarray(states, dtype=np.uint8)
        assert a.shape == (self.T, self.P)
        self._check(self.lib.phb_tlk_set_tip_states(self.h, a.ctypes.data_as(_bp)))

    def set_tip_partials(self, partials):
        a = _f64(partials)
        assert a.shape == (self.T, self.P, self.S)
        self._check(self.lib.phb_tlk_set_tip_partials(self.h, a.ctypes.data_as(_dp)))

    def set_pattern_weights(self, w):
        a = _f64(w)
        assert a.shape == (self.P,)
        self._check(self.lib.phb_tlk_set_pattern_weights(self.h, a.ctypes.data_as(_dp)))

    def set_eigen(self, evec, eval_, ivec):
        e, v, i = _f64(evec), _f64(eval_), _f64(ivec)
        assert e.shape == (self.S, self.S) and v.shape == (self.S,) and i.shape == (self.S, self.S)
        self._check(self.lib.phb_tlk_set_eigen(self.h, e.ctypes.data_as(_dp), v.ctypes.data_as(_dp), i.ctypes.data_as(_dp)))

    def set_matrices(self, P, dP):
        a, b = _f64(P), _f64(dP)
        assert a.shape == (self.N, self.C, self.S, self.S) == b.shape
        self._check(self.lib.phb_tlk_set_matrices(self.h, a.ctypes.data_as(_dp), b.ctypes.data_as(_dp)))

    def set_frequencies(self, freqs):
        a = _f64(freqs)
        assert a.shape == (self.S,)
        self._check(self.lib.phb_tlk_set_frequencies(self.h, a.ctypes.data_as(_dp)))

    def set_site_model(self, rates, props):
        r, p = _f64(rates), _f64(props)
        assert r.shape == (self.C,) == p.shape
        self._check(self.lib.phb_tlk_set_site_model(self.h, r.ctypes.data_as(_dp), p.ctypes.data_as(_dp)))

    def set_branch_lengths(self, bl):
        a = _f64(bl)
        assert a.shape == (self.N,)
        self._check(self.lib.phb_tlk_set_branch_lengths(self.h, a.ctypes.data_as(_dp)))

    def set_branch_length(self, node, bl):
        self._check(self.lib.phb_tlk_set_branch_length(self.h, int(node), float(bl)))

    def set_option(self, option, value):
        self._check(self.lib.phb_tlk_set_option(self.h, int(option), int(value)))

    # -- reference-named operations -----------------------------------------------------------
    def update_all_nodes(self):
        self.lib.phb_tlk_update_all_nodes(self.h)

    def update_one_node(self, node):
        self._check(self.lib.phb_tlk_update_one_node(self.h, int(node)))

    def update_three_nodes(self, node):
        self._check(self.lib.phb_tlk_update_three_nodes(self.h, int(node)))

    def store(self):
        self._check(self.lib.phb_tlk_store(self.h))

    def restore(self):
        self._check(self.lib.phb_tlk_restore(self.h))

    def use_rescaling(self, use: bool):
        self._check(self.lib.phb_tlk_use_rescaling(self.h, int(use)))

    def rescaling(self) -> bool:
        return bool(self.lib.phb_tlk_rescaling(self.h))

    def calculate(self) -> float:
        out = C.c_double(0.0)
        self._check(self.lib.phb_tlk_calculate(self.h, C.byref(out)))
        return out.value

    def pattern_log_likelihoods(self):
        out = np.zeros(self.P)
        self._check(self.lib.phb_tlk_pattern_log_likelihoods(self.h, out.ctypes.data_as(_dp)))
        return out

    def initialize_gradient(self, flags=FLAG_TREE_MODEL) -> int:
        return int(self.lib.phb_tlk_initialize_gradient(self.h, int(flags)))

    def gradient(self):
        """TreeLikelihood_gradient: copy of the tlk-owned gradient buffer (branch lengths by node id)."""
        ptr = _dp()
        self._check(self.lib.phb_tlk_gradient(self.h, C.byref(ptr)))
        return np.ctypeslib.as_array(ptr, shape=(self.N,)).copy()

    def cat_branch_gradient(self):
        out = np.zeros((self.N, self.C))
        self._check(self.lib.phb_tlk_cat_branch_gradient(self.h, out.ctypes.data_as(_dp)))
        return out

    def matrix_gradient(self, M):
        """calculate_dlnl_dQ's node sweep for sets of per-node matrices M [nsets][N][C][S][S] (e.g. dP/d theta)."""
        a = _f64(M)
        assert a.ndim == 5 and a.shape[1:] == (self.N, self.C, self.S, self.S)
        out = np.zeros(a.shape[0])
        self._check(self.lib.phb_tlk_matrix_gradient(self.h, a.shape[0], a.ctypes.data_as(_dp), out.ctypes.data_as(_dp)))
        return out

    def root_frequency_gradient(self):
        """d lnL / d pi_i at fixed partials: the root term of the frequency parameters in calculate_dlnl_dQ (treelikelihood.c:2371-2404)."""
        out = np.zeros(self.S)
        self._check(self.lib.phb_tlk_root_frequency_gradient(self.h, out.ctypes.data_as(_dp)))
        return out

    def category_gradient(self):
        """d lnL / d prop_c at fixed conditional likelihoods (root term of gradient_pinv_sitemodel, treelikelihood.c:2943-3001)."""
        out = np.zeros(self.C)
        self._check(self.lib.phb_tlk_category_gradient(self.h, out.ctypes.data_as(_dp)))
        return out

    def update_uppers(self):
        """SingleTreeLikelihood_update_uppers (treelikelihood.c:1530-1538): lnL, then every upper partial, kept on the device."""
        self._check(self.lib.phb_tlk_update_uppers(self.h))

    def calculate_branch(self, node, bl):
        """_calculate_uppper + calculate_dldt_uppper + d2lnldt2_uppper (treelikelihood.c:2592-2686, 2195-2335) for candidate
        lengths `bl` of the branch above `node`: arrays lnL, d lnL/dt, d2 lnL/dt2."""
        a = np.atleast_1d(_f64(bl))
        lnl, d1, d2 = np.zeros(a.size), np.zeros(a.size), np.zeros(a.size)
        self._check(self.lib.phb_tlk_calculate_branch(self.h, int(node), int(a.size), a.ctypes.data_as(_dp), lnl.ctypes.data_as(_dp),
                                                      d1.ctypes.data_as(_dp), d2.ctypes.data_as(_dp)))
        return lnl, d1, d2

    def branch_hessian_diagonal(self):
        """lnL, d lnL/dt_n and d2 lnL/dt_n^2 of every branch (by node id) at the current lengths, in one call: (lnl, grad[N], hess[N]).
        hess[n] is what calculate_branch(n, [t_n]) returns as d2 lnL/dt2 (d2lnldt2_uppper, treelikelihood.c:2267-2335)."""
        lnl = C.c_double(0.0)
        grad, hess = np.zeros(self.N), np.zeros(self.N)
        self._check(self.lib.phb_tlk_branch_hessian_diagonal(self.h, C.byref(lnl), grad.ctypes.data_as(_dp), hess.ctypes.data_as(_dp)))
        return lnl.value, grad, hess

    def nni_moves(self):
        """The NNI neighbourhood of the current tree as moves (x, y), int32 [n, 2] (see phb_tlk_nni_moves; PHB_OPT_UNROOTED decides
        whether the moves across the root replace the rooted moves at the root's children)."""
        n = self.lib.phb_tlk_nni_moves(self.h, None)
        if n < 0:
            self._check(n)
        moves = np.zeros((n, 2), dtype=np.int32)
        if n:
            self.lib.phb_tlk_nni_moves(self.h, moves.ctypes.data_as(_ip))
        return moves

    def nni_scores(self, moves=None, t_central=None):
        """lnL, d lnL/dt_v and d2 lnL/dt_v2 of the tree each move (x, y) produces, its central branch (above v = parent[y]) at
        t_central[k] (None: the current length), in one call on resident partials: (lnl of the current tree, out[n, 3]).
        moves=None scores the whole neighbourhood, nni_moves()."""
        m = self.nni_moves() if moves is None else np.ascontiguousarray(moves, dtype=np.int32).reshape(-1, 2)
        tc = None if t_central is None else np.ascontiguousarray(t_central, dtype=np.float64).reshape(-1)
        if tc is not None and tc.shape[0] != m.shape[0]:
            raise ValueError("t_central needs one length per move")
        out = np.zeros((m.shape[0], 3))
        lnl = C.c_double(0.0)
        self._check(self.lib.phb_tlk_nni_scores(self.h, int(m.shape[0]), m.ctypes.data_as(_ip), None if tc is None else tc.ctypes.data_as(_dp),
                                                C.byref(lnl), out.ctypes.data_as(_dp)))
        return lnl.value, out

    def spr_targets(self, s):
        """The regraft targets of the subtree of s, int32 [n] (see phb_tlk_spr_targets; PHB_OPT_UNROOTED decides whether targets that
        give the same unrooted tree are listed once)."""
        n = self.lib.phb_tlk_spr_targets(self.h, int(s), None)
        if n < 0:
            self._check(n)
        targets = np.zeros(n, dtype=np.int32)
        if n:
            self.lib.phb_tlk_spr_targets(self.h, int(s), targets.ctypes.data_as(_ip))
        return targets

    def spr_scores(self, s, targets=None, t_pendant=None):
        """lnL, d lnL/dt_s and d2 lnL/dt_s2 of the tree the subtree of s (pruned with its parent) regrafted on the branch above each
        target gives, its pendant branch (above s) at t_pendant[k] (None: the current length), in one call on resident partials:
        (lnl of the current tree, out[n, 3]).  targets=None scores every target of spr_targets(s)."""
        tg = self.spr_targets(s) if targets is None else np.ascontiguousarray(targets, dtype=np.int32).reshape(-1)
        tp = None if t_pendant is None else np.ascontiguousarray(t_pendant, dtype=np.float64).reshape(-1)
        if tp is not None and tp.shape[0] != tg.shape[0]:
            raise ValueError("t_pendant needs one length per target")
        out = np.zeros((tg.shape[0], 3))
        lnl = C.c_double(0.0)
        self._check(self.lib.phb_tlk_spr_scores(self.h, int(s), int(tg.shape[0]), tg.ctypes.data_as(_ip),
                                                None if tp is None else tp.ctypes.data_as(_dp), C.byref(lnl), out.ctypes.data_as(_dp)))
        return lnl.value, out

    def update_partials(self, out, p1, m1, p2=-1, m2=-1, mirror=True):
        """tlk->update_partials(tlk, out, p1, m1, p2, m2) (treelikelihood.h:91) on the resident device buffers; returns the result."""
        buf = np.zeros((self.C, self.P, self.S)) if mirror else None
        self._check(self.lib.phb_tlk_update_partials(self.h, int(out), int(p1), int(m1), int(p2), int(m2), buf.ctypes.data_as(_dp) if mirror else None))
        return buf

    def get_partials(self, index):
        out = np.zeros((self.C, self.P, self.S))
        self._check(self.lib.phb_tlk_get_partials(self.h, int(index), out.ctypes.data_as(_dp)))
        return out

    def get_matrices(self):
        Pm = np.zeros((self.N, self.C, self.S, self.S))
        dPm = np.zeros_like(Pm)
        self._check(self.lib.phb_tlk_get_matrices(self.h, Pm.ctypes.data_as(_dp), dPm.ctypes.data_as(_dp)))
        return Pm, dPm

    # -- multi-GPU / batched ------------------------------------------------------------------
    def gradient_device(self, out_ptr: int):
        """[lnL, grad[0..N)] of this shard into device memory at `out_ptr`, ordered on the tlk stream."""
        self._check(self.lib.phb_tlk_gradient_device(self.h, C.c_void_p(out_ptr)))

    def gradient_allreduce_device(self, comm) -> int:
        """This rank's shard evaluated and [lnL, grad[N], inf flag] all-reduced in place over `comm` (NCCL, on the tlk's stream);
        only enqueues.  Returns the device address of the tlk-owned [N + 2] buffer."""
        out = C.c_void_p(0)
        self._check(self.lib.phb_tlk_gradient_allreduce_device(self.h, comm.h if comm is not None else None, C.byref(out)))
        return int(out.value or 0)

    def gradient_allreduce(self, comm):
        """(lnL, gradient) of the WHOLE alignment on every rank, the reference's inf / NaN / unrooted conventions applied to the
        reduced values."""
        lnl, ptr = C.c_double(0.0), _dp()
        self._check(self.lib.phb_tlk_gradient_allreduce(self.h, comm.h if comm is not None else None, C.byref(lnl), C.byref(ptr)))
        return lnl.value, np.ctypeslib.as_array(ptr, shape=(self.N,)).copy()

    def stream(self) -> int:
        return int(self.lib.phb_tlk_stream(self.h) or 0)

    def synchronize(self):
        self._check(self.lib.phb_tlk_synchronize(self.h))

    def gradient_batch(self, bl, want_gradient=True):
        a = _f64(bl)
        assert a.ndim == 2 and a.shape[1] == self.N
        B = a.shape[0]
        lnl = np.zeros(B)
        grad = np.zeros((B, self.N)) if want_gradient else None
        self._check(self.lib.phb_tlk_gradient_batch(self.h, B, a.ctypes.data_as(_dp), lnl.ctypes.data_as(_dp),
                                                    grad.ctypes.data_as(_dp) if want_gradient else None))
        return lnl, grad

    # -- time trees ---------------------------------------------------------------------------
    def set_time_tree(self, tip_heights):
        a = _f64(tip_heights)
        assert a.shape == (self.T,)
        self._check(self.lib.phb_tlk_set_time_tree(self.h, a.ctypes.data_as(_dp)))

    def gradient_batch_time(self, ratios, rates, include_jacobian=False, want_gradient=True):
        """B samples of (ratios | root height)[T-1] and clock rates -> lnl[B], log_jacobian[B], grad_ratios[B][T-1], grad_rates[B][R]."""
        r, c = _f64(ratios), _f64(rates)
        assert r.ndim == 2 and r.shape[1] == self.T - 1 and c.ndim == 2 and c.shape[0] == r.shape[0] and c.shape[1] in (1, self.N)
        B, R = r.shape[0], c.shape[1]
        lnl, lj = np.zeros(B), np.zeros(B)
        gr = np.zeros((B, self.T - 1)) if want_gradient else None
        gc = np.zeros((B, R)) if want_gradient else None
        self._check(self.lib.phb_tlk_gradient_batch_time(
            self.h, B, r.ctypes.data_as(_dp), c.ctypes.data_as(_dp), R, int(bool(include_jacobian)), lnl.ctypes.data_as(_dp),
            lj.ctypes.data_as(_dp), gr.ctypes.data_as(_dp) if want_gradient else None, gc.ctypes.data_as(_dp) if want_gradient else None))
        return lnl, lj, gr, gc

    def kernel_time(self):
        """(total ms, launches) of the dominant kernel since OPT_TIMING was switched on."""
        ms, n = C.c_double(0.0), C.c_longlong(0)
        self._check(self.lib.phb_tlk_kernel_time(self.h, C.byref(ms), C.byref(n)))
        return ms.value, int(n.value)

    def launch_count(self) -> int:
        return int(self.lib.phb_tlk_launch_count(self.h))

    def last_kernels(self) -> int:
        """Kernel family of the last evaluation: RAN_GENERIC, RAN_WALK (fused 4-state walk) or RAN_TENSOR (FP64 tensor cores)."""
        return int(self.lib.phb_tlk_last_kernels(self.h))


class TreeLikelihoodGroup:
    """One tree likelihood sharded over several GPUs from one host thread (phb_group, csrc/phb_group.c): pattern-indexed inputs for the
    whole alignment, model inputs broadcast, every evaluation launched on all shards before any result is collected."""

    def __init__(self, devices, left, right, root, nstate, ncat, npatterns, use_tip_states=True):
        if len(set(int(d) for d in devices)) > 1:
            _preload_nccl()  # the group reduces over NCCL when its shards sit on distinct devices
        self.lib = load_library()
        self.left = np.ascontiguousarray(left, dtype=np.int32)
        self.right = np.ascontiguousarray(right, dtype=np.int32)
        self.N = int(self.left.shape[0])
        self.T = (self.N + 1) // 2
        self.S, self.C, self.P = int(nstate), int(ncat), int(npatterns)
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        self.h = self.lib.phb_group_create(int(dev.size), dev.ctypes.data_as(_ip), self.T, self.S, self.C, self.P, self.left.ctypes.data_as(_ip),
                                           self.right.ctypes.data_as(_ip), int(root), int(bool(use_tip_states)))
        if not self.h:
            raise PhysherB200Error((self.lib.phb_last_error() or b"").decode() or "phb_group_create failed")

    @classmethod
    def from_problem(cls, pb, devices):
        g = cls(devices, pb.left, pb.right, pb.root, pb.nstate, pb.ncat, pb.npatterns, use_tip_states=pb.use_tip_states)
        if pb.use_tip_states:
            a = np.ascontiguousarray(pb.tip_states, dtype=np.uint8)
            g._check(g.lib.phb_group_set_tip_states(g.h, a.ctypes.data_as(_bp)))
        else:
            g._check(g.lib.phb_group_set_tip_partials(g.h, _f64(pb.tip_partials).ctypes.data_as(_dp)))
        g._check(g.lib.phb_group_set_pattern_weights(g.h, _f64(pb.weights).ctypes.data_as(_dp)))
        g._check(g.lib.phb_group_set_eigen(g.h, _f64(pb.evec).ctypes.data_as(_dp), _f64(pb.eval).ctypes.data_as(_dp), _f64(pb.ivec).ctypes.data_as(_dp)))
        g._check(g.lib.phb_group_set_frequencies(g.h, _f64(pb.freqs).ctypes.data_as(_dp)))
        g._check(g.lib.phb_group_set_site_model(g.h, _f64(pb.rates).ctypes.data_as(_dp), _f64(pb.props).ctypes.data_as(_dp)))
        g.set_branch_lengths(pb.bl)
        g.set_option(OPT_UNROOTED, int(pb.unrooted))
        if getattr(pb, "scale", False):
            g.use_rescaling(True)
        return g

    def _check(self, rc):
        if rc != 0:
            raise PhysherB200Error(f"[{rc}] {(self.lib.phb_last_error() or b'').decode()}")

    def size(self):
        return int(self.lib.phb_group_size(self.h))

    def shard_range(self, shard):
        b, e = C.c_int(0), C.c_int(0)
        self._check(self.lib.phb_group_shard_range(self.h, int(shard), C.byref(b), C.byref(e)))
        return b.value, e.value

    def set_branch_lengths(self, bl):
        a = _f64(bl)
        assert a.shape == (self.N,)
        self._check(self.lib.phb_group_set_branch_lengths(self.h, a.ctypes.data_as(_dp)))

    def set_option(self, option, value):
        self._check(self.lib.phb_group_set_option(self.h, int(option), int(value)))

    def use_rescaling(self, use):
        self._check(self.lib.phb_group_use_rescaling(self.h, int(bool(use))))

    def rescaling(self):
        return bool(self.lib.phb_group_rescaling(self.h))

    def set_reduction(self, how):
        self._check(self.lib.phb_group_set_reduction(self.h, int(how)))

    def reduction(self) -> int:
        return int(self.lib.phb_group_reduction(self.h))

    def calculate(self):
        v = C.c_double(0.0)
        self._check(self.lib.phb_group_calculate(self.h, C.byref(v)))
        return v.value

    def gradient(self):
        v, p = C.c_double(0.0), _dp()
        self._check(self.lib.phb_group_gradient(self.h, C.byref(v), C.byref(p)))
        return v.value, np.ctypeslib.as_array(p, shape=(self.N,)).copy()

    def close(self):
        if getattr(self, "h", None):
            self.lib.phb_group_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
