"""Python host-side mirror of the C ABI in include/bfhe.h (ctypes; plumbing only).

The product is the sm_100a shared library ``libbfhe_b200.so`` built in-tree by ``build.py``;
this module binds it 1:1.  It contains no arithmetic and no fallback: if the library is missing,
import fails loudly; if no CUDA device is present, every Eval* call raises BfheError.

Directory name contains '-', so import it through ``load_package()`` in ``bfhe_loader.py`` at the repo
root (tests/conftest.py and bench.py do), which registers it as module ``bfhe_b200``.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbfhe_b200.so")

TOY, STD128_OPT = 0, 5
AP, GINX = 0, 1
OR, AND, NOR, NAND, XOR_FAST, XNOR_FAST, XOR, XNOR, BOOTSTRAP = range(9)
NEG0, NEG1 = 0x100, 0x200
OFHE_SECRET_KEY, OFHE_REFRESH_KEY, OFHE_SWITCH_KEY = 0, 1, 2
ERR_ARG, ERR_STATE, ERR_CUDA, ERR_FORMAT, ERR_ALIAS, ERR_NCCL, ERR_IO = -1, -2, -3, -4, -5, -6, -7

# netlist gate kinds: GateEnum of the reference (src/gate.h:51), then EvalBinGate's other native gate types
(K_INPUT, K_OUTPUT, K_NOT, K_AND, K_OR, K_XOR, K_DFF, K_LUT3, K_LUT4, K_NAND, K_NOR, K_XNOR, K_XOR_FAST, K_XNOR_FAST) = range(14)

GATE_DTYPE = np.dtype([("op", "<u4"), ("in0", "<u4"), ("in1", "<u4"), ("out", "<u4")])


class Params(C.Structure):
    _fields_ = [("paramset", C.c_uint32), ("method", C.c_uint32), ("n", C.c_uint32), ("N", C.c_uint32),
                ("q", C.c_uint32), ("Q", C.c_uint64), ("qKS", C.c_uint64), ("baseKS", C.c_uint32),
                ("dKS", C.c_uint32), ("baseG", C.c_uint32), ("dG", C.c_uint32), ("baseR", C.c_uint32),
                ("dR", C.c_uint32), ("ct_words", C.c_uint32), ("ct_stride", C.c_uint32)]


class BfheError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("bfhe error %d: %s" % (code, msg))
        self.code = code


# every symbol include/bfhe.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "bfhe_create", "bfhe_destroy", "bfhe_get_params", "bfhe_last_error", "bfhe_set_stream", "bfhe_sync",
    "bfhe_keygen", "bfhe_btkeygen", "bfhe_keyblob_size", "bfhe_export_keys", "bfhe_import_keys", "bfhe_save_keys",
    "bfhe_load_keys", "bfhe_encrypt", "bfhe_decrypt", "bfhe_slab_alloc", "bfhe_slab_free", "bfhe_slab_upload",
    "bfhe_slab_download", "bfhe_eval_not_batch", "bfhe_eval_bingate_batch", "bfhe_bootstrap_batch",
    "bfhe_eval_bingate_host", "bfhe_profile_enable", "bfhe_profile_read", "bfhe_microbench_int",
    "bfhe_dbg_ntt_roundtrip", "bfhe_dbg_blind_rotate", "bfhe_dbg_set_gates_per_cta", "bfhe_dbg_cluster_limits",
    "bfhe_circuit_create", "bfhe_circuit_destroy", "bfhe_circuit_read_file", "bfhe_circuit_read_bristol",
    "bfhe_circuit_set_flags", "bfhe_circuit_info", "bfhe_circuit_set_sharding", "bfhe_get_nccl_unique_id",
    "bfhe_circuit_set_wave_capacity",
    "bfhe_circuit_reset", "bfhe_circuit_set_input", "bfhe_circuit_clock", "bfhe_circuit_stats",
    "bfhe_circuit_level_plan", "bfhe_circuit_plan_misc", "bfhe_circuit_use_graph", "bfhe_circuit_download_slab",
    "bfhe_circuit_dump_gate_count", "bfhe_circuit_load_netlist", "bfhe_circuit_get_netlist", "bfhe_circuit_write_out",
    "bfhe_circuit_load_netlist_ex", "bfhe_circuit_set_shard_threshold", "bfhe_circuit_dump_gate_count_ex",
    "bfhe_circuit_dump_text", "bfhe_circuit_dff_plan", "bfhe_circuit_get_schedule",
    "bfhe_circuit_exchange_mode", "bfhe_circuit_set_input_ct", "bfhe_circuit_clock_ct",
    "bfhe_import_openfhe_json", "bfhe_export_openfhe_json", "bfhe_import_openfhe_ct_json", "bfhe_export_openfhe_ct_json",
    "bfhe_btkeygen_compact", "bfhe_keyblob_compact_size", "bfhe_export_keys_compact", "bfhe_dbg_expand_keys",
]

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("libbfhe_b200.so is not built: run `python __graft_entry__.py` (build()) first; "
                          "there is no fallback implementation")
    L = C.CDLL(LIB_PATH)
    vp, u32p, u8p, sz = C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.c_size_t
    L.bfhe_create.restype = vp
    L.bfhe_create.argtypes = [C.c_int, C.c_int, C.c_int]
    L.bfhe_destroy.argtypes = [vp]
    L.bfhe_destroy.restype = None
    L.bfhe_get_params.argtypes = [vp, C.POINTER(Params)]
    L.bfhe_last_error.restype = C.c_char_p
    L.bfhe_set_stream.argtypes = [vp, vp, C.c_int]
    L.bfhe_sync.argtypes = [vp]
    L.bfhe_keygen.argtypes = [vp, C.c_uint64]
    L.bfhe_btkeygen.argtypes = [vp, C.c_uint64]
    L.bfhe_keyblob_size.restype = sz
    L.bfhe_keyblob_size.argtypes = [vp]
    L.bfhe_export_keys.argtypes = [vp, vp, sz, C.c_int]
    L.bfhe_import_keys.argtypes = [vp, vp, sz]
    L.bfhe_btkeygen_compact.argtypes = [vp, C.c_uint64]
    L.bfhe_keyblob_compact_size.restype = sz
    L.bfhe_keyblob_compact_size.argtypes = [vp]
    L.bfhe_export_keys_compact.argtypes = [vp, vp, sz, C.c_int]
    L.bfhe_dbg_expand_keys.argtypes = [vp, vp, sz, vp, sz]
    L.bfhe_save_keys.argtypes = [vp, C.c_char_p, C.c_int]
    L.bfhe_load_keys.argtypes = [vp, C.c_char_p]
    L.bfhe_encrypt.argtypes = [vp, vp, sz, C.c_uint64, vp]
    L.bfhe_decrypt.argtypes = [vp, vp, sz, vp]
    L.bfhe_slab_alloc.argtypes = [vp, sz, C.POINTER(vp)]
    L.bfhe_slab_free.argtypes = [vp, vp]
    L.bfhe_slab_upload.argtypes = [vp, vp, sz, vp, sz]
    L.bfhe_slab_download.argtypes = [vp, vp, sz, vp, sz]
    L.bfhe_eval_not_batch.argtypes = [vp, vp, vp, vp, sz]
    L.bfhe_eval_bingate_batch.argtypes = [vp, vp, vp, sz]
    L.bfhe_bootstrap_batch.argtypes = [vp, vp, vp, vp, sz]
    L.bfhe_eval_bingate_host.argtypes = [vp, vp, sz, vp, sz, vp, sz]
    L.bfhe_profile_enable.argtypes = [vp, C.c_int]
    L.bfhe_profile_read.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.bfhe_microbench_int.argtypes = [vp, C.c_int, C.POINTER(C.c_double)]
    L.bfhe_dbg_ntt_roundtrip.argtypes = [vp, vp, sz, vp, vp, vp]
    L.bfhe_dbg_blind_rotate.argtypes = [vp, vp, vp, sz, vp]
    L.bfhe_dbg_set_gates_per_cta.argtypes = [vp, C.c_int]
    L.bfhe_dbg_cluster_limits.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.bfhe_circuit_create.restype = vp
    L.bfhe_circuit_create.argtypes = [vp]
    L.bfhe_circuit_destroy.restype = None
    L.bfhe_circuit_destroy.argtypes = [vp]
    L.bfhe_circuit_read_file.argtypes = [vp, C.c_char_p]
    L.bfhe_circuit_read_bristol.argtypes = [vp, C.c_char_p, C.c_int]
    L.bfhe_circuit_set_flags.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.bfhe_circuit_info.argtypes = [vp, u32p, u32p, u32p, u32p, u32p, u32p, u32p]
    L.bfhe_circuit_set_sharding.argtypes = [vp, C.c_int, C.c_int, vp]
    L.bfhe_circuit_set_wave_capacity.argtypes = [vp, C.c_int]
    L.bfhe_get_nccl_unique_id.argtypes = [vp]
    L.bfhe_circuit_reset.argtypes = [vp]
    L.bfhe_circuit_set_input.argtypes = [vp, vp, sz, C.c_uint64]
    L.bfhe_circuit_clock.argtypes = [vp, vp, sz, vp]
    L.bfhe_circuit_set_input_ct.argtypes = [vp, vp, sz, C.c_int]
    L.bfhe_circuit_clock_ct.argtypes = [vp, vp, sz, C.c_int]
    L.bfhe_circuit_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.bfhe_circuit_level_plan.argtypes = [vp, C.c_uint32, C.c_int, C.c_int, vp, sz, u32p, u32p, u32p]
    L.bfhe_circuit_plan_misc.argtypes = [vp, u32p, u32p, u32p, vp, u32p, C.c_uint32, vp]
    L.bfhe_circuit_use_graph.argtypes = [vp, C.c_int]
    L.bfhe_circuit_download_slab.argtypes = [vp, vp, sz]
    L.bfhe_circuit_dump_gate_count.argtypes = [vp, u32p, u32p, u32p, u32p, u32p, u32p]
    L.bfhe_circuit_load_netlist.argtypes = [vp, vp, vp, vp, vp, sz, C.c_uint32, vp, C.c_uint32, C.c_uint32]
    L.bfhe_circuit_get_netlist.argtypes = [vp, vp, vp, vp, vp, sz, u32p, u32p]
    L.bfhe_circuit_write_out.argtypes = [vp, C.c_char_p]
    L.bfhe_circuit_load_netlist_ex.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, sz, C.c_uint32, vp, C.c_uint32, C.c_uint32]
    L.bfhe_circuit_set_shard_threshold.argtypes = [vp, C.c_int]
    L.bfhe_circuit_dump_gate_count_ex.argtypes = [vp, u32p]
    L.bfhe_circuit_dump_text.argtypes = [vp, C.c_int, C.c_char_p, sz, C.POINTER(sz)]
    L.bfhe_circuit_dff_plan.argtypes = [vp, u32p, vp, sz]
    L.bfhe_circuit_get_schedule.argtypes = [vp, u32p, u32p, u32p, C.POINTER(C.c_double)]
    L.bfhe_circuit_exchange_mode.argtypes = [vp]
    L.bfhe_import_openfhe_json.argtypes = [vp, C.c_int, C.c_char_p]
    L.bfhe_export_openfhe_json.argtypes = [vp, C.c_int, C.c_char_p]
    L.bfhe_import_openfhe_ct_json.argtypes = [vp, C.c_char_p, vp]
    L.bfhe_export_openfhe_ct_json.argtypes = [vp, vp, C.c_char_p]
    _lib = L
    return L


def _ptr(a):
    return a.ctypes.data if a is not None else None


class Slab:
    """A device array of ciphertext rows (wire storage)."""

    def __init__(self, ctx, rows):
        self.ctx, self.rows = ctx, rows
        p = C.c_void_p()
        ctx._ck(ctx.L.bfhe_slab_alloc(ctx.h, rows, C.byref(p)))
        self.ptr = p.value

    def upload(self, host, first_row=0):
        host = np.ascontiguousarray(host, dtype=np.uint32)
        assert host.ndim == 2 and host.shape[1] == self.ctx.stride
        self.ctx._ck(self.ctx.L.bfhe_slab_upload(self.ctx.h, self.ptr, first_row, _ptr(host), host.shape[0]))
        self.ctx.sync()

    def download(self, first_row=0, rows=None):
        rows = self.rows - first_row if rows is None else rows
        out = np.empty((rows, self.ctx.stride), dtype=np.uint32)
        self.ctx._ck(self.ctx.L.bfhe_slab_download(self.ctx.h, self.ptr, first_row, _ptr(out), rows))
        return out

    def free(self):
        if self.ptr:
            self.ctx.L.bfhe_slab_free(self.ctx.h, self.ptr)
            self.ptr = None

    def range(self, first_row=0, rows=None):
        """rows [first_row, first_row + rows) as a device buffer for Circuit.set_input_ct / clock_ct"""
        rows = self.rows - first_row if rows is None else rows
        if first_row < 0 or rows < 0 or first_row + rows > self.rows:
            raise ValueError("rows %d..%d outside a slab of %d rows" % (first_row, first_row + rows, self.rows))
        return SlabRows(self, first_row, rows)


class SlabRows:
    """A row range of a Slab (Slab.range)."""

    def __init__(self, slab, first_row, rows):
        self.slab, self.first_row, self.rows = slab, first_row, rows
        self.ptr = slab.ptr + first_row * slab.ctx.stride * 4


def _device_rows(buf, stride):
    """(device pointer, rows) of a Slab, a SlabRows or an object exposing __cuda_array_interface__ with shape (rows, stride), 4-byte
    integers and C-contiguous layout.  The library checks that the memory is on the context's device."""
    if isinstance(buf, (Slab, SlabRows)):
        if buf.ptr is None:
            raise ValueError("slab has been freed")
        return buf.ptr, buf.rows
    cai = getattr(buf, "__cuda_array_interface__", None)
    if cai is None:
        raise TypeError("expected a Slab, Slab.range(...) or an object with __cuda_array_interface__, got %s" % type(buf).__name__)
    shape = tuple(cai["shape"])
    if len(shape) != 2 or shape[1] != stride:
        raise ValueError("device buffer shape %s, expected (rows, %d)" % (shape, stride))
    if cai["typestr"][1:] not in ("i4", "u4") or cai["typestr"][0] == ">":
        raise TypeError("device buffer element type %s, expected 4-byte integers (int32 or uint32)" % cai["typestr"])
    strides = cai.get("strides")
    if strides is not None and tuple(strides) != (stride * 4, 4) and shape[0] > 1:
        raise ValueError("device buffer is not C-contiguous (strides %s)" % (tuple(strides),))
    return cai["data"][0], shape[0]


class Context:
    """BinFHEContext-shaped handle: GenerateBinFHEContext / KeyGen / BTKeyGen / Encrypt / Decrypt /
    EvalNOT / EvalBinGate / Bootstrap (src/circuit.cpp:88-91,506,800; src/gate.cpp:112,133 in the reference)."""

    def __init__(self, paramset=STD128_OPT, method=GINX, device=0):
        self.L = lib()
        self.h = self.L.bfhe_create(paramset, method, device)
        if not self.h:
            raise BfheError(ERR_ARG, self.L.bfhe_last_error().decode())
        self.p = Params()
        self.L.bfhe_get_params(self.h, C.byref(self.p))
        self.stride = self.p.ct_stride
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.bfhe_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise BfheError(rc, self.L.bfhe_last_error().decode())

    # keys
    def keygen(self, seed=1):
        self._ck(self.L.bfhe_keygen(self.h, seed))

    def btkeygen(self, seed=2):
        self._ck(self.L.bfhe_btkeygen(self.h, seed))

    def export_keys(self, include_sk=True):
        n = self.L.bfhe_keyblob_size(self.h)
        buf = np.empty(n, dtype=np.uint8)
        self._ck(self.L.bfhe_export_keys(self.h, _ptr(buf), n, int(include_sk)))
        return buf

    def btkeygen_compact(self, seed=2):
        """btkeygen with every public mask expanded from a fresh mask seed, so that export_keys_compact can ship seed and bodies only"""
        self._ck(self.L.bfhe_btkeygen_compact(self.h, seed))

    def export_keys_compact(self, include_sk=True):
        """the BFHEKEY2 blob (include/bfhe.h): mask seed and bodies; keys from btkeygen_compact or a BFHEKEY2 import only"""
        n = self.L.bfhe_keyblob_compact_size(self.h)
        buf = np.empty(n, dtype=np.uint8)
        self._ck(self.L.bfhe_export_keys_compact(self.h, _ptr(buf), n, int(include_sk)))
        return buf

    def import_keys(self, blob):
        """a BFHEKEY1 (export_keys) or BFHEKEY2 (export_keys_compact) blob"""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._ck(self.L.bfhe_import_keys(self.h, _ptr(blob), blob.size))

    def save_keys(self, path, include_sk=True):
        self._ck(self.L.bfhe_save_keys(self.h, path.encode(), int(include_sk)))

    def load_keys(self, path):
        self._ck(self.L.bfhe_load_keys(self.h, path.encode()))

    # OpenFHE 1.0.x cereal JSON objects (row f-3): what = OFHE_SECRET_KEY / OFHE_REFRESH_KEY / OFHE_SWITCH_KEY
    def import_openfhe_json(self, what, path):
        self._ck(self.L.bfhe_import_openfhe_json(self.h, what, path.encode()))

    def export_openfhe_json(self, what, path):
        self._ck(self.L.bfhe_export_openfhe_json(self.h, what, path.encode()))

    def import_openfhe_ct_json(self, path):
        row = np.zeros(self.stride, dtype=np.uint32)
        self._ck(self.L.bfhe_import_openfhe_ct_json(self.h, path.encode(), _ptr(row)))
        return row

    def export_openfhe_ct_json(self, ct_row, path):
        row = np.ascontiguousarray(ct_row, dtype=np.uint32).reshape(self.stride)
        self._ck(self.L.bfhe_export_openfhe_ct_json(self.h, _ptr(row), path.encode()))

    # host LWE
    def encrypt(self, bits, seed=0):
        bits = np.ascontiguousarray(np.asarray(bits).ravel(), dtype=np.uint8)
        out = np.zeros((bits.size, self.stride), dtype=np.uint32)
        self._ck(self.L.bfhe_encrypt(self.h, _ptr(bits), bits.size, seed, _ptr(out)))
        return out

    def decrypt(self, cts):
        cts = np.ascontiguousarray(cts, dtype=np.uint32).reshape(-1, self.stride)
        out = np.zeros(cts.shape[0], dtype=np.uint8)
        self._ck(self.L.bfhe_decrypt(self.h, _ptr(cts), cts.shape[0], _ptr(out)))
        return out

    # device
    def set_stream(self, cuda_stream_handle, use_own=False):
        """cuda_stream_handle: integer cudaStream_t (0 / None = legacy default stream); use_own: private stream"""
        self._ck(self.L.bfhe_set_stream(self.h, cuda_stream_handle or None, int(use_own)))

    def sync(self):
        self._ck(self.L.bfhe_sync(self.h))

    def slab(self, rows):
        return Slab(self, rows)

    @staticmethod
    def _slab_ptr(slab):
        return slab.ptr if isinstance(slab, Slab) else int(slab)

    def eval_not_batch(self, slab, in_rows, out_rows):
        i = np.ascontiguousarray(in_rows, dtype=np.uint32)
        o = np.ascontiguousarray(out_rows, dtype=np.uint32)
        self._ck(self.L.bfhe_eval_not_batch(self.h, self._slab_ptr(slab), _ptr(i), _ptr(o), i.size))

    def eval_bingate_batch(self, slab, gates):
        g = np.ascontiguousarray(gates, dtype=GATE_DTYPE)
        self._ck(self.L.bfhe_eval_bingate_batch(self.h, self._slab_ptr(slab), _ptr(g), g.size))

    def bootstrap_batch(self, slab, in_rows, out_rows):
        i = np.ascontiguousarray(in_rows, dtype=np.uint32)
        o = np.ascontiguousarray(out_rows, dtype=np.uint32)
        self._ck(self.L.bfhe_bootstrap_batch(self.h, self._slab_ptr(slab), _ptr(i), _ptr(o), i.size))

    def eval_bingate_host(self, gates, in_host, out_rows, out_host=None):
        g = np.ascontiguousarray(gates, dtype=GATE_DTYPE)
        assert in_host.dtype == np.uint32 and in_host.flags["C_CONTIGUOUS"]
        if out_host is None:
            out_host = np.empty((out_rows, self.stride), dtype=np.uint32)
        self._ck(self.L.bfhe_eval_bingate_host(self.h, _ptr(g), g.size, _ptr(in_host), in_host.shape[0], _ptr(out_host),
                                               out_rows))
        return out_host

    # single-gate conveniences with the reference's method names (batch of one)
    def EvalBinGate(self, gate, ct1, ct2):
        inp = np.stack([np.asarray(ct1, dtype=np.uint32), np.asarray(ct2, dtype=np.uint32)])
        g = np.array([(gate, 0, 1, 2)], dtype=GATE_DTYPE)
        return self.eval_bingate_host(g, np.ascontiguousarray(inp), 1)[0]

    def EvalNOT(self, ct):
        s = self.slab(2)
        s.upload(np.asarray(ct, dtype=np.uint32).reshape(1, -1))
        self.eval_not_batch(s, [0], [1])
        out = s.download(1, 1)[0]
        s.free()
        return out

    def Bootstrap(self, ct):
        inp = np.ascontiguousarray(np.asarray(ct, dtype=np.uint32).reshape(1, -1))
        g = np.array([(BOOTSTRAP, 0, 0, 1)], dtype=GATE_DTYPE)
        return self.eval_bingate_host(g, inp, 1)[0]

    # measurement
    def profile_enable(self, on=True):
        self._ck(self.L.bfhe_profile_enable(self.h, int(on)))

    def profile_read(self, kernel):
        ms, n = C.c_double(), C.c_uint64()
        self._ck(self.L.bfhe_profile_read(self.h, kernel, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def microbench_int(self, which):
        v = C.c_double()
        self._ck(self.L.bfhe_microbench_int(self.h, which, C.byref(v)))
        return v.value

    # debug / parity
    def dbg_ntt_roundtrip(self, a, b=None):
        a = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, self.p.N)
        rt = np.empty_like(a)
        prod = np.empty_like(a) if b is not None else None
        if b is not None:
            b = np.ascontiguousarray(b, dtype=np.uint32).reshape(-1, self.p.N)
        self._ck(self.L.bfhe_dbg_ntt_roundtrip(self.h, _ptr(a), a.shape[0], _ptr(rt), _ptr(prod), _ptr(b)))
        return rt, prod

    def dbg_blind_rotate(self, slab, gates):
        g = np.ascontiguousarray(gates, dtype=GATE_DTYPE)
        acc = np.empty((g.size, 2, self.p.N), dtype=np.uint32)
        self._ck(self.L.bfhe_dbg_blind_rotate(self.h, self._slab_ptr(slab), _ptr(g), g.size, _ptr(acc)))
        return acc

    def dbg_set_gates_per_cta(self, g):
        self._ck(self.L.bfhe_dbg_set_gates_per_cta(self.h, g))

    def dbg_expand_keys(self, compact_blob):
        """import a BFHEKEY2 blob through the device expansion and return the BFHEKEY1 blob it produced"""
        blob = np.ascontiguousarray(compact_blob, dtype=np.uint8)
        n = self.L.bfhe_keyblob_size(self.h)
        out = np.zeros(n, dtype=np.uint8)
        self._ck(self.L.bfhe_dbg_expand_keys(self.h, _ptr(blob), blob.size, _ptr(out), n))
        return out

    def dbg_cluster_limits(self):
        a, b = C.c_int(), C.c_int()
        self._ck(self.L.bfhe_dbg_cluster_limits(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value


def nccl_unique_id():
    buf = np.zeros(128, dtype=np.uint8)
    rc = lib().bfhe_get_nccl_unique_id(buf.ctypes.data)
    if rc:
        raise BfheError(rc, lib().bfhe_last_error().decode())
    return buf


class Circuit:
    """Mirror of the reference's ``class Circuit`` (src/circuit.h:56-72): ReadFile / Reset / SetInput / Clock /
    set{Plaintext,Encrypted,Verify} / dumpGateCount, evaluated level-synchronously on the GPU."""

    def __init__(self, ctx):
        self.ctx, self.L = ctx, ctx.L
        self.h = self.L.bfhe_circuit_create(ctx.h)
        self._flags = [False, False, False]
        self.world_size = 1

    def close(self):
        if getattr(self, "h", None):
            self.L.bfhe_circuit_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        self.ctx._ck(rc)

    def ReadFile(self, path):
        self._ck(self.L.bfhe_circuit_read_file(self.h, str(path).encode()))
        return True

    def ReadBristol(self, path, new_format=False):
        self._ck(self.L.bfhe_circuit_read_bristol(self.h, str(path).encode(), int(new_format)))
        return True

    def load_netlist(self, kind, in0, in1, out, n_wires, in_bits, out_bits):
        kind = np.ascontiguousarray(kind, dtype=np.uint8)
        in0, in1, out = (np.ascontiguousarray(a, dtype=np.uint32) for a in (in0, in1, out))
        ib = np.ascontiguousarray(in_bits, dtype=np.uint32)
        self._ck(self.L.bfhe_circuit_load_netlist(self.h, _ptr(kind), _ptr(in0), _ptr(in1), _ptr(out), kind.size, int(n_wires),
                                                  _ptr(ib), ib.size, int(out_bits)))

    def load_netlist_ex(self, kind, in0, in1, in2, in3, table, out, n_wires, in_bits, out_bits):
        kind = np.ascontiguousarray(kind, dtype=np.uint8)
        in0, in1, in2, in3, table, out = (np.ascontiguousarray(a, dtype=np.uint32) for a in (in0, in1, in2, in3, table, out))
        ib = np.ascontiguousarray(in_bits, dtype=np.uint32)
        self._ck(self.L.bfhe_circuit_load_netlist_ex(self.h, _ptr(kind), _ptr(in0), _ptr(in1), _ptr(in2), _ptr(in3), _ptr(table), _ptr(out),
                                                     kind.size, int(n_wires), _ptr(ib), ib.size, int(out_bits)))

    def load_npz(self, path):
        d = np.load(path)
        self.load_netlist(d["kind"], d["in0"], d["in1"], d["out"], int(d["n_wires"]), d["in_bits"], int(d["out_bits"]))

    def get_netlist(self):
        cnt, nw = C.c_uint32(), C.c_uint32()
        self._ck(self.L.bfhe_circuit_get_netlist(self.h, None, None, None, None, 0, C.byref(cnt), C.byref(nw)))
        kind = np.zeros(cnt.value, dtype=np.uint8)
        in0, in1, out = (np.zeros(cnt.value, dtype=np.uint32) for _ in range(3))
        self._ck(self.L.bfhe_circuit_get_netlist(self.h, _ptr(kind), _ptr(in0), _ptr(in1), _ptr(out), cnt.value, C.byref(cnt),
                                                 C.byref(nw)))
        i = self.info()
        return dict(kind=kind, in0=in0, in1=in1, out=out, n_wires=nw.value, in_bits=np.array(i["input_bits"], dtype=np.uint32),
                    out_bits=i["output_bits"])

    def write_out(self, path):
        self._ck(self.L.bfhe_circuit_write_out(self.h, str(path).encode()))

    def info(self):
        v = [C.c_uint32() for _ in range(6)]
        bits = (C.c_uint32 * 8)()
        self._ck(self.L.bfhe_circuit_info(self.h, C.byref(v[0]), bits, C.byref(v[1]), C.byref(v[2]), C.byref(v[3]),
                                          C.byref(v[4]), C.byref(v[5])))
        return dict(n_inputs=v[0].value, input_bits=list(bits)[: v[0].value], output_bits=v[1].value, gates=v[2].value,
                    bootstraps=v[3].value, levels=v[4].value, max_width=v[5].value)

    def dumpGateCount(self):
        v = [C.c_uint32() for _ in range(6)]
        self._ck(self.L.bfhe_circuit_dump_gate_count(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("input", "output", "and", "or", "xor", "not"), [x.value for x in v]))

    def dumpGateCountEx(self):
        v = (C.c_uint32 * 8)()
        self._ck(self.L.bfhe_circuit_dump_gate_count_ex(self.h, v))
        return dict(zip(("dff", "lut3", "lut4", "nand", "nor", "xnor", "xor_fast", "xnor_fast"), list(v)))

    def _dump_text(self, what):
        need = C.c_size_t()
        self._ck(self.L.bfhe_circuit_dump_text(self.h, what, None, 0, C.byref(need)))
        buf = C.create_string_buffer(need.value + 1)
        self._ck(self.L.bfhe_circuit_dump_text(self.h, what, buf, need.value + 1, C.byref(need)))
        return buf.value.decode()

    def dumpNetList(self):
        """text of Circuit::dumpNetList (src/circuit.cpp:844-855)"""
        return self._dump_text(0)

    def dumpGates(self):
        """text of Circuit::dumpGates (src/circuit.cpp:856-865)"""
        return self._dump_text(1)

    def dff_plan(self):
        n = C.c_uint32()
        self._ck(self.L.bfhe_circuit_dff_plan(self.h, C.byref(n), None, 0))
        q = np.zeros((n.value, 4), dtype=np.uint32)
        if n.value:
            self._ck(self.L.bfhe_circuit_dff_plan(self.h, C.byref(n), _ptr(q), n.value))
        return q

    def schedule(self):
        cap, nl, ns = C.c_uint32(), C.c_uint32(), C.c_uint32()
        cost = (C.c_double * 4)()
        self._ck(self.L.bfhe_circuit_get_schedule(self.h, C.byref(cap), C.byref(nl), C.byref(ns), cost))
        return dict(wave_cap=cap.value, n_levels=nl.value, n_sharded=ns.value, cost_ms=dict(zip(("cl4", "cl2", "lat", "thr"), list(cost))))

    def set_shard_threshold(self, min_bootstraps):
        self._ck(self.L.bfhe_circuit_set_shard_threshold(self.h, min_bootstraps))

    def _push_flags(self):
        self._ck(self.L.bfhe_circuit_set_flags(self.h, *[int(f) for f in self._flags]))

    def setPlaintext(self, f):
        self._flags[0] = bool(f)
        self._push_flags()

    def setEncrypted(self, f):
        self._flags[1] = bool(f)
        self._push_flags()

    def setVerify(self, f):
        self._flags[2] = bool(f)
        if f:  # src/circuit.cpp:833-840
            self._flags[0] = self._flags[1] = True
        self._push_flags()

    def getPlaintext(self):
        return self._flags[0]

    def getEncrypted(self):
        return self._flags[1]

    def getVerify(self):
        return self._flags[2]

    def Reset(self):
        self._flags = [False, False, False]  # src/circuit.cpp:378-381
        self._push_flags()
        self._ck(self.L.bfhe_circuit_reset(self.h))

    def set_wave_capacity(self, cap):
        """0 = the reference's ASAP waves; n > 0 = ready gates packed into waves of <= n bootstraps; -1 = one gate per SM and rank."""
        self._ck(self.L.bfhe_circuit_set_wave_capacity(self.h, cap))

    def set_sharding(self, rank, world, unique_id=None):
        self._ck(self.L.bfhe_circuit_set_sharding(self.h, rank, world, _ptr(unique_id)))
        self.world_size = world

    def exchange_mode(self):
        """0 = single rank, 1 = ncclAllGather per sharded level, 2 = fused into the key switch (stores into the peers' slabs)"""
        return self.L.bfhe_circuit_exchange_mode(self.h)

    def use_graph(self, on):
        self._ck(self.L.bfhe_circuit_use_graph(self.h, int(on)))

    def SetInput(self, inputs, verbose=False, seed=0):
        """inputs: list of bit lists, one per input bus (Inputs = vector<vector<unsigned>>, src/circuit.h:50)."""
        flat = np.ascontiguousarray(np.concatenate([np.asarray(i, dtype=np.uint8).ravel() for i in inputs]), dtype=np.uint8)
        self._ck(self.L.bfhe_circuit_set_input(self.h, _ptr(flat), flat.size, seed))

    def set_input_ct(self, cts):
        """SetInput on ciphertexts (bfhe_circuit_set_input_ct): needs the evaluation keys only.  cts: host numpy array (nbits, ct_stride)
        of uint32 (int32 accepted), or a device buffer (Slab, Slab.range(...), or __cuda_array_interface__ with that shape).  Sharded
        circuits: rank 0's rows are used; other ranks may pass None."""
        stride = self.ctx.stride
        if cts is None:
            self._ck(self.L.bfhe_circuit_set_input_ct(self.h, None, sum(self.info()["input_bits"]), 0))
        elif isinstance(cts, np.ndarray):
            if cts.ndim != 2 or cts.shape[1] != stride:
                raise ValueError("ciphertext array shape %s, expected (nbits, %d)" % (cts.shape, stride))
            if cts.dtype not in (np.uint32, np.int32):
                raise TypeError("ciphertext array dtype %s, expected uint32" % cts.dtype)
            a = np.ascontiguousarray(cts).view(np.uint32)
            self._ck(self.L.bfhe_circuit_set_input_ct(self.h, _ptr(a), a.shape[0], 0))
        else:
            ptr, rows = _device_rows(cts, stride)
            self._ck(self.L.bfhe_circuit_set_input_ct(self.h, ptr, rows, 1))

    def clock_ct(self, out=None):
        """Clock with the outputs left encrypted (bfhe_circuit_clock_ct): a numpy array (out_bits, ct_stride) of uint32, or, with `out`
        a device buffer as in set_input_ct with at least out_bits rows, the rows written there (and `out` returned)."""
        if out is None:
            host = np.zeros((self.info()["output_bits"], self.ctx.stride), dtype=np.uint32)
            self._ck(self.L.bfhe_circuit_clock_ct(self.h, _ptr(host), host.shape[0], 0))
            return host
        ptr, rows = _device_rows(out, self.ctx.stride)
        self._ck(self.L.bfhe_circuit_clock_ct(self.h, ptr, rows, 1))
        return out

    def Clock(self):
        """returns Outputs = [[bits of OUT:0]]; the plaintext pass result is kept in self.plain_out"""
        n = self.info()["output_bits"]
        out = np.zeros(n, dtype=np.uint8)
        pout = np.zeros(n, dtype=np.uint8)
        self._ck(self.L.bfhe_circuit_clock(self.h, _ptr(out), n, _ptr(pout)))
        self.plain_out = [pout.tolist()]
        if self._flags[1]:
            return [out.tolist()]
        return [pout.tolist()]

    def stats(self):
        d, h, m = C.c_double(), C.c_double(), C.c_uint64()
        self._ck(self.L.bfhe_circuit_stats(self.h, C.byref(d), C.byref(h), C.byref(m)))
        return dict(device_ms=d.value, host_ms=h.value, verify_mismatches=m.value)

    def level_plan(self, level, rank, world):
        cnt, first, rpr = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._ck(self.L.bfhe_circuit_level_plan(self.h, level, rank, world, None, 0, C.byref(cnt), C.byref(first), C.byref(rpr)))
        g = np.zeros(cnt.value, dtype=GATE_DTYPE)
        self._ck(self.L.bfhe_circuit_level_plan(self.h, level, rank, world, _ptr(g), g.size, C.byref(cnt), C.byref(first),
                                                C.byref(rpr)))
        return g, first.value, rpr.value

    def plan_misc(self, level=0):
        tot, fresh, nl, nc = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        outs = np.zeros(self.info()["output_bits"], dtype=np.uint32)
        self._ck(self.L.bfhe_circuit_plan_misc(self.h, C.byref(tot), C.byref(fresh), C.byref(nl), _ptr(outs), C.byref(nc), level, None))
        pairs = np.zeros((nc.value, 2), dtype=np.uint32)
        if nc.value:
            self._ck(self.L.bfhe_circuit_plan_misc(self.h, None, None, None, None, C.byref(nc), level, _ptr(pairs)))
        return dict(total_rows=tot.value, fresh_base=fresh.value, n_levels=nl.value, out_rows=outs, nots=pairs)

    def download_slab(self):
        rows = self.plan_misc()["total_rows"]
        out = np.zeros((rows, self.ctx.stride), dtype=np.uint32)
        self._ck(self.L.bfhe_circuit_download_slab(self.h, _ptr(out), rows))
        return out
