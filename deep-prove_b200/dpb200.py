"""ctypes view of the product: libdeepprove_b200.so (C ABI, include/deepprove_b200.h) and
libdeepprove_host.so (C++ host mirror of the reference crates).  Plumbing for tests/bench only --
a Rust host binds the same C ABI directly (INTEGRATION.md).  Never imports anything from oracle/.
Fails loudly when the CUDA library is missing: there is no CPU fallback.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdeepprove_b200.so")
HOST_LIB_PATH = os.path.join(_HERE, "libdeepprove_host.so")

P = 0xFFFFFFFF00000001
DP_OK, DP_ERR_INVALID, DP_ERR_CUDA, DP_ERR_NO_DEVICE, DP_ERR_STATE, DP_ERR_UNSUPPORTED = range(6)

# every symbol include/deepprove_b200.h declares (tests check the .so exports each one)
ABI_SYMBOLS = [
    "dp_init", "dp_shutdown", "dp_device_count", "dp_last_error", "dp_version", "dp_set_stream", "dp_synchronize",
    "dp_kernel_launches", "dp_set_wait_mode", "dp_get_wait_mode", "dp_profile_enable", "dp_profile_reset", "dp_profile_read", "dp_profile_read_ex", "dp_profile_flush",
    "dp_mle_upload", "dp_mle_wrap_device", "dp_mle_clone", "dp_mle_download", "dp_mle_info", "dp_mle_device_ptr",
    "dp_mle_free", "dp_mle_fix_high", "dp_mle_fix_high_new", "dp_mle_fix_low", "dp_mle_evaluate", "dp_mle_evaluate_many", "dp_eq_build",
    "dp_sc_create", "dp_sc_round", "dp_sc_finish", "dp_sc_destroy", "dp_sc_last_round_bytes", "dp_sc_current_mle", "dp_sc_set_resident_tail",
    "dp_poseidon2_init", "dp_set_merkle_hasher", "dp_get_merkle_hasher", "dp_pcs_commit", "dp_pcs_commit_many", "dp_pcs_batch_commit", "dp_pcs_comm_num_polys", "dp_pcs_comm_part", "dp_pcs_comm_info", "dp_pcs_comm_codeword", "dp_pcs_comm_bh_evals", "dp_pcs_comm_free",
    "dp_pcs_open_begin", "dp_pcs_open_round", "dp_pcs_open_final_message", "dp_pcs_open_query_words", "dp_pcs_open_query",
    "dp_pcs_open_free", "dp_pcs_commit_shard", "dp_pcs_comm_shard_info", "dp_pcs_comm_set_shard_roots", "dp_pcs_open_set_shard_roots",
    "dp_logup_build", "dp_logup_num_vars", "dp_logup_outputs", "dp_logup_layer_mles", "dp_logup_free", "dp_mle_linear_combination",
    "dp_wit_begin", "dp_wit_dense", "dp_wit_matmul", "dp_wit_requant", "dp_wit_relu", "dp_wit_pool", "dp_wit_finish", "dp_wit_free",
    "dp_fft_rows", "dp_pad_rows", "dp_conv_prod", "dp_conv_output_elements", "dp_phi_g_init", "dp_phi_level", "dp_mle_repeat",
]


# must be in the environment before CUDA initialises (see dp_init): 32 hardware work queues instead of 8
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")


class DpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("deepprove_b200 error %d: %s" % (code, msg))
        self.code = code


class ScProduct(C.Structure):
    _fields_ = [("coef", C.c_uint64 * 2), ("n_idx", C.c_uint32), ("idx", C.c_uint32 * 5)]


_lib = None
_host = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not built: run `make` (or __graft_entry__.build()); the CUDA extension is "
                              "mandatory, there is no CPU fallback" % LIB_PATH)
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _lib.dp_last_error.restype = C.c_char_p
        _lib.dp_version.restype = C.c_char_p
        _lib.dp_kernel_launches.restype = C.c_uint64
        _lib.dp_mle_device_ptr.restype = C.c_void_p
        _lib.dp_sc_last_round_bytes.restype = C.c_uint64
        _lib.dp_mle_device_ptr.argtypes = [C.c_void_p]
        _lib.dp_sc_last_round_bytes.argtypes = [C.c_void_p]
        _lib.dp_set_stream.argtypes = [C.c_void_p]
        _lib.dp_mle_upload.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]
        _lib.dp_mle_wrap_device.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]
        _lib.dp_mle_clone.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        _lib.dp_mle_download.argtypes = [C.c_void_p, C.c_void_p]
        _lib.dp_mle_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_uint32)]
        _lib.dp_mle_free.argtypes = [C.c_void_p]
        _lib.dp_mle_fix_high.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        _lib.dp_mle_fix_low.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        _lib.dp_mle_evaluate.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
        _lib.dp_eq_build.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
        _lib.dp_sc_create.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(ScProduct), C.c_uint32, C.c_uint32,
                                      C.c_uint32, C.POINTER(C.c_void_p)]
        _lib.dp_sc_round.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.dp_sc_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.dp_sc_destroy.argtypes = [C.c_void_p]
    return _lib


def host():
    global _host
    if _host is None:
        lib()
        if not os.path.exists(HOST_LIB_PATH):
            raise ImportError("%s not built: run `make`" % HOST_LIB_PATH)
        _host = C.CDLL(HOST_LIB_PATH)
        _host.dph_last_error.restype = C.c_char_p
        _host.dph_transcript_new.restype = C.c_void_p
        _host.dph_transcript_new.argtypes = [C.c_char_p]
        _host.dph_transcript_free.argtypes = [C.c_void_p]
        _host.dph_transcript_append_f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        _host.dph_transcript_append_msg.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
        _host.dph_transcript_append_e.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        _host.dph_transcript_challenge.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p]
        _host.dph_poseidon2_permute.argtypes = [C.c_void_p]
        _host.dph_sumcheck_prove_parallel.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(ScProduct), C.c_uint32,
                                                      C.c_uint32, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                      C.c_void_p, C.POINTER(C.c_uint32)]
    return _host


def check(rc):
    if rc != 0:
        raise DpError(rc, lib().dp_last_error().decode())


def hcheck(rc):
    if rc != 0:
        raise DpError(rc, host().dph_last_error().decode())


def init(device=0):
    check(lib().dp_init(int(device)))


def set_wait_mode(mode):
    """0 = every proving thread spins on its completion word (lowest latency); 1 = threads sleep and ONE poller thread of the
    library wakes them (many more proofs than CPUs in flight)"""
    check(lib().dp_set_wait_mode(int(mode)))


def device_count():
    return lib().dp_device_count()


def use_torch_stream():
    """Launch on torch's current CUDA stream so torch.cuda.Event brackets our kernels."""
    import torch
    check(lib().dp_set_stream(C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def _u64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.uint64))


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Mle:
    """Device-resident DenseMultilinearExtension (handle owner)."""

    def __init__(self, handle, keepalive=None):
        self.h = C.c_void_p(handle)
        self._keep = keepalive

    @staticmethod
    def upload(evals, is_ext):
        a = _u64(evals).reshape(-1)
        n = a.size // (2 if is_ext else 1)
        h = C.c_void_p()
        check(lib().dp_mle_upload(_ptr(a), n, int(bool(is_ext)), C.byref(h)))
        return Mle(h.value)

    @staticmethod
    def wrap_torch(t, is_ext):
        """Non-owning view of a torch int64/uint64 CUDA tensor holding canonical limbs."""
        n = t.numel() // (2 if is_ext else 1)
        h = C.c_void_p()
        check(lib().dp_mle_wrap_device(C.c_void_p(t.data_ptr()), n, int(bool(is_ext)), C.byref(h)))
        return Mle(h.value, keepalive=t)

    @staticmethod
    def eq(point):
        p = _u64(point).reshape(-1)
        h = C.c_void_p()
        check(lib().dp_eq_build(_ptr(p), p.size // 2, C.byref(h)))
        return Mle(h.value)

    def info(self):
        ln, ext, nv = C.c_uint64(), C.c_int(), C.c_uint32()
        check(lib().dp_mle_info(self.h, C.byref(ln), C.byref(ext), C.byref(nv)))
        return ln.value, bool(ext.value), nv.value

    def download(self):
        ln, ext, _ = self.info()
        out = np.empty(ln * (2 if ext else 1), dtype=np.uint64)
        check(lib().dp_mle_download(self.h, _ptr(out)))
        return out.reshape(-1, 2) if ext else out

    def fix_high(self, point):
        p = _u64(point).reshape(-1)
        check(lib().dp_mle_fix_high(self.h, _ptr(p), p.size // 2))
        return self

    def fix_low(self, point):
        p = _u64(point).reshape(-1)
        h = C.c_void_p()
        check(lib().dp_mle_fix_low(self.h, _ptr(p), p.size // 2, C.byref(h)))
        return Mle(h.value)

    def evaluate(self, point):
        p = _u64(point).reshape(-1)
        out = np.zeros(2, dtype=np.uint64)
        check(lib().dp_mle_evaluate(self.h, _ptr(p), p.size // 2, _ptr(out)))
        return out

    def clone(self):
        h = C.c_void_p()
        check(lib().dp_mle_clone(self.h, C.byref(h)))
        return Mle(h.value)

    def free(self):
        if self.h:
            lib().dp_mle_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Witness:
    """dp_wit_*: quantised inference ops and lookup-witness columns on the device (one object per proof)."""

    def __init__(self, tables):
        """tables: list of (kind, size) -- kind 0 Relu, 2 Range, 3 Clamping(size)"""
        self.n = len(tables)
        k = (C.c_uint32 * self.n)(*[int(t[0]) for t in tables]); z = (C.c_uint32 * self.n)(*[int(t[1]) for t in tables])
        self.h = C.c_void_p()
        check(lib().dp_wit_begin(self.n, k, z, C.byref(self.h)))

    @staticmethod
    def dense(w, bias, x, nrows, ncols):
        h = C.c_void_p()
        check(lib().dp_wit_dense(w.h, bias.h, x.h, int(nrows), int(ncols), C.byref(h)))
        return Mle(h.value)

    def requant(self, x, shift, fpm, intermediate_bits, clamp_table, range_table):
        nc = 2 + shift // 8
        cols = (C.c_void_p * nc)()
        check(lib().dp_wit_requant(self.h, x.h, int(shift), C.c_int64(int(fpm)), int(intermediate_bits), int(clamp_table), int(range_table), cols, nc))
        return [Mle(c) for c in cols]

    def relu(self, x, relu_table):
        h = C.c_void_p()
        check(lib().dp_wit_relu(self.h, x.h, int(relu_table), C.byref(h)))
        return Mle(h.value)

    def pool(self, x, c, hh, w, range_table):
        cols = (C.c_void_p * 5)()
        check(lib().dp_wit_pool(self.h, x.h, int(c), int(hh), int(w), int(range_table), cols))
        return [Mle(v) for v in cols]

    def finish(self):
        mu = (C.c_void_p * self.n)(); bits = C.c_uint32()
        check(lib().dp_wit_finish(self.h, mu, C.byref(bits)))
        return [Mle(v) for v in mu], bits.value

    def free(self):
        if self.h:
            lib().dp_wit_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def set_hasher(kind):
    """0 = PoseidonHasher + BasicTranscript (default), 1 = BlakeHasher + BlakeTranscript (the reference's `blake` feature); process-wide"""
    hcheck(host().dph_set_hasher(int(kind)))


def profile_enable(on=True):
    check(lib().dp_profile_enable(int(on)))


def profile_reset():
    check(lib().dp_profile_reset())


def profile_read(cap=96, with_units=False):
    """-> {kernel name: (launches, total_ms, algorithmic_bytes[, units])}; process-wide (all proving threads)"""
    names = ((C.c_char * 64) * cap)()
    counts = (C.c_uint64 * cap)()
    ms = (C.c_double * cap)()
    by = (C.c_uint64 * cap)()
    un = (C.c_uint64 * cap)()
    n = lib().dp_profile_read_ex(names, counts, ms, by, un, cap)
    if with_units:
        return {names[i].value.decode(): (counts[i], ms[i], by[i], un[i]) for i in range(min(n, cap))}
    return {names[i].value.decode(): (counts[i], ms[i], by[i]) for i in range(min(n, cap))}


def make_products(products):
    """products: list of (coef (c0,c1), [mle indices])"""
    arr = (ScProduct * len(products))()
    for i, (coef, idx) in enumerate(products):
        arr[i].coef[0], arr[i].coef[1] = int(coef[0]), int(coef[1])
        arr[i].n_idx = len(idx)
        for j, v in enumerate(idx[:5]):
            arr[i].idx[j] = int(v)
    return arr


class Sumcheck:
    """Round-granular device sumcheck prover (dp_sc_*)."""

    def __init__(self, mles, products, max_nv, max_deg):
        self.mles = list(mles)
        hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
        self.prods = make_products(products)
        self.max_deg = max_deg
        self.h = C.c_void_p()
        check(lib().dp_sc_create(hs, len(mles), self.prods, len(products), max_nv, max_deg, C.byref(self.h)))

    def round(self, challenge=None):
        out = np.zeros(2 * (self.max_deg + 1), dtype=np.uint64)
        c = None if challenge is None else _u64(challenge)
        check(lib().dp_sc_round(self.h, None if c is None else _ptr(c), _ptr(out)))
        return out.reshape(-1, 2)

    def finish(self, challenge):
        out = np.zeros(2 * len(self.mles), dtype=np.uint64)
        c = _u64(challenge)
        check(lib().dp_sc_finish(self.h, _ptr(c), _ptr(out)))
        return out.reshape(-1, 2)

    def last_round_bytes(self):
        return lib().dp_sc_last_round_bytes(self.h)

    def destroy(self):
        if self.h:
            lib().dp_sc_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def sumcheck_prove_parallel(mles, products, max_nv, label=b"m2vec"):
    """IOPProverState::prove_parallel through the C++ host mirror (host Poseidon2 Fiat-Shamir).
    Returns (point[nv,2], msgs[nv,deg+1,2], final_evals[n_mles,2])."""
    hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
    prods = make_products(products)
    max_deg = max(len(p[1]) for p in products)
    point = np.zeros((max_nv, 2), dtype=np.uint64)
    msgs = np.zeros((max_nv, max_deg + 1, 2), dtype=np.uint64)
    fin = np.zeros((len(mles), 2), dtype=np.uint64)
    deg = C.c_uint32()
    hcheck(host().dph_sumcheck_prove_parallel(hs, len(mles), prods, len(products), max_nv, label, None, _ptr(point),
                                              _ptr(msgs), _ptr(fin), C.byref(deg)))
    return point, msgs, fin


# ---- mpcs (Basefold) -------------------------------------------------------------------------------
def _pcs_setup():
    L = lib()
    if getattr(L, "_pcs_ready", False):
        return L
    L.dp_pcs_commit.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    L.dp_pcs_comm_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
    L.dp_pcs_comm_codeword.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.dp_pcs_comm_bh_evals.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
    L.dp_pcs_comm_free.argtypes = [C.c_void_p]
    L.dp_pcs_open_begin.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p), C.c_void_p]
    L.dp_pcs_open_round.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
    L.dp_pcs_open_final_message.argtypes = [C.c_void_p, C.c_void_p]
    L.dp_pcs_open_query_words.argtypes = [C.c_void_p]
    L.dp_pcs_open_query_words.restype = C.c_uint64
    L.dp_pcs_open_query.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]
    L.dp_pcs_open_free.argtypes = [C.c_void_p]
    L.dp_poseidon2_init.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    H = host()
    H.dph_pcs_open.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p]
    H.dph_pcs_batch_open.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64,
                                     C.POINTER(C.c_uint64)]
    L._pcs_ready = True
    return L


class Commitment:
    """BasefoldCommitmentWithWitness on device (dp_pcs_comm)."""

    def __init__(self, mle, full_log):
        L = _pcs_setup()
        self.h = C.c_void_p()
        check(L.dp_pcs_commit(mle.h, full_log, C.byref(self.h)))
        nv, b, t = C.c_uint32(), C.c_int(), C.c_int()
        self.root = np.zeros(4, dtype=np.uint64)
        check(L.dp_pcs_comm_info(self.h, C.byref(nv), C.byref(b), C.byref(t), _ptr(self.root)))
        self.num_vars, self.is_base, self.trivial = nv.value, bool(b.value), bool(t.value)

    def codeword(self):
        v = C.c_void_p()
        check(lib().dp_pcs_comm_codeword(self.h, C.byref(v)))
        return Mle(v.value).download()

    def bh_evals(self):
        v = C.c_void_p()
        check(lib().dp_pcs_comm_bh_evals(self.h, C.byref(v)))
        return Mle(v.value).download()

    def free(self):
        if self.h:
            lib().dp_pcs_comm_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pcs_open(mle, full_log, point, label=b"m2vec", cap=1 << 24):
    """Basefold::commit + Basefold::open through the C++ host mirror; returns (root, flat proof)."""
    _pcs_setup()
    p = _u64(point).reshape(-1)
    out = np.zeros(cap, dtype=np.uint64)
    n = C.c_uint64()
    root = np.zeros(4, dtype=np.uint64)
    hcheck(host().dph_pcs_open(mle.h, full_log, _ptr(p), label, _ptr(out), cap, C.byref(n), _ptr(root)))
    return root, out[: n.value].copy()


def pcs_batch_open(mles, full_log, points, label=b"m2vec", cap=1 << 25):
    """commit each polynomial, then Basefold::batch_open with Evaluation::new(i, i, poly_i(point_i))."""
    _pcs_setup()
    hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
    p = np.concatenate([_u64(x).reshape(-1) for x in points])
    out = np.zeros(cap, dtype=np.uint64)
    n = C.c_uint64()
    hcheck(host().dph_pcs_batch_open(hs, len(mles), full_log, _ptr(p), label, _ptr(out), cap, C.byref(n)))
    return out[: n.value].copy()


def pcs_batch_open_evals(mles, full_log, points, eval_poly, eval_point, label=b"m2vec", cap=1 << 25):
    """commit each polynomial, then Basefold::batch_open with an explicit evaluation list (several polynomials may share a point)"""
    _pcs_setup()
    H = host()
    H.dph_pcs_batch_open_evals.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_char_p,
                                           C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
    p = np.concatenate([_u64(x).reshape(-1) for x in points])
    pnv = np.ascontiguousarray([_u64(x).reshape(-1, 2).shape[0] for x in points], dtype=np.uint32)
    ep = np.ascontiguousarray(eval_poly, dtype=np.uint32); eq = np.ascontiguousarray(eval_point, dtype=np.uint32)
    out = np.zeros(cap, dtype=np.uint64)
    n = C.c_uint64()
    hcheck(H.dph_pcs_batch_open_evals(hs, len(mles), full_log, p.ctypes.data, pnv.ctypes.data, len(pnv), ep.ctypes.data, eq.ctypes.data, len(ep), label, out.ctypes.data, cap, C.byref(n)))
    return out[: n.value].copy()


def pcs_simple_batch(mles, full_log, point=None, evals=None, label=b"m2vec", cap=1 << 24):
    """Basefold::batch_commit of same-size device MLEs (+ simple_batch_open at `point` with the claimed `evals`): (root, flat | None)"""
    _pcs_setup()
    H = host()
    H.dph_pcs_simple_batch.argtypes = [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
    root = np.zeros(4, dtype=np.uint64)
    n = C.c_uint64()
    if point is None:
        hcheck(H.dph_pcs_simple_batch(hs, len(mles), full_log, None, 0, None, label, root.ctypes.data, None, 0, C.byref(n)))
        return root, None
    pt = _u64(point).reshape(-1); ev = _u64(evals).reshape(-1)
    out = np.zeros(cap, dtype=np.uint64)
    hcheck(H.dph_pcs_simple_batch(hs, len(mles), full_log, pt.ctypes.data, pt.size // 2, ev.ctypes.data, label, root.ctypes.data, out.ctypes.data, cap, C.byref(n)))
    return root, out[: n.value].copy()


# ---- zkml MLP prover (host mirror of zkml::{Context, Prover}) -----------------------------------------
class ZkmlContext:
    """Context::generate for n_layers x [Dense(width x width)+bias -> Requant -> ReLU]: weights, bias and lookup
    tables uploaded once and committed (setup).  rq: (n_layers, 4) int64 = right_shift, fp_scale,
    fixed_point_multiplier, intermediate_bit_size."""

    def __init__(self, n_layers, width, weights, bias, rq):
        _pcs_setup()
        H = host()
        H.dph_zkml_context_new.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        H.dph_zkml_context_free.argtypes = [C.c_void_p]
        H.dph_zkml_prove.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        self.n_layers, self.width = n_layers, width
        w = np.ascontiguousarray(weights, dtype=np.int64)
        b = np.ascontiguousarray(bias, dtype=np.int64)
        r = np.ascontiguousarray(rq, dtype=np.int64)
        self.h = C.c_void_p()
        hcheck(H.dph_zkml_context_new(n_layers, width, _ptr(w), _ptr(b), _ptr(r), C.byref(self.h)))
        self._out = np.zeros(1 << 22, dtype=np.uint64)

    def prove(self, x, label=b"m2vec"):
        """inference + Prover::prove + flat proof, from a host input vector (end to end)"""
        x = np.ascontiguousarray(x, dtype=np.int64)
        n = C.c_uint64()
        hcheck(host().dph_zkml_prove(self.h, _ptr(x), 0, label, _ptr(self._out), self._out.size, C.byref(n)))
        return self._out[: n.value].copy()

    def run_inference(self, x):
        x = np.ascontiguousarray(x, dtype=np.int64)
        hcheck(host().dph_zkml_prove(self.h, _ptr(x), 1, b"", None, 0, None))

    def prove_trace(self, label=b"m2vec", want_proof=False):
        """Prover::prove on the stored inference trace (what zkml/src/bin/bench.rs:390-408 times)"""
        n = C.c_uint64()
        hcheck(host().dph_zkml_prove(self.h, None, 2, label, _ptr(self._out) if want_proof else None, self._out.size, C.byref(n)))
        return self._out[: n.value].copy() if want_proof else None

    def prove_concurrent(self, n_workers, n_proofs, device=0, e2e=False, label=b"m2vec"):
        """n_workers persistent host threads (own stream + device arena each) prove until n_proofs are done; returns wall
        seconds.  e2e=False: Prover::prove on the stored trace; e2e=True: inference + prove + serialised proof per job."""
        H = host()
        H.dph_zkml_prove_concurrent.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_char_p, C.POINTER(C.c_double)]
        sec = C.c_double()
        hcheck(H.dph_zkml_prove_concurrent(self.h, int(device), int(n_workers), int(n_proofs), int(bool(e2e)), label, C.byref(sec)))
        return sec.value

    def last_concurrent_proof(self):
        """flat proof (as prove() returns it) of the job claimed last in the most recent prove_concurrent call"""
        H = host()
        H.dph_zkml_last_concurrent_proof.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        n = C.c_uint64()
        hcheck(H.dph_zkml_last_concurrent_proof(self.h, _ptr(self._out), self._out.size, C.byref(n)))
        return self._out[: n.value].copy()

    def free(self):
        if self.h:
            host().dph_zkml_context_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ModelContext(ZkmlContext):
    """Context::generate for a general layer list (Dense / Requant / ReLU / Convolution / Maxpool2D), see
    dph_model_context_new: desc (n_nodes, 9) int64, data = weights in node order, input_len = padded input length."""

    def __init__(self, desc, data, input_len):
        _pcs_setup()
        H = host()
        H.dph_model_context_new.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]
        H.dph_zkml_context_free.argtypes = [C.c_void_p]
        H.dph_zkml_prove.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        d = np.ascontiguousarray(desc, dtype=np.int64).reshape(-1, 9)
        w = np.ascontiguousarray(data, dtype=np.int64)
        self.h = C.c_void_p()
        hcheck(H.dph_model_context_new(_ptr(d), d.shape[0], _ptr(w), int(input_len), C.byref(self.h)))
        self._out = np.zeros(1 << 23, dtype=np.uint64)


def sumcheck_prove_batch_polys(T, mles, products, max_nv, label=b"m2vec"):
    """IOPProverState::prove_batch_polys (devirgo split into T contiguous slices) through the C++ host mirror."""
    H = host()
    H.dph_sumcheck_prove_batch_polys.argtypes = [C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(ScProduct), C.c_uint32, C.c_uint32,
                                                 C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p]
    hs = (C.c_void_p * len(mles))(*[m.h for m in mles])
    prods = make_products(products)
    max_deg = max(len(p[1]) for p in products)
    point = np.zeros((max_nv, 2), dtype=np.uint64)
    msgs = np.zeros((max_nv, max_deg + 1, 2), dtype=np.uint64)
    fin = np.zeros((len(mles), 2), dtype=np.uint64)
    hcheck(H.dph_sumcheck_prove_batch_polys(T, hs, len(mles), prods, len(products), max_nv, label, _ptr(point), _ptr(msgs), _ptr(fin)))
    return point, msgs, fin


# ---- FFT-convolution layer (host/conv.hpp) -------------------------------------------------------------
def conv_prove(filt, bias, unpadded_out, x, label=b"m2vec", cap=1 << 20, prove=True):
    """Convolution::op (+ prove_convolution_step when `prove`) on a padded layer: filt [kw, kx, real_nw, real_nw],
    bias [kw], x [kx, n_x, n_x] (int64).  Returns (after_bias, cleared, flat_proof | None)."""
    H = host()
    filt = np.ascontiguousarray(filt, dtype=np.int64); bias = np.ascontiguousarray(bias, dtype=np.int64); x = np.ascontiguousarray(x, dtype=np.int64)
    kw, kx, rn, _ = filt.shape
    n_x = x.shape[1]
    uo = np.ascontiguousarray(unpadded_out, dtype=np.uint32)
    after = np.zeros((kw, n_x, n_x), dtype=np.int64)
    cleared = np.zeros((kw, n_x, n_x), dtype=np.int64)
    out = np.zeros(cap if prove else 1, dtype=np.uint64)
    n = C.c_uint64()
    H.dph_conv_prove.argtypes = [C.c_uint32] * 4 + [C.c_void_p] * 4 + [C.c_char_p] + [C.c_void_p] * 3 + [C.c_uint64, C.c_void_p]
    hcheck(H.dph_conv_prove(kw, kx, n_x, rn, filt.ctypes.data, bias.ctypes.data, uo.ctypes.data, x.ctypes.data, label, after.ctypes.data, cleared.ctypes.data,
                            out.ctypes.data if prove else None, cap, C.addressof(n) if prove else None))
    return after, cleared, (out[:n.value].copy() if prove else None)
