"""scroll-prover_b200 — B200-native Halo2/KZG polynomial-arithmetic backend (host-side Python driver).

This package is the pytest/bench driver over the C ABI in include/b200zk.h (libb200zk.so, hand-written
sm_100a CUDA).  It mirrors the names and argument meaning of the halo2_proofs functions the library
replaces (scroll-tech/halo2 @ e5ddf67, pin /root/reference/Cargo.lock:1886-1888):

    best_multiexp(coeffs, bases)            halo2_proofs::arithmetic::best_multiexp
    best_fft(a, omega, log_n)               halo2_proofs::arithmetic::best_fft
    EvaluationDomain(j, k)                  halo2_proofs::poly::EvaluationDomain::new
        .lagrange_to_coeff / .coeff_to_extended / .extended_to_coeff
    ParamsKZG(g, g_lagrange)                halo2_proofs::poly::kzg::commitment::ParamsKZG
        .commit / .commit_lagrange
    eval_polynomial / kate_division / batch_invert

Field elements are numpy uint64 arrays (n, 4) of raw Montgomery limbs (memcpy-compatible with
halo2curves Fr); affine points (n, 8); a G1 result is a (12,) normalised Jacobian (x, y, 1).
torch CUDA tensors (uint8/int64 storage) can be passed wherever an array is accepted: their
device pointer is handed to the library unchanged.

There is NO CPU fallback and this package never imports oracle/: if libb200zk.so is missing or
no CUDA device is present, constructing a Context raises.

(The directory name contains a hyphen, as the task layout requires; import it with
 importlib.import_module("scroll-prover_b200") — tests/conftest.py and bench.py do that.)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200zk.so")

R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
_R_MONT = 1 << 256
FR_S = 28
_ROOT_OF_UNITY = pow(7, (R_MOD - 1) >> FR_S, R_MOD)
_ZETA = pow(7, 2 * (R_MOD - 1) // 3, R_MOD)

OK, E_INVALID, E_CUDA, E_OOM, E_UNSUPPORTED = 0, -1, -2, -3, -4
SRS_G, SRS_G_LAGRANGE = 0, 1
COSET_NONE, COSET_PRE, COSET_POST = 0, 1, 2


class B200zkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200zk error {code}: {msg}")
        self.code = code


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not built; run `python scroll-prover_b200/build.py` (needs nvcc). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
    sig = {
        "b200zk_ctx_create": [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)],
        "b200zk_ctx_destroy": [vp],
        "b200zk_ctx_set_stream": [vp, vp],
        "b200zk_ctx_synchronize": [vp],
        "b200zk_ctx_launch_count": [vp, C.POINTER(u64)],
        "b200zk_buf_alloc": [vp, u64, C.POINTER(vp)],
        "b200zk_buf_free": [vp, vp],
        "b200zk_buf_upload": [vp, vp, vp, u64],
        "b200zk_buf_download": [vp, vp, vp, u64],
        "b200zk_srs_register": [vp, vp, u64, u32, C.POINTER(vp)],
        "b200zk_srs_release": [vp, vp],
        "b200zk_srs_set_precompute": [vp, C.c_int],
        "b200zk_srs_len": [vp, C.POINTER(u64)],
        "b200zk_msm_g1": [vp, vp, vp, u64, vp],
        "b200zk_msm_g1_bases": [vp, vp, vp, u64, vp],
        "b200zk_msm_g1_batch": [vp, vp, C.POINTER(vp), u32, u64, vp],
        "b200zk_msm_g1_range": [vp, vp, vp, u64, u64, vp],
        "b200zk_msm_g1_sharded": [vp, vp, vp, u64, vp],
        "b200zk_comm_unique_id": [vp],
        "b200zk_ctx_comm_init": [vp, vp, C.c_int, C.c_int],
        "b200zk_ctx_comm_info": [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)],
        "b200zk_shard_range": [u64, C.c_int, C.c_int, C.POINTER(u64), C.POINTER(u64)],
        "b200zk_g1_sum": [vp, vp, u64, vp],
        "b200zk_g1_generator_mul_batch": [vp, vp, u64, vp],
        "b200zk_fft_g1": [vp, vp, u32, vp],
        "b200zk_g_to_lagrange": [vp, vp, u32, vp],
        "b200zk_ntt_fr": [vp, vp, u32, vp, C.c_int, C.c_int],
        "b200zk_ntt_fr_ext": [vp, vp, u32, vp, u32, vp, C.c_int, C.c_int],
        "b200zk_ctx_set_overlap": [vp, C.c_int],
        "b200zk_run_column_jobs": [vp, vp, u32, u32, vp, vp, vp, u32, vp],
        "b200zk_commit_columns": [vp, vp, C.POINTER(vp), u32, u32, vp, vp, u32, vp, C.POINTER(vp), C.POINTER(vp), C.c_int],
        "b200zk_poly_add": [vp, vp, vp, vp, u64],
        "b200zk_poly_sub": [vp, vp, vp, vp, u64],
        "b200zk_poly_mul": [vp, vp, vp, vp, u64],
        "b200zk_poly_scale": [vp, vp, vp, vp, u64],
        "b200zk_poly_axpy": [vp, vp, vp, vp, vp, u64],
        "b200zk_eval_poly": [vp, vp, u64, vp, vp],
        "b200zk_inner_product": [vp, vp, vp, u64, vp],
        "b200zk_batch_invert": [vp, vp, u64],
        "b200zk_kate_division": [vp, vp, vp, u64, vp],
        "b200zk_prefix_scan": [vp, C.c_int, vp, u64, vp, vp],
        "b200zk_poly_lincomb": [vp, vp, C.POINTER(vp), vp, u32, u64],
        "b200zk_permutation_product": [vp, C.POINTER(vp), C.POINTER(vp), u32, vp, vp, vp, vp, vp, u32, vp, vp],
        "b200zk_logup_running_sum": [vp, C.POINTER(vp), u32, vp, vp, vp, u32, vp, vp],
        "b200zk_graph_create": [vp, vp, u32, vp, u32, vp, u32, vp, u32, C.POINTER(vp)],
        "b200zk_graph_check": [vp, u32, vp, u32, u32, u32, C.POINTER(u32), C.POINTER(u32), C.c_char_p, u64],
        "b200zk_graph_destroy": [vp, vp],
        "b200zk_graph_info": [vp, C.POINTER(u32), C.POINTER(u32)],
        "b200zk_graph_evaluate": [vp, vp, C.POINTER(vp), u32, C.POINTER(vp), u32, C.POINTER(vp), u32, vp, u32, vp, vp, vp, vp, vp,
                                  vp, u32, i32],
        "b200zk_graph_evaluate_rows": [vp, vp, C.POINTER(vp), u32, C.POINTER(vp), u32, C.POINTER(vp), u32, vp, u32, vp, vp, vp, vp, vp,
                                       vp, u32, i32, u64, u64],
        "b200zk_allgather_rows": [vp, vp, u32],
        "b200zk_coeff_to_extended_parts": [vp, C.POINTER(vp), u32, u32, u32, u32, C.POINTER(vp)],
        "b200zk_graph_evaluate_part": [vp, vp, C.POINTER(vp), u32, C.POINTER(vp), u32, C.POINTER(vp), u32, vp, u32, vp, vp, vp, vp, u32,
                                       u32, u32, vp],
        "b200zk_extended_parts_to_coeff": [vp, vp, u32, u32, u32, C.c_int, vp],
        "b200zk_debug_field_op": [vp, C.c_int, C.c_int, vp, vp, vp, u64],
        "b200zk_profile_enable": [vp, C.c_int],
        "b200zk_profile_reset": [vp],
        "b200zk_profile_read": [vp, C.c_char_p, C.POINTER(C.c_double), C.POINTER(u64)],
        "b200zk_msm_set_window": [vp, u32],
        "b200zk_msm_last_stats": [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u64)],
        "b200zk_msm_total_adds": [vp, C.POINTER(u64), C.c_int],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = i32
    lib.b200zk_last_error.argtypes = [vp]
    lib.b200zk_last_error.restype = C.c_char_p
    return lib


ABI_SYMBOLS = [
    "b200zk_ctx_create", "b200zk_ctx_destroy", "b200zk_last_error", "b200zk_ctx_set_stream", "b200zk_ctx_synchronize",
    "b200zk_ctx_launch_count", "b200zk_buf_alloc", "b200zk_buf_free", "b200zk_buf_upload", "b200zk_buf_download",
    "b200zk_srs_register", "b200zk_srs_set_precompute", "b200zk_srs_release", "b200zk_srs_len", "b200zk_msm_g1", "b200zk_msm_g1_bases", "b200zk_msm_g1_batch", "b200zk_msm_g1_range", "b200zk_msm_g1_sharded",
    "b200zk_comm_unique_id", "b200zk_ctx_comm_init", "b200zk_ctx_comm_info", "b200zk_shard_range", "b200zk_g1_sum",
    "b200zk_g1_generator_mul_batch", "b200zk_fft_g1", "b200zk_g_to_lagrange", "b200zk_ntt_fr", "b200zk_ntt_fr_ext", "b200zk_ctx_set_overlap", "b200zk_run_column_jobs", "b200zk_commit_columns", "b200zk_poly_add", "b200zk_poly_sub",
    "b200zk_poly_mul", "b200zk_poly_scale", "b200zk_poly_axpy", "b200zk_eval_poly", "b200zk_inner_product", "b200zk_batch_invert",
    "b200zk_kate_division", "b200zk_prefix_scan", "b200zk_poly_lincomb", "b200zk_permutation_product", "b200zk_logup_running_sum", "b200zk_graph_create", "b200zk_graph_check",
    "b200zk_graph_destroy", "b200zk_graph_info", "b200zk_graph_evaluate", "b200zk_graph_evaluate_rows", "b200zk_allgather_rows", "b200zk_coeff_to_extended_parts", "b200zk_graph_evaluate_part", "b200zk_extended_parts_to_coeff", "b200zk_debug_field_op", "b200zk_profile_enable", "b200zk_profile_reset", "b200zk_profile_read", "b200zk_msm_set_window", "b200zk_msm_last_stats", "b200zk_msm_total_adds",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = _load()
    return _lib


# ---------------------------------------------------------------- pointer helpers
def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _ptr(x):
    """(void*, keepalive) of a numpy array or a torch tensor (host or CUDA)."""
    if x is None:
        return None, None
    if _is_torch(x):
        assert x.is_contiguous()
        return C.c_void_p(x.data_ptr()), x
    a = np.ascontiguousarray(x)
    return C.c_void_p(a.ctypes.data), a


def fr_from_int(v: int) -> np.ndarray:
    v = (v % R_MOD) * _R_MONT % R_MOD
    return np.array([(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(4)], dtype=np.uint64)


def fr_to_int(a) -> int:
    a = np.asarray(a, dtype=np.uint64).reshape(-1)
    return sum(int(x) << (64 * i) for i, x in enumerate(a)) * pow(_R_MONT, -1, R_MOD) % R_MOD


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = lib().b200zk_comm_unique_id(buf)
    if rc != OK:
        raise B200zkError(rc, "b200zk_comm_unique_id failed (NCCL not loadable?)")
    return buf.raw


def shard_range(n: int, rank: int, world: int):
    first, cnt = C.c_uint64(), C.c_uint64()
    rc = lib().b200zk_shard_range(n, rank, world, C.byref(first), C.byref(cnt))
    if rc != OK:
        raise B200zkError(rc, "b200zk_shard_range: bad arguments")
    return first.value, cnt.value


class Context:
    """One per process per GPU (b200zk_ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        devs = (C.c_int * 1)(device)
        rc = lib().b200zk_ctx_create(devs, 1, C.byref(self._h))
        if rc != OK:
            raise B200zkError(rc, "b200zk_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self.device = device

    def close(self):
        if self._h:
            lib().b200zk_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc: int):
        if rc != OK:
            raise B200zkError(rc, lib().b200zk_last_error(self._h).decode())

    def set_stream(self, cuda_stream: int | None):
        self._ck(lib().b200zk_ctx_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def synchronize(self):
        self._ck(lib().b200zk_ctx_synchronize(self._h))

    def buf_upload(self, dev, host):
        """b200zk_buf_upload: host array / pinned tensor -> device tensor (H2D on the context stream, synchronous)."""
        nbytes = _count(host, 1)
        assert _count(dev, 1) >= nbytes
        pd, k1 = _ptr(dev)
        ph, k2 = _ptr(host)
        self._ck(lib().b200zk_buf_upload(self._h, pd, ph, nbytes))

    # ---- multi-GPU: the context owns its NCCL communicator
    def comm_init(self, unique_id: bytes | None, rank: int, world: int):
        buf = C.create_string_buffer(unique_id, 128) if unique_id is not None else None
        self._ck(lib().b200zk_ctx_comm_init(self._h, buf, rank, world))

    def comm_init_torch(self, dist):
        """Joins this context into a communicator spanning an initialised torch.distributed job: rank 0 draws the
        NCCL unique id, torch broadcasts its 128 bytes (the bootstrap channel), every rank calls b200zk_ctx_comm_init."""
        import torch

        rank, world = dist.get_rank(), dist.get_world_size()
        if world == 1:
            return self.comm_init(None, 0, 1)
        backend = dist.get_backend()
        dev = torch.device("cuda", self.device) if backend == "nccl" else torch.device("cpu")
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            t = torch.frombuffer(bytearray(comm_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(t, 0)
        self.comm_init(bytes(t.cpu().numpy().tobytes()), rank, world)

    def allgather_rows(self, values, log_size: int):
        """b200zk_allgather_rows: collective; every rank contributes its shard_range slice of `values` (a CUDA tensor)."""
        assert _count(values, 32) == 1 << log_size
        pv, kv = _ptr(values)
        self._ck(lib().b200zk_allgather_rows(self._h, pv, log_size))
        return values

    def comm_info(self):
        r, w = C.c_int(), C.c_int()
        self._ck(lib().b200zk_ctx_comm_info(self._h, C.byref(r), C.byref(w)))
        return r.value, w.value

    def set_overlap(self, on: bool):
        self._ck(lib().b200zk_ctx_set_overlap(self._h, int(on)))

    def launch_count(self) -> int:
        v = C.c_uint64()
        self._ck(lib().b200zk_ctx_launch_count(self._h, C.byref(v)))
        return v.value

    PROFILE_CLASSES = ("ntt_pass", "ntt_table", "msm_count", "msm_scan", "msm_scatter", "msm_accumulate", "msm_combine",
                       "msm_reduce", "msm_finish", "poly")

    def profile_enable(self, on: bool = True):
        self._ck(lib().b200zk_profile_enable(self._h, int(on)))

    def profile_reset(self):
        self._ck(lib().b200zk_profile_reset(self._h))

    def profile_read(self) -> dict:
        out = {}
        for name in self.PROFILE_CLASSES:
            ms, cnt = C.c_double(), C.c_uint64()
            self._ck(lib().b200zk_profile_read(self._h, name.encode(), C.byref(ms), C.byref(cnt)))
            out[name] = {"ms": ms.value, "count": cnt.value}
        return out

    # ---- SRS / MSM
    def srs_register(self, bases, tag: int = SRS_G) -> "Srs":
        return Srs(self, bases, tag)

    def srs_set_precompute(self, on: bool):
        self._ck(lib().b200zk_srs_set_precompute(self._h, int(on)))

    def msm_set_window(self, c: int):
        self._ck(lib().b200zk_msm_set_window(self._h, c))

    def msm_last_stats(self):
        c, w, a = C.c_uint32(), C.c_uint32(), C.c_uint64()
        self._ck(lib().b200zk_msm_last_stats(self._h, C.byref(c), C.byref(w), C.byref(a)))
        return {"window_bits": c.value, "n_windows": w.value, "n_bucket_adds": a.value}

    def msm_total_adds(self, reset: bool = False) -> int:
        v = C.c_uint64()
        self._ck(lib().b200zk_msm_total_adds(self._h, C.byref(v), int(reset)))
        return v.value

    def best_multiexp(self, coeffs, bases) -> np.ndarray:
        """arithmetic::best_multiexp(coeffs, bases): panics (AssertionError) if lengths differ."""
        n = _count(coeffs, 32)
        assert n == _count(bases, 64), "assert_eq!(coeffs.len(), bases.len())"
        out = np.zeros(12, np.uint64)
        pc, k1 = _ptr(coeffs)
        pb, k2 = _ptr(bases)
        self._ck(lib().b200zk_msm_g1_bases(self._h, pb, pc, n, out.ctypes.data))
        return out

    def g1_sum(self, jac_points) -> np.ndarray:
        cnt = _count(jac_points, 96)
        out = np.zeros(12, np.uint64)
        p, k = _ptr(jac_points)
        self._ck(lib().b200zk_g1_sum(self._h, p, cnt, out.ctypes.data))
        return out

    def g1_generator_mul_batch(self, scalars, out=None):
        n = _count(scalars, 32)
        if out is None:
            out = np.zeros((n, 8), np.uint64)
        ps, k1 = _ptr(scalars)
        po, k2 = _ptr(out)
        self._ck(lib().b200zk_g1_generator_mul_batch(self._h, ps, n, po))
        return out

    def best_fft_g1(self, jac_points, omega, log_n: int):
        """arithmetic::best_fft::<Fr, G1> in place on (2^log_n, 12) Jacobian points."""
        assert _count(jac_points, 96) == 1 << log_n
        pa, k1 = _ptr(jac_points)
        po, k2 = _ptr(omega)
        self._ck(lib().b200zk_fft_g1(self._h, pa, log_n, po))
        if not _is_torch(jac_points) and k1 is not jac_points:
            jac_points[...] = k1.reshape(np.asarray(jac_points).shape)
        return jac_points

    def g_to_lagrange(self, g, k: int, out=None):
        """poly::kzg::commitment::g_to_lagrange (Params::downsize): affine (2^k, 8) -> affine (2^k, 8)."""
        assert _count(g, 64) == 1 << k
        if out is None:
            out = _like(g)
        pg, k1 = _ptr(g)
        po, k2 = _ptr(out)
        self._ck(lib().b200zk_g_to_lagrange(self._h, pg, k, po))
        return out

    # ---- NTT
    def best_fft(self, a, omega, log_n: int, inverse_scale: bool = False, coset_mode: int = COSET_NONE):
        """arithmetic::best_fft(a, omega, log_n) in place (numpy arrays are transformed in place too)."""
        assert _count(a, 32) == 1 << log_n, "assert_eq!(a.len(), 1 << log_n)"
        pa, k1 = _ptr(a)
        po, k2 = _ptr(omega)
        self._ck(lib().b200zk_ntt_fr(self._h, pa, log_n, po, int(inverse_scale), coset_mode))
        if not _is_torch(a) and k1 is not a:
            a[...] = k1.reshape(np.asarray(a).shape)
        return a

    def ntt_ext(self, a_in, log_in: int, out, log_n: int, omega, inverse_scale: bool = False, coset_mode: int = COSET_NONE):
        assert _count(a_in, 32) == 1 << log_in and _count(out, 32) == 1 << log_n
        pi, k1 = _ptr(a_in)
        po, k2 = _ptr(out)
        pw, k3 = _ptr(omega)
        self._ck(lib().b200zk_ntt_fr_ext(self._h, pi, log_in, po, log_n, pw, int(inverse_scale), coset_mode))
        return out

    # ---- quotient construction (device-resident columns: CUDA tensors)
    @staticmethod
    def _dev_table(cols):
        ptrs = [_ptr(c) for c in cols]
        return (C.c_void_p * max(1, len(ptrs)))(*[p.value for p, _ in ptrs]), ptrs

    def prefix_scan(self, op: int, a, init, out=None):
        """out[0] = init, out[i] = out[i-1] (* | +) a[i-1]: the z(X) / phi(X) loops of the permutation / lookup provers."""
        n = _count(a, 32)
        out = _like(a) if out is None else out
        pa, k1 = _ptr(a)
        pi, k2 = _ptr(init)
        po, k3 = _ptr(out)
        self._ck(lib().b200zk_prefix_scan(self._h, op, pa, n, pi, po))
        return out

    def poly_lincomb(self, polys, scalars, out):
        """out = sum_j scalars[j] * polys[j] in one pass (device-resident polynomials)."""
        n = _count(out, 32)
        tp, kp = self._dev_table(polys)
        sc = np.ascontiguousarray(np.asarray(scalars, dtype=np.uint64).reshape(-1, 4))
        assert len(sc) == len(polys)
        po, ko = _ptr(out)
        self._ck(lib().b200zk_poly_lincomb(self._h, po, tp, C.c_void_p(sc.ctypes.data) if len(sc) else None, len(polys), n))
        return out

    def permutation_product(self, values, sigma, beta, gamma, delta_omega_start, delta, omega, k: int, z_init, out):
        """permutation::Argument::commit, one column set: z(X) in Lagrange form (blinding rows left to the caller)."""
        assert len(values) == len(sigma) and _count(out, 32) == 1 << k
        tv, kv = self._dev_table(values)
        ts, ks = self._dev_table(sigma)
        sc = [_ptr(x) for x in (beta, gamma, delta_omega_start, delta, omega)]
        pz, kz = _ptr(z_init)
        po, ko = _ptr(out)
        self._ck(lib().b200zk_permutation_product(self._h, tv, ts, len(values), *[p for p, _ in sc], k, pz, po))
        return out

    def logup_running_sum(self, inputs, table, m, beta, k: int, phi_init, out):
        """mv_lookup prover: phi(X) running sum over sum_j 1/(f_j + beta) - m/(t + beta)."""
        ti, ki = self._dev_table(inputs)
        pt, k1 = _ptr(table)
        pm, k2 = _ptr(m)
        pb, k3 = _ptr(beta)
        pp, k4 = _ptr(phi_init)
        po, k5 = _ptr(out)
        self._ck(lib().b200zk_logup_running_sum(self._h, ti, len(inputs), pt, pm, pb, k, pp, po))
        return out

    def graph(self, calcs, constants, rotations) -> "Graph":
        return Graph(self, calcs, constants, rotations)

    # ---- poly ops
    def _ew(self, fn, r, *args, n):
        ptrs = [_ptr(x) for x in (r,) + args]
        self._ck(fn(self._h, *[p for p, _ in ptrs], n))
        return r

    def poly_add(self, a, b, out=None):
        n = _count(a, 32)
        out = _like(a) if out is None else out
        return self._ew(lib().b200zk_poly_add, out, a, b, n=n)

    def poly_sub(self, a, b, out=None):
        n = _count(a, 32)
        out = _like(a) if out is None else out
        return self._ew(lib().b200zk_poly_sub, out, a, b, n=n)

    def poly_mul(self, a, b, out=None):
        n = _count(a, 32)
        out = _like(a) if out is None else out
        return self._ew(lib().b200zk_poly_mul, out, a, b, n=n)

    def poly_scale(self, a, s, out=None):
        n = _count(a, 32)
        out = _like(a) if out is None else out
        return self._ew(lib().b200zk_poly_scale, out, a, s, n=n)

    def poly_axpy(self, a, s, b, out=None):
        n = _count(a, 32)
        out = _like(a) if out is None else out
        return self._ew(lib().b200zk_poly_axpy, out, a, s, b, n=n)

    def eval_polynomial(self, poly, point) -> np.ndarray:
        n = _count(poly, 32)
        out = np.zeros(4, np.uint64)
        pp, k1 = _ptr(poly)
        px, k2 = _ptr(point)
        self._ck(lib().b200zk_eval_poly(self._h, pp, n, px, out.ctypes.data))
        return out

    def compute_inner_product(self, a, b) -> np.ndarray:
        n = _count(a, 32)
        assert n == _count(b, 32)
        out = np.zeros(4, np.uint64)
        pa, k1 = _ptr(a)
        pb, k2 = _ptr(b)
        self._ck(lib().b200zk_inner_product(self._h, pa, pb, n, out.ctypes.data))
        return out

    def batch_invert(self, data):
        n = _count(data, 32)
        p, k = _ptr(data)
        self._ck(lib().b200zk_batch_invert(self._h, p, n))
        if not _is_torch(data) and k is not data:
            data[...] = k.reshape(np.asarray(data).shape)
        return data

    def kate_division(self, a, b) -> np.ndarray:
        n = _count(a, 32)
        assert n >= 1
        q = np.zeros((n - 1, 4), np.uint64)
        pa, k1 = _ptr(a)
        pb, k2 = _ptr(b)
        self._ck(lib().b200zk_kate_division(self._h, q.ctypes.data if n > 1 else None, pa, n, pb))
        return q

    def debug_field_op(self, field: int, op: int, a, b):
        n = _count(a, 32)
        r = np.zeros((n, 4), np.uint64)
        pa, k1 = _ptr(a)
        pb, k2 = _ptr(b)
        self._ck(lib().b200zk_debug_field_op(self._h, field, op, r.ctypes.data, pa, pb, n))
        return r


def _count(x, elem_bytes: int) -> int:
    if _is_torch(x):
        return x.numel() * x.element_size() // elem_bytes
    a = np.asarray(x)
    return a.size * a.itemsize // elem_bytes


def _like(a):
    if _is_torch(a):
        import torch

        return torch.empty_like(a)
    return np.zeros_like(np.asarray(a))


class Srs:
    """Device-resident bases (b200zk_srs): ParamsKZG::g or ::g_lagrange uploaded once."""

    def __init__(self, ctx: Context, bases, tag: int):
        self.ctx = ctx
        self.n = _count(bases, 64)
        self._h = C.c_void_p()
        p, k = _ptr(bases)
        ctx._ck(lib().b200zk_srs_register(ctx._h, p, self.n, tag, C.byref(self._h)))

    def msm(self, scalars, n: int | None = None) -> np.ndarray:
        n = _count(scalars, 32) if n is None else n
        out = np.zeros(12, np.uint64)
        p, k = _ptr(scalars)
        self.ctx._ck(lib().b200zk_msm_g1(self.ctx._h, self._h, p, n, out.ctypes.data))
        return out

    def msm_batch(self, columns, n: int | None = None) -> np.ndarray:
        """b200zk_msm_g1_batch: (count, 12) commitments of `columns` (host arrays / CUDA tensors) over the same bases."""
        count = len(columns)
        n = _count(columns[0], 32) if (n is None and count) else (n or 0)
        keep = [_ptr(c) for c in columns]
        arr = (C.c_void_p * max(count, 1))(*[p.value for p, _ in keep])
        out = np.zeros((count, 12), np.uint64)
        self.ctx._ck(lib().b200zk_msm_g1_batch(self.ctx._h, self._h, arr, count, n, out.ctypes.data))
        return out

    def msm_range(self, scalars, first: int, n: int | None = None) -> np.ndarray:
        """b200zk_msm_g1_range: sum_i scalars[i] * srs[first + i]."""
        n = _count(scalars, 32) if n is None else n
        out = np.zeros(12, np.uint64)
        p, k = _ptr(scalars)
        self.ctx._ck(lib().b200zk_msm_g1_range(self.ctx._h, self._h, p, first, n, out.ctypes.data))
        return out

    def msm_sharded(self, scalars_slice, n_total: int) -> np.ndarray:
        """b200zk_msm_g1_sharded: collective over the context's communicator; pass this rank's scalar slice."""
        out = np.zeros(12, np.uint64)
        p, k = _ptr(scalars_slice)
        self.ctx._ck(lib().b200zk_msm_g1_sharded(self.ctx._h, self._h, p, n_total, out.ctypes.data))
        return out

    def release(self):
        if self._h:
            lib().b200zk_srs_release(self.ctx._h, self._h)
            self._h = C.c_void_p()


class _ValueSource(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("index", C.c_uint32), ("rotation", C.c_uint32)]


class _Calculation(C.Structure):
    _fields_ = [("op", C.c_uint32), ("a", _ValueSource), ("b", _ValueSource), ("parts_offset", C.c_uint32), ("parts_len", C.c_uint32)]


# ValueSource kinds / Calculation ops of include/b200zk.h (plonk::evaluation, upstream declaration order)
SRC_CONSTANT, SRC_INTERMEDIATE, SRC_FIXED, SRC_ADVICE, SRC_INSTANCE, SRC_CHALLENGE, SRC_BETA, SRC_GAMMA, SRC_THETA, SRC_Y, \
    SRC_PREVIOUS_VALUE, SRC_EXTENDED_X = range(12)
CALC_ADD, CALC_SUB, CALC_MUL, CALC_SQUARE, CALC_DOUBLE, CALC_NEGATE, CALC_HORNER, CALC_STORE = range(8)
SCAN_PRODUCT, SCAN_SUM = 0, 1


def _pack_calcs(calcs):
    parts = []
    arr = (_Calculation * max(1, len(calcs)))()
    for i, (op, a, b, ps) in enumerate(calcs):
        arr[i].op = op
        arr[i].a = _ValueSource(*a)
        arr[i].b = _ValueSource(*(b if b is not None else (0, 0, 0)))
        arr[i].parts_offset = len(parts)
        arr[i].parts_len = len(ps or [])
        parts.extend(ps or [])
    parr = (_ValueSource * max(1, len(parts)))(*[_ValueSource(*q) for q in parts])
    return arr, parr, len(parts)


def graph_check(calcs, n_constants: int, n_rotations: int) -> dict:
    """b200zk_graph_check: validate + lower a program without a context or a device; raises B200zkError with the reason."""
    arr, parr, n_parts = _pack_calcs(calcs)
    ni, ns = C.c_uint32(), C.c_uint32()
    msg = C.create_string_buffer(256)
    rc = lib().b200zk_graph_check(C.cast(arr, C.c_void_p), len(calcs), C.cast(parr, C.c_void_p), n_parts, n_constants, n_rotations,
                                  C.byref(ni), C.byref(ns), msg, 256)
    if rc != OK:
        raise B200zkError(rc, msg.value.decode())
    return {"n_instructions": ni.value, "n_slots": ns.value}


class Graph:
    """plonk::evaluation::GraphEvaluator on the device (b200zk_graph).

    calcs: list of (op, a, b, parts); a / b / parts entries are ValueSources (kind, index, rotation_index); b is None
    for unary calculations, parts is a list only for CALC_HORNER (a = start value, b = factor)."""

    def __init__(self, ctx: Context, calcs, constants, rotations):
        self.ctx = ctx
        self._h = C.c_void_p()
        parts = []
        arr = (_Calculation * max(1, len(calcs)))()
        for i, (op, a, b, ps) in enumerate(calcs):
            arr[i].op = op
            arr[i].a = _ValueSource(*a)
            arr[i].b = _ValueSource(*(b if b is not None else (0, 0, 0)))
            arr[i].parts_offset = len(parts)
            arr[i].parts_len = len(ps or [])
            parts.extend(ps or [])
        parr = (_ValueSource * max(1, len(parts)))(*[_ValueSource(*q) for q in parts])
        consts = np.ascontiguousarray(np.asarray(constants, dtype=np.uint64).reshape(-1, 4))
        rots = np.ascontiguousarray(np.asarray(rotations, dtype=np.int32).reshape(-1))
        ctx._ck(lib().b200zk_graph_create(ctx._h, C.cast(arr, C.c_void_p), len(calcs), C.cast(parr, C.c_void_p), len(parts),
                                          C.c_void_p(consts.ctypes.data), len(consts), C.c_void_p(rots.ctypes.data), len(rots),
                                          C.byref(self._h)))

    def info(self):
        ni, ns = C.c_uint32(), C.c_uint32()
        lib().b200zk_graph_info(self._h, C.byref(ni), C.byref(ns))
        return {"n_instructions": ni.value, "n_slots": ns.value}

    def evaluate(self, values, log_size: int, rot_scale: int, fixed=(), advice=(), instance=(), challenges=None, beta=None,
                 gamma=None, theta=None, y=None, extended_omega=None, rows=None):
        """values[row] = GraphEvaluator::evaluate(.., previous_value = values[row], ..) for every row of the extended domain
        (rows = (first, count): only that slice -- evaluate_h sharded by row range, see Context.allgather_rows)."""
        assert _count(values, 32) == 1 << log_size
        if rows is not None:
            zero = np.zeros(4, np.uint64)
            tf, kf = Context._dev_table(fixed)
            ta, ka = Context._dev_table(advice)
            ti, ki = Context._dev_table(instance)
            ch = np.ascontiguousarray(np.asarray(challenges if challenges is not None else [], dtype=np.uint64).reshape(-1, 4))
            sc = [_ptr(zero if v is None else v) for v in (beta, gamma, theta, y)]
            pw, kw = _ptr(extended_omega)
            pv, kv = _ptr(values)
            self.ctx._ck(lib().b200zk_graph_evaluate_rows(self.ctx._h, self._h, tf, len(fixed), ta, len(advice), ti, len(instance),
                                                          C.c_void_p(ch.ctypes.data) if len(ch) else None, len(ch), *[p for p, _ in sc], pw,
                                                          pv, log_size, rot_scale, rows[0], rows[1]))
            return values
        zero = np.zeros(4, np.uint64)
        tf, kf = Context._dev_table(fixed)
        ta, ka = Context._dev_table(advice)
        ti, ki = Context._dev_table(instance)
        ch = np.ascontiguousarray(np.asarray(challenges if challenges is not None else [], dtype=np.uint64).reshape(-1, 4))
        sc = [_ptr(zero if v is None else v) for v in (beta, gamma, theta, y)]
        pw, kw = _ptr(extended_omega)
        pv, kv = _ptr(values)
        self.ctx._ck(lib().b200zk_graph_evaluate(self.ctx._h, self._h, tf, len(fixed), ta, len(advice), ti, len(instance),
                                                 C.c_void_p(ch.ctypes.data) if len(ch) else None, len(ch), *[p for p, _ in sc], pw, pv,
                                                 log_size, rot_scale))
        return values

    def evaluate_part(self, values, k: int, extended_k: int, part: int, fixed=(), advice=(), instance=(), challenges=None, beta=None,
                      gamma=None, theta=None, y=None):
        """The same on the 2^k rows of part `part` of the extended coset (b200zk_graph_evaluate_part): columns hold that part's
        values (EvaluationDomain.coeff_to_extended_parts), rotations wrap within the part."""
        assert _count(values, 32) == 1 << k
        zero = np.zeros(4, np.uint64)
        tf, kf = Context._dev_table(fixed)
        ta, ka = Context._dev_table(advice)
        ti, ki = Context._dev_table(instance)
        ch = np.ascontiguousarray(np.asarray(challenges if challenges is not None else [], dtype=np.uint64).reshape(-1, 4))
        sc = [_ptr(zero if v is None else v) for v in (beta, gamma, theta, y)]
        pv, kv = _ptr(values)
        self.ctx._ck(lib().b200zk_graph_evaluate_part(self.ctx._h, self._h, tf, len(fixed), ta, len(advice), ti, len(instance),
                                                      C.c_void_p(ch.ctypes.data) if len(ch) else None, len(ch), *[p for p, _ in sc], k,
                                                      extended_k, part, pv))
        return values

    def release(self):
        if self._h:
            lib().b200zk_graph_destroy(self.ctx._h, self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class _ColumnJob(C.Structure):
    _fields_ = [("host_values", C.c_void_p), ("srs", C.c_void_p), ("mode", C.c_int32), ("coeff_out_dev", C.c_void_p),
                ("ext_out_dev", C.c_void_p)]


def run_column_jobs(ctx: "Context", jobs, k: int, omega_inv=None, extended_omega=None, extended_omega_inv=None,
                    extended_k: int = 0) -> np.ndarray:
    """b200zk_run_column_jobs: jobs = [(host_values, srs_or_None, mode, coeff_out_or_None, ext_out_or_None), ...]."""
    count = len(jobs)
    arr = (_ColumnJob * max(count, 1))()
    keep = []
    for i, (vals, srs, mode, co, eo) in enumerate(jobs):
        pv, k1 = _ptr(vals)
        pc, k2 = _ptr(co)
        pe, k3 = _ptr(eo)
        keep += [k1, k2, k3]
        arr[i].host_values = pv.value
        arr[i].srs = srs._h.value if srs is not None else None
        arr[i].mode = mode
        arr[i].coeff_out_dev = pc.value if pc is not None else None
        arr[i].ext_out_dev = pe.value if pe is not None else None
    out = np.zeros((count, 12), np.uint64)
    po, k4 = _ptr(omega_inv)
    pe1, k5 = _ptr(extended_omega)
    pe2, k6 = _ptr(extended_omega_inv)
    ctx._ck(lib().b200zk_run_column_jobs(ctx._h, C.cast(arr, C.c_void_p), count, k, po, pe1, pe2, extended_k, out.ctypes.data))
    return out


def commit_columns(ctx: "Context", srs: "Srs", host_cols, k: int, mode: int = 0, omega_inv=None, extended_omega=None,
                   extended_k: int = 0, coeff_out=None, ext_out=None) -> np.ndarray:
    """b200zk_commit_columns: host columns (numpy arrays or pinned torch CPU tensors, 2^k x 4 u64 each) ->
    (count, 12) commitments; mode 1/2 also runs lagrange_to_coeff / coeff_to_extended on the device."""
    count = len(host_cols)
    keep = [_ptr(c) for c in host_cols]
    arr = (C.c_void_p * max(count, 1))(*[p for p, _ in keep])
    out = np.zeros((count, 12), np.uint64)

    def ptr_array(bufs):
        if bufs is None:
            return None, None
        ks = [_ptr(b) for b in bufs]
        return (C.c_void_p * max(count, 1))(*[p for p, _ in ks]), ks

    ca, k1 = ptr_array(coeff_out)
    ea, k2 = ptr_array(ext_out)
    po, k3 = _ptr(omega_inv)
    pe, k4 = _ptr(extended_omega)
    ctx._ck(lib().b200zk_commit_columns(ctx._h, srs._h if srs is not None else None, arr, count, k, po, pe, extended_k,
                                        out.ctypes.data, ca, ea, mode))
    return out


class ParamsKZG:
    """halo2_proofs::poly::kzg::commitment::ParamsKZG<Bn256> with device-resident g / g_lagrange."""

    def __init__(self, ctx: Context, k: int, g, g_lagrange=None):
        self.ctx, self.k, self.n = ctx, k, 1 << k
        assert _count(g, 64) == self.n
        self._g = ctx.srs_register(g, SRS_G)
        self._gl = ctx.srs_register(g_lagrange, SRS_G_LAGRANGE) if g_lagrange is not None else None

    def commit(self, poly) -> np.ndarray:
        """ParamsProver::commit(poly, Blind): best_multiexp over g[..poly.len()] (blind ignored for KZG)."""
        return self._g.msm(poly)

    def commit_lagrange(self, poly) -> np.ndarray:
        assert self._gl is not None
        return self._gl.msm(poly)

    def release(self):
        self._g.release()
        if self._gl:
            self._gl.release()


class EvaluationDomain:
    """halo2_proofs::poly::EvaluationDomain::new(j, k) (poly/domain.rs): host constants + device transforms."""

    def __init__(self, ctx: Context, j: int, k: int):
        self.ctx, self.k = ctx, k
        self.quotient_poly_degree = j - 1
        self.n = 1 << k
        ek = k
        while (1 << ek) < self.n * self.quotient_poly_degree:
            ek += 1
        assert ek <= FR_S
        self.extended_k = ek
        eo = pow(_ROOT_OF_UNITY, 1 << (FR_S - ek), R_MOD)
        om = pow(eo, 1 << (ek - k), R_MOD)
        self.extended_omega, self.omega = fr_from_int(eo), fr_from_int(om)
        self.extended_omega_inv, self.omega_inv = fr_from_int(pow(eo, -1, R_MOD)), fr_from_int(pow(om, -1, R_MOD))
        self.g_coset, self.g_coset_inv = fr_from_int(_ZETA), fr_from_int(_ZETA * _ZETA % R_MOD)
        self.ifft_divisor = fr_from_int(pow(self.n, -1, R_MOD))
        self.extended_ifft_divisor = fr_from_int(pow(1 << ek, -1, R_MOD))

    def lagrange_to_coeff(self, a):
        """ifft(a, omega_inv, k, ifft_divisor) in place."""
        return self.ctx.best_fft(a, self.omega_inv, self.k, inverse_scale=True)

    def coeff_to_extended(self, a, out=None):
        """distribute_powers_zeta(into_coset) + zero-extend + best_fft(extended_omega): n -> 2^extended_k."""
        if out is None:
            if _is_torch(a):
                import torch

                out = torch.empty((1 << self.extended_k, 4), dtype=a.dtype, device=a.device)
            else:
                out = np.zeros((1 << self.extended_k, 4), np.uint64)
        return self.ctx.ntt_ext(a, self.k, out, self.extended_k, self.extended_omega, False, COSET_PRE)

    def extended_to_coeff(self, a):
        """ifft(extended_omega_inv) + distribute_powers_zeta(out of coset); returns the first n*(j-1) coefficients."""
        self.ctx.best_fft(a, self.extended_omega_inv, self.extended_k, inverse_scale=True, coset_mode=COSET_POST)
        return a[: self.n * self.quotient_poly_degree]

    @property
    def n_parts(self) -> int:
        """J = 2^(extended_k - k): the extended coset is J parts of n points, part r = zeta * extended_omega^r * <omega>."""
        return 1 << (self.extended_k - self.k)

    def coeff_to_extended_parts(self, coeffs, part: int, outs):
        """outs[j][i] = coeffs[j](zeta * extended_omega^part * omega^i): coeff_to_extended(coeffs[j])[part::J] (outs: CUDA tensors)."""
        assert len(coeffs) == len(outs)
        assert all(_count(c, 32) == self.n for c in coeffs) and all(_count(o, 32) == self.n for o in outs)
        ti, ki = Context._dev_table(coeffs)
        to, ko = Context._dev_table(outs)
        self.ctx._ck(lib().b200zk_coeff_to_extended_parts(self.ctx._h, ti, len(coeffs), self.k, self.extended_k, part, to))
        return outs

    def extended_parts_to_coeff(self, parts, divide_by_vanishing: bool = False, n_pieces: int | None = None, out=None):
        """parts: CUDA tensor of 2^extended_k elements, part-major (consumed).  Returns n_pieces * n coefficients (default
        n_pieces = quotient_poly_degree): extended_to_coeff of the interleaved vector, after divide_by_vanishing_poly if asked."""
        assert _count(parts, 32) == 1 << self.extended_k
        n_pieces = self.quotient_poly_degree if n_pieces is None else n_pieces
        out = parts if out is None else out
        pp, kp = _ptr(parts)
        po, ko = _ptr(out)
        self.ctx._ck(lib().b200zk_extended_parts_to_coeff(self.ctx._h, pp, self.k, self.extended_k, n_pieces, int(divide_by_vanishing), po))
        return out[: n_pieces * self.n]
