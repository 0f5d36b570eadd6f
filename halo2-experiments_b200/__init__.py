"""Host-side mirror of the halo2_proofs back-end interface over libb200zk.so (ctypes).

Names and argument meaning follow halo2_proofs v2023_02_02 (the crate the reference
pins at /root/reference/Cargo.toml:10 and calls from
/root/reference/src/circuits/utils.rs:22-70):

    best_multiexp(coeffs, bases) -> G1            arithmetic.rs
    best_fft(a, omega, log_n)                     arithmetic.rs
    EvaluationDomain(j, k).lagrange_to_coeff / coeff_to_extended /
        extended_to_coeff / divide_by_vanishing_poly      poly/domain.rs
    ParamsKZG.load / setup / downsize, .commit, .commit_lagrange      poly/kzg/commitment.rs
    g_to_lagrange(backend, g, k)                  arithmetic.rs

Arrays are numpy uint64, shape (n, 4) for Fr (Montgomery limbs, the memory layout of
halo2curves' Fr), (n, 8) for G1Affine, (12,) for a G1 result.  Everything computes on
the GPU through the C ABI declared in include/b200zk.h; there is no CPU fallback —
importing works anywhere, but creating a Backend without a CUDA device raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200zk.so")

OK, EINVAL, ENODEV, ECUDA, ENOMEM, ESYNTH, EVERIFY = 0, -1, -2, -3, -4, -5, -6


class B200zkError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libb200zk.so (fails loudly if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200zkError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        L = ctypes.CDLL(LIB_PATH)
        L.b200zk_last_error.restype = ctypes.c_char_p
        L.b200zk_launch_count.restype = ctypes.c_uint64
        L.b200zk_domain_k.restype = ctypes.c_uint32
        L.b200zk_domain_extended_k.restype = ctypes.c_uint32
        L.b200zk_domain_quotient_poly_degree.restype = ctypes.c_uint32
        L.b200zk_domain_destroy.restype = None
        L.b200zk_params_destroy.restype = None
        L.b200zk_ctx_destroy.restype = None
        _lib = L
    return _lib


def _p(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(ctypes.c_void_p)
    return a


def _fr(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    a = a.reshape(-1, 4)
    if n is not None and a.shape[0] != n:
        raise B200zkError(f"expected {n} field elements, got {a.shape[0]}")
    return a


class DeviceBuffer:
    """Device memory owned by a Backend (b200zk_malloc)."""

    def __init__(self, backend, nbytes):
        self.backend, self.nbytes = backend, int(nbytes)
        ptr = ctypes.c_void_p()
        backend._check(lib().b200zk_malloc(backend._ctx, ctypes.c_size_t(self.nbytes), ctypes.byref(ptr)))
        self.ptr = ptr

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        self.backend._check(lib().b200zk_upload(self.backend._ctx, self.ptr, _p(arr), ctypes.c_size_t(arr.nbytes)))
        return self

    def download(self, shape, dtype=np.uint64):
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        self.backend._check(lib().b200zk_download(self.backend._ctx, _p(out), self.ptr, ctypes.c_size_t(out.nbytes)))
        return out

    def free(self):
        if self.ptr is not None:
            lib().b200zk_free(self.backend._ctx, self.ptr)
            self.ptr = None


class Backend:
    """One CUDA device + stream + scratch (b200zk_ctx)."""

    def __init__(self, device=0, _ctx=None):
        self._borrowed = _ctx is not None           # a group's ctx: the group destroys it
        if _ctx is not None:
            self._ctx = _ctx
            return
        self._ctx = ctypes.c_void_p()
        rc = lib().b200zk_ctx_create(ctypes.c_int32(device), ctypes.byref(self._ctx))
        if rc != OK:
            self._ctx = None
            raise B200zkError(f"b200zk_ctx_create(device={device}) failed with code {rc}: no usable sm_100 CUDA device "
                              "(this backend has no CPU fallback)")

    def close(self):
        if self._ctx and not self._borrowed:
            lib().b200zk_ctx_destroy(self._ctx)
        self._ctx = None

    # -- one proof over several GPUs, one process per GPU (NCCL inside the library) --
    @staticmethod
    def comm_unique_id():
        """128-byte rendezvous id (rank 0 creates it and hands it to the other ranks, e.g. with
        torch.distributed.broadcast_object_list)."""
        buf = (ctypes.c_uint8 * 128)()
        rc = lib().b200zk_comm_unique_id(buf)
        if rc != OK:
            raise B200zkError(f"b200zk_comm_unique_id failed: {rc} (libnccl.so.2 not loadable?)")
        return bytes(buf)

    def comm_init(self, world, rank, unique_id):
        """Collective: after it, create_proof on this backend's proving keys is rank `rank` of one proof
        sharded over `world` GPUs (every rank calls it with the same inputs, every rank gets the proof)."""
        self._check(lib().b200zk_ctx_comm_init(self._ctx, ctypes.c_uint32(world), ctypes.c_uint32(rank),
                                               (ctypes.c_uint8 * 128).from_buffer_copy(unique_id)))

    def comm_destroy(self):
        self._check(lib().b200zk_ctx_comm_destroy(self._ctx))

    def _check(self, rc):
        if rc != OK:
            raise B200zkError(f"b200zk error {rc}: {lib().b200zk_last_error(self._ctx).decode()}")

    # -- plumbing --
    def sync(self):
        self._check(lib().b200zk_sync(self._ctx))

    def profiler_range(self, start):
        self._check(lib().b200zk_profiler_range(self._ctx, ctypes.c_int32(1 if start else 0)))

    def launch_count(self):
        return int(lib().b200zk_launch_count(self._ctx))

    def event_record(self, slot):
        self._check(lib().b200zk_event_record(self._ctx, ctypes.c_uint32(slot)))

    def event_elapsed_ms(self, a, b):
        ms = ctypes.c_float()
        self._check(lib().b200zk_event_elapsed_ms(self._ctx, ctypes.c_uint32(a), ctypes.c_uint32(b), ctypes.byref(ms)))
        return float(ms.value)

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, arr.nbytes).upload(arr)

    def pinned_empty(self, shape, dtype=np.uint64):
        """numpy view over cudaHostAlloc'ed memory (kept alive by the returned array's base)."""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = ctypes.c_void_p()
        self._check(lib().b200zk_host_alloc(self._ctx, ctypes.c_size_t(nbytes), ctypes.byref(ptr)))
        buf = (ctypes.c_uint8 * nbytes).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def set_msm_window(self, c):
        self._check(lib().b200zk_msm_set_window(self._ctx, ctypes.c_int32(c)))

    # -- arithmetic.rs --
    def best_multiexp(self, coeffs, bases):
        """sum coeffs[i] * bases[i]; panics upstream on length mismatch -> raises here."""
        coeffs = _fr(coeffs)
        bases = np.ascontiguousarray(bases, dtype=np.uint64).reshape(-1, 8)
        if coeffs.shape[0] != bases.shape[0]:
            raise B200zkError("best_multiexp: coeffs.len() != bases.len()")
        out = np.zeros(12, dtype=np.uint64)
        self._check(lib().b200zk_msm(self._ctx, _p(coeffs), _p(bases), ctypes.c_size_t(coeffs.shape[0]), _p(out)))
        return out

    def best_multiexp_dev(self, d_coeffs, d_bases, n):
        out = np.zeros(12, dtype=np.uint64)
        self._check(lib().b200zk_msm_dev(self._ctx, d_coeffs.ptr, d_bases.ptr, ctypes.c_size_t(n), _p(out)))
        return out

    def best_fft(self, a, omega, log_n):
        """In-place on a copy; returns the transformed array (natural order, unscaled)."""
        a = np.array(_fr(a, 1 << log_n))
        self._check(lib().b200zk_fft(self._ctx, _p(a), _p(_fr(omega, 1)), ctypes.c_uint32(log_n)))
        return a

    def best_fft_dev(self, d_a, omega, log_n):
        self._check(lib().b200zk_fft_dev(self._ctx, d_a.ptr, _p(_fr(omega, 1)), ctypes.c_uint32(log_n)))

    def g_to_lagrange_dev(self, d_g, k, d_out):
        """arithmetic::g_to_lagrange on 2^k device-resident G1Affine points; d_out may be d_g."""
        self._check(lib().b200zk_g_to_lagrange_dev(self._ctx, _p(d_g.ptr if d_g is not None else None), ctypes.c_uint32(k),
                                                   _p(d_out.ptr if d_out is not None else None)))

    def eval_polynomial(self, poly, x):
        poly = _fr(poly)
        out = np.zeros(4, dtype=np.uint64)
        self._check(lib().b200zk_eval_polynomial(self._ctx, _p(poly), ctypes.c_size_t(poly.shape[0]), _p(_fr(x, 1)), _p(out)))
        return out

    def eval_polynomial_dev(self, d_poly, n, x):
        out = np.zeros(4, dtype=np.uint64)
        self._check(lib().b200zk_eval_polynomial_dev(self._ctx, d_poly.ptr, ctypes.c_size_t(n), _p(_fr(x, 1)), _p(out)))
        return out

    def kate_division(self, a, b):
        """Quotient of a(X) by (X - b): len(a) - 1 coefficients."""
        a = _fr(a)
        n = a.shape[0]
        d_a, d_q = self.to_device(a), self.alloc(max(n - 1, 1) * 32)
        try:
            self._check(lib().b200zk_kate_division_dev(self._ctx, d_a.ptr, ctypes.c_size_t(n), _p(_fr(b, 1)), d_q.ptr))
            return d_q.download((n - 1, 4))
        finally:
            d_a.free(); d_q.free()

    def batch_invert(self, a, field=0):
        a = _fr(a)
        d = self.to_device(a)
        try:
            self._check(lib().b200zk_batch_invert_dev(self._ctx, d.ptr, ctypes.c_size_t(a.shape[0]), ctypes.c_int32(field)))
            return d.download(a.shape)
        finally:
            d.free()

    def prefix_product(self, p, z0):
        """z[0] = z0, z[i] = z[i-1] * p[i-1]."""
        p = _fr(p)
        d = self.to_device(p)
        try:
            self._check(lib().b200zk_prefix_product_dev(self._ctx, d.ptr, d.ptr, ctypes.c_size_t(p.shape[0]), _p(_fr(z0, 1))))
            return d.download(p.shape)
        finally:
            d.free()


class EvaluationDomain:
    """poly::EvaluationDomain<Fr>::new(j, k) on a Backend."""
    _CONSTS = ["omega", "omega_inv", "extended_omega", "extended_omega_inv", "g_coset", "g_coset_inv",
               "ifft_divisor", "extended_ifft_divisor", "barycentric_weight"]

    def __init__(self, backend, j, k):
        self.backend = backend
        self._h = ctypes.c_void_p()
        backend._check(lib().b200zk_domain_create(backend._ctx, ctypes.c_uint32(j), ctypes.c_uint32(k), ctypes.byref(self._h)))
        self.k = int(lib().b200zk_domain_k(self._h))
        self.n = 1 << self.k
        self.extended_k = int(lib().b200zk_domain_extended_k(self._h))
        self.quotient_poly_degree = int(lib().b200zk_domain_quotient_poly_degree(self._h))
        for i, name in enumerate(self._CONSTS):
            v = np.zeros(4, dtype=np.uint64)
            backend._check(lib().b200zk_domain_constant(self._h, ctypes.c_uint32(i), _p(v)))
            setattr(self, name, v)

    def close(self):
        if self._h:
            lib().b200zk_domain_destroy(self._h)
            self._h = None

    def extended_len(self):
        return 1 << self.extended_k

    def lagrange_to_coeff(self, a):
        a = np.array(_fr(a, self.n))
        self.backend._check(lib().b200zk_lagrange_to_coeff(self._h, _p(a)))
        return a

    def coeff_to_extended(self, a):
        a = _fr(a, self.n)
        out = np.empty((self.extended_len(), 4), dtype=np.uint64)
        self.backend._check(lib().b200zk_coeff_to_extended(self._h, _p(a), _p(out)))
        return out

    def extended_to_coeff(self, a):
        a = _fr(a, self.extended_len())
        out = np.empty((self.n * self.quotient_poly_degree, 4), dtype=np.uint64)
        self.backend._check(lib().b200zk_extended_to_coeff(self._h, _p(a), _p(out)))
        return out

    def divide_by_vanishing_poly(self, a):
        a = np.array(_fr(a, self.extended_len()))
        self.backend._check(lib().b200zk_divide_by_vanishing_poly(self._h, _p(a)))
        return a

    def rotate_omega(self, value, rotation):
        out = np.zeros(4, dtype=np.uint64)
        self.backend._check(lib().b200zk_domain_rotate_omega(self._h, _p(_fr(value, 1)), ctypes.c_int32(rotation), _p(out)))
        return out

    def l_i_range(self, x, rot_lo, rot_hi):
        """l_i(x) for i in rot_lo..=rot_hi (upstream's l_i_range(x, x^n, rot_lo..=rot_hi))."""
        out = np.zeros((rot_hi - rot_lo + 1, 4), dtype=np.uint64)
        self.backend._check(lib().b200zk_domain_l_i_range(self._h, _p(_fr(x, 1)), ctypes.c_int32(rot_lo), ctypes.c_int32(rot_hi), _p(out)))
        return out

    def rotate_extended(self, a, rotation):
        a = _fr(a, self.extended_len())
        d_in, d_out = self.backend.to_device(a), self.backend.alloc(a.nbytes)
        self.backend._check(lib().b200zk_rotate_extended_dev(self._h, d_in.ptr, ctypes.c_int32(rotation), d_out.ptr))
        out = d_out.download(a.shape)
        d_in.free(); d_out.free()
        return out

    # device-resident variants (DeviceBuffer in, DeviceBuffer out)
    def lagrange_to_coeff_dev(self, d_a):
        self.backend._check(lib().b200zk_lagrange_to_coeff_dev(self._h, d_a.ptr))

    def coeff_to_extended_dev(self, d_coeffs, d_out):
        self.backend._check(lib().b200zk_coeff_to_extended_dev(self._h, d_coeffs.ptr, d_out.ptr))

    def extended_to_coeff_dev(self, d_ext, d_out):
        self.backend._check(lib().b200zk_extended_to_coeff_dev(self._h, d_ext.ptr, d_out.ptr))

    def divide_by_vanishing_poly_dev(self, d_ext):
        self.backend._check(lib().b200zk_divide_by_vanishing_poly_dev(self._h, d_ext.ptr))


ESYNTH = -5


def _ptr_array(arrays):
    """(void* const*) over a list of contiguous numpy arrays (kept alive by the caller)."""
    arr = (ctypes.c_void_p * max(len(arrays), 1))()
    for i, a in enumerate(arrays):
        arr[i] = a.ctypes.data
    return arr


class ProvingKey:
    """plonk::ProvingKey built by keygen_pk, resident on the device (b200zk_pk_create)."""

    def __init__(self, params, cs, k, fixed_columns, map_col, map_row):
        self.params, self.backend, self.cs, self.k, self.n = params, params.backend, cs, k, 1 << k
        blob = np.ascontiguousarray(cs.to_blob(k), dtype=np.uint32)
        fixed = [np.ascontiguousarray(f, dtype=np.uint64).reshape(self.n, 4) for f in fixed_columns]
        if len(fixed) != cs.num_fixed:
            raise B200zkError("fixed column count does not match the constraint system")
        mc = None if map_col is None else np.ascontiguousarray(map_col, dtype=np.uint32)
        mr = None if map_row is None else np.ascontiguousarray(map_row, dtype=np.uint32)
        self._h = ctypes.c_void_p()
        L = lib()
        L.b200zk_pk_proof_size.restype = ctypes.c_size_t
        L.b200zk_pk_rng_draws.restype = ctypes.c_size_t
        L.b200zk_pk_blinding_factors.restype = ctypes.c_uint32
        L.b200zk_pk_degree.restype = ctypes.c_uint32
        L.b200zk_pk_destroy.restype = None
        self.backend._check(L.b200zk_pk_create(params._h, _p(blob), ctypes.c_size_t(blob.shape[0]), _ptr_array(fixed),
                                               _p(mc), _p(mr), ctypes.byref(self._h)))
        self.proof_size = int(L.b200zk_pk_proof_size(self._h))
        self.rng_draws = int(L.b200zk_pk_rng_draws(self._h))
        self.blinding_factors = int(L.b200zk_pk_blinding_factors(self._h))
        self.degree = int(L.b200zk_pk_degree(self._h))

    def close(self):
        if self._h:
            lib().b200zk_pk_destroy(self._h)
            self._h = None

    def _instances(self, instances):
        cols = [np.ascontiguousarray(c, dtype=np.uint64).reshape(-1, 4) for c in instances]
        lens = np.array([c.shape[0] for c in cols], dtype=np.uint32)
        keep = [c if c.shape[0] else np.zeros((1, 4), dtype=np.uint64) for c in cols]
        return keep, _ptr_array(keep), lens

    def create_proof(self, advice_columns, instances, rng_wide, transcript_repr):
        """plonk::create_proof for one circuit.  advice_columns: A arrays (n,4) as synthesised
        (unblinded); instances: list of (len,4) Montgomery arrays; rng_wide: (rng_draws, 8) uint64,
        the 512-bit inputs of each Fr::random call in order; transcript_repr: Fr (4,)."""
        adv = [np.ascontiguousarray(a, dtype=np.uint64).reshape(self.n, 4) for a in advice_columns]
        if len(adv) != self.cs.num_advice:
            raise B200zkError("advice column count does not match the constraint system")
        keep, inst_ptrs, lens = self._instances(instances)
        wide = np.ascontiguousarray(rng_wide, dtype=np.uint64).reshape(-1, 8)
        if wide.shape[0] < self.rng_draws:
            raise B200zkError(f"rng stream too short: need {self.rng_draws} draws")
        out = np.zeros(self.proof_size, dtype=np.uint8)
        ln = ctypes.c_size_t()
        self.backend._check(lib().b200zk_create_proof(self._h, _ptr_array(adv), inst_ptrs, _p(lens), _p(wide), _p(_fr(transcript_repr, 1)),
                                                       _p(out), ctypes.c_size_t(out.shape[0]), ctypes.byref(ln)))
        return bytes(out[: ln.value])

    def create_proof_dev(self, d_advice, instances, d_rng_wide, transcript_repr):
        """Same with the A x n advice block and the rng stream already in device memory."""
        keep, inst_ptrs, lens = self._instances(instances)
        out = np.zeros(self.proof_size, dtype=np.uint8)
        ln = ctypes.c_size_t()
        self.backend._check(lib().b200zk_create_proof_dev(self._h, d_advice.ptr, inst_ptrs, _p(lens), d_rng_wide.ptr, _p(_fr(transcript_repr, 1)),
                                                           _p(out), ctypes.c_size_t(out.shape[0]), ctypes.byref(ln)))
        return bytes(out[: ln.value])

    def reserve_lanes(self, want=0):
        """Reserve up to `want` proof lanes for create_proofs (0 = the planner's default) and keep that request for later
        batches; returns the number of lanes memory allowed (>= 1)."""
        got = ctypes.c_uint32()
        self.backend._check(lib().b200zk_pk_reserve_lanes(self._h, ctypes.c_uint32(want), ctypes.byref(got)))
        return int(got.value)

    def _batch(self, fn, count, advice_ptrs, instances_list, rng_ptrs, transcript_repr):
        if len(instances_list) != count:
            raise B200zkError("one instance list per proof")
        keep, lens = [], []
        for instances in instances_list:
            if len(instances) != self.cs.num_instance:
                raise B200zkError("instance column count does not match the constraint system")
            k, _, ln = self._instances(instances)
            keep += k
            lens.append(ln)
        lens = np.concatenate(lens) if lens else np.zeros(0, dtype=np.uint32)
        out = np.zeros((count, self.proof_size), dtype=np.uint8)
        status = np.zeros(count, dtype=np.int32)
        rc = fn(self._h, ctypes.c_uint32(count), advice_ptrs, _ptr_array(keep), _p(lens), rng_ptrs, _p(_fr(transcript_repr, 1)),
                _p(out), ctypes.c_size_t(out.nbytes), _p(status))
        if rc != ESYNTH:
            self.backend._check(rc)
        return [None if status[i] == ESYNTH else bytes(out[i]) for i in range(count)]

    def create_proofs(self, advice_list, instances_list, rng_list, transcript_repr):
        """create_proof for several witnesses of this key at once, on concurrent lanes of its device: proof i is exactly
        create_proof(advice_list[i], instances_list[i], rng_list[i], transcript_repr).  Returns a list of bytes, None
        where the witness hit ConstraintSystemFailure (or its instances were too large)."""
        count = len(advice_list)
        if len(rng_list) != count:
            raise B200zkError("one rng stream per proof")
        adv = []
        for advice in advice_list:
            cols = [np.ascontiguousarray(a, dtype=np.uint64).reshape(self.n, 4) for a in advice]
            if len(cols) != self.cs.num_advice:
                raise B200zkError("advice column count does not match the constraint system")
            adv += cols
        wides = [np.ascontiguousarray(w, dtype=np.uint64).reshape(-1, 8) for w in rng_list]
        if any(w.shape[0] < self.rng_draws for w in wides):
            raise B200zkError(f"rng stream too short: need {self.rng_draws} draws")
        return self._batch(lib().b200zk_create_proofs, count, _ptr_array(adv), instances_list, _ptr_array(wides), transcript_repr)

    def create_proofs_dev(self, d_advice_list, instances_list, d_rng_list, transcript_repr):
        """Same with proof i's A x n advice block and rng stream already in device memory (DeviceBuffers)."""
        count = len(d_advice_list)
        if len(d_rng_list) != count:
            raise B200zkError("one rng stream per proof")
        adv = (ctypes.c_void_p * max(count, 1))(*[d.ptr.value for d in d_advice_list])
        rng = (ctypes.c_void_p * max(count, 1))(*[d.ptr.value for d in d_rng_list])
        return self._batch(lib().b200zk_create_proofs_dev, count, adv, instances_list, rng, transcript_repr)

    def vk_commitments(self):
        """keygen_vk's commitments: (fixed (F, 8), sigma (P, 8)) G1Affine Montgomery limbs, computed on the device."""
        fixed = np.zeros((max(self.cs.num_fixed, 1), 8), dtype=np.uint64)
        sigma = np.zeros((max(len(self.cs.permutation), 1), 8), dtype=np.uint64)
        self.backend._check(lib().b200zk_pk_vk_commitments(self._h, _p(fixed), _p(sigma)))
        return fixed[: self.cs.num_fixed], sigma[: len(self.cs.permutation)]

    def quotient_muls(self):
        """{gates, permutation, lookups} field multiplications per row of evaluate_h, and the coset counts."""
        out = (ctypes.c_uint32 * 5)()
        self.backend._check(lib().b200zk_pk_quotient_muls(self._h, out))
        return {"gates": out[0], "permutation": out[1], "lookups": out[2], "cosets": out[3], "lookup_cosets": out[4]}

    def last_trace(self):
        """[(label, ms since the call)] at the synchronisation points of the last create_proof (host wall clock)."""
        buf = ctypes.create_string_buffer(4096)
        self.backend._check(lib().b200zk_pk_last_trace(self._h, buf, ctypes.c_size_t(4096)))
        return [(a, float(b)) for a, b in (item.split(":") for item in buf.value.decode().split(";") if item)]

    def last_phase_ms(self):
        out = (ctypes.c_float * 7)()
        self.backend._check(lib().b200zk_pk_last_phase_ms(self._h, out))
        return dict(zip(["msm", "ntt", "quotient", "lookup", "permutation", "open", "other"], [float(x) for x in out]))


class Group:
    """Several GPUs driven from this process (b200zk_group_*): `backends[r]` is rank r's Backend.  Build the
    params and a ProvingKey on every backend, then `create_proof(pks, ...)` shards ONE proof over the ranks.
    `devices` may repeat a device (ranks then share it: the single-GPU test configuration)."""

    def __init__(self, devices):
        L = lib()
        L.b200zk_group_ctx.restype = ctypes.c_void_p
        L.b200zk_group_size.restype = ctypes.c_uint32
        L.b200zk_group_destroy.restype = None
        self._h = ctypes.c_void_p()
        arr = (ctypes.c_int32 * len(devices))(*devices)
        rc = L.b200zk_group_create(arr, ctypes.c_uint32(len(devices)), ctypes.byref(self._h))
        if rc != OK:
            self._h = None
            raise B200zkError(f"b200zk_group_create({list(devices)}) failed with code {rc}")
        self.backends = [Backend(_ctx=ctypes.c_void_p(L.b200zk_group_ctx(self._h, ctypes.c_uint32(r)))) for r in range(len(devices))]

    def close(self):
        if self._h:
            lib().b200zk_group_destroy(self._h)
            self._h = None
            for b in self.backends:
                b._ctx = None

    def best_multiexp(self, coeffs, bases):
        """arithmetic::best_multiexp split by point range over the group's GPUs (partial sums combined in the library)."""
        coeffs = _fr(coeffs)
        bases = np.ascontiguousarray(bases, dtype=np.uint64).reshape(-1, 8)
        if coeffs.shape[0] != bases.shape[0]:
            raise B200zkError("best_multiexp: coeffs.len() != bases.len()")
        out = np.zeros(12, dtype=np.uint64)
        self.backends[0]._check(lib().b200zk_group_msm(self._h, _p(coeffs), _p(bases), ctypes.c_size_t(coeffs.shape[0]), _p(out)))
        return out

    def best_fft(self, a, omega, log_n):
        """arithmetic::best_fft, four-step over the group's GPUs with the exchange fused into the column-step kernel."""
        a = np.array(_fr(a, 1 << log_n))
        self.backends[0]._check(lib().b200zk_group_fft(self._h, _p(a), _p(_fr(omega, 1)), ctypes.c_uint32(log_n)))
        return a

    def create_proof(self, pks, advice_columns, instances, rng_wide, transcript_repr):
        """One plonk::create_proof over all ranks from host inputs (pks[r] built on backends[r])."""
        pk0 = pks[0]
        adv = [np.ascontiguousarray(a, dtype=np.uint64).reshape(pk0.n, 4) for a in advice_columns]
        keep, inst_ptrs, lens = pk0._instances(instances)
        wide = np.ascontiguousarray(rng_wide, dtype=np.uint64).reshape(-1, 8)
        if wide.shape[0] < pk0.rng_draws:
            raise B200zkError(f"rng stream too short: need {pk0.rng_draws} draws")
        out = np.zeros(pk0.proof_size, dtype=np.uint8)
        ln = ctypes.c_size_t()
        handles = (ctypes.c_void_p * len(pks))(*[p._h for p in pks])
        self.backends[0]._check(lib().b200zk_group_create_proof(self._h, handles, _ptr_array(adv), inst_ptrs, _p(lens), _p(wide),
                                                                _p(_fr(transcript_repr, 1)), _p(out), ctypes.c_size_t(out.shape[0]), ctypes.byref(ln)))
        return bytes(out[: ln.value])

    def create_proof_dev(self, pks, d_advice, instances, d_rng_wide, transcript_repr):
        """Same with rank r's inputs resident on its device: d_advice[r], d_rng_wide[r] DeviceBuffers."""
        pk0 = pks[0]
        keep, inst_ptrs, lens = pk0._instances(instances)
        out = np.zeros(pk0.proof_size, dtype=np.uint8)
        ln = ctypes.c_size_t()
        handles = (ctypes.c_void_p * len(pks))(*[p._h for p in pks])
        adv = (ctypes.c_void_p * len(pks))(*[d.ptr for d in d_advice])
        rng = (ctypes.c_void_p * len(pks))(*[d.ptr for d in d_rng_wide])
        self.backends[0]._check(lib().b200zk_group_create_proof_dev(self._h, handles, adv, inst_ptrs, _p(lens), rng, _p(_fr(transcript_repr, 1)),
                                                                    _p(out), ctypes.c_size_t(out.shape[0]), ctypes.byref(ln)))
        return bytes(out[: ln.value])


class ParamsKZG:
    """poly::kzg::commitment::ParamsKZG<Bn256> with the SRS resident in HBM."""

    def __init__(self, backend, handle, k):
        self.backend, self._h, self.k, self.n = backend, handle, k, 1 << k

    @classmethod
    def load(cls, backend, k, g, g_lagrange=None):
        g = np.ascontiguousarray(g, dtype=np.uint64).reshape(1 << k, 8)
        gl = None if g_lagrange is None else np.ascontiguousarray(g_lagrange, dtype=np.uint64).reshape(1 << k, 8)
        h = ctypes.c_void_p()
        backend._check(lib().b200zk_params_load(backend._ctx, ctypes.c_uint32(k), _p(g), _p(gl), ctypes.byref(h)))
        return cls(backend, h, k)

    @classmethod
    def setup(cls, backend, k, s):
        """ParamsKZG::setup(k, rng) with s = Fr::random(rng) drawn by the caller."""
        h = ctypes.c_void_p()
        backend._check(lib().b200zk_params_setup(backend._ctx, ctypes.c_uint32(k), _p(_fr(s, 1)), ctypes.byref(h)))
        return cls(backend, h, k)

    def downsize(self, k):
        """ParamsKZG::downsize(k) as new params: g[..2^k] of these params and its Lagrange basis.  Unlike
        upstream's in-place downsize, these params stay as they are, and so do proving keys built on them."""
        h = ctypes.c_void_p()
        self.backend._check(lib().b200zk_params_downsize(self._h, ctypes.c_uint32(k), ctypes.byref(h)))
        return ParamsKZG(self.backend, h, k)

    def close(self):
        if self._h:
            lib().b200zk_params_destroy(self._h)
            self._h = None

    def read(self, lagrange=True):
        g = np.empty((self.n, 8), dtype=np.uint64)
        gl = np.empty((self.n, 8), dtype=np.uint64) if lagrange else None
        self.backend._check(lib().b200zk_params_read(self._h, _p(g), _p(gl)))
        return g, gl

    def to_bytes(self, g2, s_g2):
        """ParamsKZG::write into memory -> bytes: k | g | g_lagrange (compressed G1) | g2 | s_g2 (compressed G2)."""
        lib().b200zk_params_serialized_size.restype = ctypes.c_size_t
        cap = int(lib().b200zk_params_serialized_size(ctypes.c_uint32(self.k), ctypes.c_int32(1)))
        out = np.zeros(cap, dtype=np.uint8)
        ln = ctypes.c_size_t()
        self.backend._check(lib().b200zk_params_serialize(self._h, _p(np.ascontiguousarray(g2, dtype=np.uint64)), _p(np.ascontiguousarray(s_g2, dtype=np.uint64)),
                                                          _p(out), ctypes.c_size_t(cap), ctypes.byref(ln)))
        return out[: ln.value].tobytes()

    @classmethod
    def from_bytes(cls, backend, data):
        """ParamsKZG::read from memory -> (params, g2, s_g2); raises on a malformed or off-curve encoding."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        h = ctypes.c_void_p()
        g2, s_g2 = np.zeros(16, dtype=np.uint64), np.zeros(16, dtype=np.uint64)
        backend._check(lib().b200zk_params_deserialize(backend._ctx, _p(buf), ctypes.c_size_t(buf.shape[0]), ctypes.byref(h), _p(g2), _p(s_g2)))
        k = int(np.frombuffer(buf[:4].tobytes(), dtype="<u4")[0])
        return cls(backend, h, k), g2, s_g2

    def commit(self, poly):
        poly = _fr(poly)
        out = np.zeros(12, dtype=np.uint64)
        self.backend._check(lib().b200zk_commit(self._h, _p(poly), ctypes.c_size_t(poly.shape[0]), _p(out)))
        return out

    def commit_lagrange(self, poly):
        poly = _fr(poly)
        out = np.zeros(12, dtype=np.uint64)
        self.backend._check(lib().b200zk_commit_lagrange(self._h, _p(poly), ctypes.c_size_t(poly.shape[0]), _p(out)))
        return out

    def commit_many_dev(self, d_polys, n, lagrange):
        """Commitments to several device-resident polynomials of length n (one batched launch sequence)."""
        ptrs = (ctypes.c_void_p * max(len(d_polys), 1))(*[d.ptr for d in d_polys])
        out = np.zeros((len(d_polys), 12), dtype=np.uint64)
        self.backend._check(lib().b200zk_commit_many_dev(self._h, ptrs, ctypes.c_uint32(len(d_polys)), ctypes.c_size_t(n),
                                                         ctypes.c_int32(1 if lagrange else 0), _p(out)))
        return out

    def commit_dev(self, d_poly, n, lagrange):
        out = np.zeros(12, dtype=np.uint64)
        self.backend._check(lib().b200zk_commit_dev(self._h, d_poly.ptr, ctypes.c_size_t(n), ctypes.c_int32(1 if lagrange else 0), _p(out)))
        return out


def g_to_lagrange(backend, g, k):
    """arithmetic::g_to_lagrange(g, k): the Lagrange basis n^-1 * FFT_{w^-1}(g) of n = 2^k G1Affine points,
    as an (n, 8) array."""
    g = np.ascontiguousarray(g, dtype=np.uint64).reshape(-1, 8)
    if g.shape[0] != 1 << k:
        raise B200zkError(f"g_to_lagrange: expected {1 << k} points, got {g.shape[0]}")
    out = np.empty((1 << k, 8), dtype=np.uint64)
    backend._check(lib().b200zk_g_to_lagrange(backend._ctx, _p(g), ctypes.c_uint32(k), _p(out)))
    return out


# ---- verifier side (host only: no Backend, no device) -------------------------------------------
def g2_mul(s, base=None):
    """[s]_2 (ParamsKZG.s_g2 for the setup secret s), or s * base: G2Affine as (16,) Montgomery limbs."""
    out = np.zeros(16, dtype=np.uint64)
    b = None if base is None else np.ascontiguousarray(base, dtype=np.uint64).reshape(16)
    rc = lib().b200zk_g2_mul(_p(b), _p(_fr(s, 1)), _p(out))
    if rc != OK:
        raise B200zkError(f"b200zk_g2_mul: error {rc}")
    return out


def pairing_check(g1_points, g2_points):
    """prod e(P_i, Q_i) == 1 for G1Affine (m, 8) and G2Affine (m, 16) Montgomery limbs."""
    a = np.ascontiguousarray(g1_points, dtype=np.uint64).reshape(-1, 8)
    b = np.ascontiguousarray(g2_points, dtype=np.uint64).reshape(-1, 16)
    if a.shape[0] != b.shape[0]:
        raise B200zkError("pairing_check: length mismatch")
    rc = lib().b200zk_pairing_check(_p(a), _p(b), ctypes.c_size_t(a.shape[0]))
    if rc not in (OK, EVERIFY):
        raise B200zkError(f"b200zk_pairing_check: error {rc}")
    return rc == OK


def pairing_checks(backend, g1_points, g2_points, m):
    """Many pairing-product checks on the device (b200zk_pairing_checks): check j is prod_{i < m} e(P[j m + i], Q[j m + i])
    == 1 over G1Affine (count * m, 8) and G2Affine (count * m, 16) Montgomery limbs.  Returns the int32 status array,
    0 where the product is one and EVERIFY where it is not."""
    a = np.ascontiguousarray(g1_points, dtype=np.uint64).reshape(-1, 8)
    b = np.ascontiguousarray(g2_points, dtype=np.uint64).reshape(-1, 16)
    if m < 1 or a.shape[0] != b.shape[0] or a.shape[0] % m:
        raise B200zkError("pairing_checks: the point counts are not count * m")
    status = np.zeros(a.shape[0] // m, dtype=np.int32)
    rc = lib().b200zk_pairing_checks(backend._ctx, _p(a), _p(b), ctypes.c_uint32(m), ctypes.c_uint32(status.shape[0]), _p(status))
    if rc != EVERIFY:
        backend._check(rc)
    return status


class VerifyingKey:
    """What plonk::verify_proof reads of a VerifyingKey: the constraint system, k, and the commitments to
    the fixed and permutation polynomials (ProvingKey.vk_commitments()); plus the verifier params
    (g1 = params.get_g()[0], g2, s_g2)."""

    def __init__(self, cs, k, fixed_commitments, sigma_commitments, g1, s_g2, g2=None):
        self.cs, self.k = cs, k
        self.blob = np.ascontiguousarray(cs.to_blob(k), dtype=np.uint32)
        self.fixed = np.ascontiguousarray(fixed_commitments, dtype=np.uint64).reshape(-1, 8)
        self.sigma = np.ascontiguousarray(sigma_commitments, dtype=np.uint64).reshape(-1, 8)
        self.g1 = np.ascontiguousarray(g1, dtype=np.uint64).reshape(8)
        self.s_g2 = np.ascontiguousarray(s_g2, dtype=np.uint64).reshape(16)
        self.g2 = g2_mul(np.array(_FR_ONE, dtype=np.uint64)) if g2 is None else np.ascontiguousarray(g2, dtype=np.uint64).reshape(16)
        if self.fixed.shape[0] != cs.num_fixed or self.sigma.shape[0] != len(cs.permutation):
            raise B200zkError("commitment counts do not match the constraint system")

    @property
    def transcript_repr(self):
        """The library-derived vk.transcript_repr (b200zk_vk_transcript_repr): a hash of k, the constraint system and the
        fixed / permutation commitments.  Not upstream's value (a hash of Rust's Debug rendering) — a Rust host passes its own."""
        out = np.zeros(4, dtype=np.uint64)
        fixed = self.fixed if self.fixed.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        sigma = self.sigma if self.sigma.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        rc = lib().b200zk_vk_transcript_repr(_p(self.blob), ctypes.c_size_t(self.blob.shape[0]), _p(fixed), _p(sigma), _p(out))
        if rc != OK:
            raise B200zkError(f"b200zk_vk_transcript_repr: error {rc}")
        return out

    def commitments_to_bytes(self):
        """The commitments part of VerifyingKey::write: fixed count (u32 BE) | fixed | permutation commitments (compressed)."""
        lib().b200zk_vk_serialized_size.restype = ctypes.c_size_t
        nf, ns = self.fixed.shape[0], self.sigma.shape[0]
        out = np.zeros(int(lib().b200zk_vk_serialized_size(ctypes.c_uint32(nf), ctypes.c_uint32(ns))), dtype=np.uint8)
        fixed = self.fixed if nf else np.zeros((1, 8), dtype=np.uint64)
        sigma = self.sigma if ns else np.zeros((1, 8), dtype=np.uint64)
        rc = lib().b200zk_vk_serialize(_p(fixed), ctypes.c_uint32(nf), _p(sigma), ctypes.c_uint32(ns), _p(out), ctypes.c_size_t(out.shape[0]))
        if rc != OK:
            raise B200zkError(f"b200zk_vk_serialize: error {rc}")
        return out.tobytes()

    @staticmethod
    def commitments_from_bytes(data, num_sigma):
        """-> (fixed (F, 8), sigma (P, 8)); raises on an invalid point encoding."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        cap = max((buf.shape[0] - 4) // 32, 1)
        fixed, sigma = np.zeros((cap, 8), dtype=np.uint64), np.zeros((max(num_sigma, 1), 8), dtype=np.uint64)
        nf = ctypes.c_uint32()
        rc = lib().b200zk_vk_deserialize(_p(buf), ctypes.c_size_t(buf.shape[0]), ctypes.c_uint32(num_sigma), _p(fixed), ctypes.c_uint32(cap), ctypes.byref(nf), _p(sigma))
        if rc != OK:
            raise B200zkError(f"b200zk_vk_deserialize: error {rc}")
        return fixed[: nf.value], sigma[:num_sigma]

    def verify_proof(self, instances, proof, transcript_repr=None):
        """plonk::verify_proof(..).is_ok() with VerifierSHPLONK / SingleStrategy / Blake2bRead.  transcript_repr: the value the
        prover absorbed (default: the library-derived one, self.transcript_repr)."""
        if transcript_repr is None:
            transcript_repr = self.transcript_repr
        cols = [np.ascontiguousarray(c, dtype=np.uint64).reshape(-1, 4) for c in instances]
        lens = np.array([c.shape[0] for c in cols] + [0], dtype=np.uint32)
        keep = [c if c.shape[0] else np.zeros((1, 4), dtype=np.uint64) for c in cols]
        buf = np.frombuffer(bytes(proof), dtype=np.uint8)
        fixed = self.fixed if self.fixed.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        sigma = self.sigma if self.sigma.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        rc = lib().b200zk_verify_proof(_p(self.blob), ctypes.c_size_t(self.blob.shape[0]), _p(fixed), _p(sigma), _p(self.g1), _p(self.g2),
                                       _p(self.s_g2), _ptr_array(keep), _p(lens), _p(_fr(transcript_repr, 1)),
                                       _p(buf) if buf.shape[0] else None, ctypes.c_size_t(buf.shape[0]))
        if rc not in (OK, EVERIFY):
            raise B200zkError(f"b200zk_verify_proof: error {rc}")
        return rc == OK

    def verify_proofs(self, backend, instances_list, proofs, transcript_repr=None, rng_wide=None, accumulator=False):
        """verify_proof for many proofs of this key with AccumulatorStrategy: one pairing check for the whole batch, the
        point decompression and the per-proof opening sums on backend's device (b200zk_verify_proofs).  rng_wide: (count, 8)
        uint64, the 512-bit input of each proof's Fr::random; default fresh os.urandom draws (they must be secret).
        Returns a list of bools, and with accumulator=True also (left, right): two (8,) G1Affine Montgomery limb arrays."""
        count = len(proofs)
        if len(instances_list) != count:
            raise B200zkError("one instance list per proof")
        if transcript_repr is None:
            transcript_repr = self.transcript_repr
        if rng_wide is None:
            wide = np.frombuffer(os.urandom(64 * max(count, 1)), dtype=np.uint64).reshape(-1, 8)
        else:
            wide = np.ascontiguousarray(rng_wide, dtype=np.uint64).reshape(-1, 8)
            if wide.shape[0] < count:
                raise B200zkError(f"rng_wide too short: need {count} draws")
        keep, lens = [], []
        for instances in instances_list:
            if len(instances) != len(instances_list[0]):
                raise B200zkError("every proof needs the same number of instance columns")
            cols = [np.ascontiguousarray(c, dtype=np.uint64).reshape(-1, 4) for c in instances]
            lens += [c.shape[0] for c in cols]
            keep += [c if c.shape[0] else np.zeros((1, 4), dtype=np.uint64) for c in cols]
        bufs = [np.frombuffer(bytes(p), dtype=np.uint8) for p in proofs]
        ptrs = (ctypes.c_void_p * max(count, 1))(*[b.ctypes.data if b.shape[0] else None for b in bufs])
        plens = np.array([b.shape[0] for b in bufs] + [0], dtype=np.uint64)
        lens = np.array(lens + [0], dtype=np.uint32)
        fixed = self.fixed if self.fixed.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        sigma = self.sigma if self.sigma.shape[0] else np.zeros((1, 8), dtype=np.uint64)
        status = np.zeros(max(count, 1), dtype=np.int32)
        acc = np.zeros((2, 8), dtype=np.uint64)
        rc = lib().b200zk_verify_proofs(backend._ctx, _p(self.blob), ctypes.c_size_t(self.blob.shape[0]), _p(fixed), _p(sigma), _p(self.g1),
                                        _p(self.g2), _p(self.s_g2), ctypes.c_uint32(count), _ptr_array(keep), _p(lens),
                                        _p(_fr(transcript_repr, 1)), ptrs, _p(plens), _p(wide), _p(status), _p(acc))
        if rc != EVERIFY:
            backend._check(rc)
        ok = [int(s) == OK for s in status[:count]]
        return (ok, (acc[0], acc[1])) if accumulator else ok


_FR_ONE = [0xac96341c4ffffffb, 0x36fc76959f60cd29, 0x666ea36f7879462e, 0x0e0a77c19a07df2f]      # R mod r
