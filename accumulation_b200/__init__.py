"""accumulation_b200 -- B200-native commitment / MSM hot path for arkworks-rs/accumulation.

Python here is only the test/bench harness binding of the C-ABI (include/accmsm.h); the product is
`libaccmsm.so` (hand-written sm_100a CUDA) plus the C++ host mirror in `host/ark_mirror.hpp`.
Names follow the reference (`PedersenCommitment.commit`, `InnerProductArgPC.cm_commit`,
`SuccinctCheckPolynomial.compute_coeffs`, `ASForHadamardProducts.decide`, `matrix_vec_mul`) so parity
tests read like the reference's own.  All arrays are numpy uint64 in the ark-ff / ark-ec memory image:
field element = 4 LE limbs (Montgomery unless stated), affine point = x[4] || y[4] + infinity flag.
There is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from ._lib import AccmsmError, load

PALLAS, VESTA = 0, 1
FP, FQ = 0, 1


def scalar_field(curve: int) -> int:
    return FQ if curve == PALLAS else FP


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pinned_array(shape, dtype=np.uint64) -> np.ndarray:
    """numpy array backed by accmsm_host_alloc (page-locked); kept alive by the array's base object"""
    lib = load()
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = lib.accmsm_host_alloc(C.c_size_t(max(nbytes, 1)))
    if not ptr:
        raise AccmsmError("accmsm_host_alloc failed")

    class _Owner:
        def __init__(self, p):
            self.p = p
            self.buf = (C.c_uint8 * max(nbytes, 1)).from_address(p)

        def __del__(self):
            lib.accmsm_host_free(C.c_void_p(self.p))
    owner = _Owner(ptr)
    arr = np.frombuffer(owner.buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED_OWNERS[arr.ctypes.data] = owner       # freed by release_pinned(arr) (or at interpreter exit)
    return arr


_PINNED_OWNERS = {}


def release_pinned(arr: np.ndarray):
    _PINNED_OWNERS.pop(arr.ctypes.data, None)


class Context:
    """One accmsm_ctx: bound to one GPU (`Context(0)`; one per process under torchrun, SURVEY.md 8e) or to a group of GPUs of
    one box (`Context(devices=[0, 1, ..])`, accmsm_init_multi): the same calls then shard keys by point range inside
    the library."""

    def __init__(self, device: int = 0, devices: Optional[Sequence[int]] = None, min_shard: Optional[int] = None):
        self._lib = load()
        h = C.c_void_p()
        if devices is not None:
            arr = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = self._lib.accmsm_init_multi(C.byref(h), arr, C.c_int(len(devices)))
        else:
            rc = self._lib.accmsm_init(C.byref(h), C.c_int(device))
        if rc != 0:
            raise AccmsmError(f"accmsm_init(device={device if devices is None else list(devices)}) failed: "
                              f"{self._lib.accmsm_strerror(rc).decode()} (a CUDA device is required; there is no CPU path)")
        self._h = h
        self._owned = True
        if min_shard is not None:
            self.set_min_shard(min_shard)

    @classmethod
    def _borrowed(cls, lib, handle):
        c = cls.__new__(cls)
        c._lib, c._h, c._owned = lib, C.c_void_p(handle), False
        return c

    def device_count(self) -> int:
        return int(self._lib.accmsm_device_count(self._h))

    def device_ctx(self, index: int) -> "Context":
        """the single-device ctx of device `index` of a group (for the device-pointer entry points); owned by the group"""
        p = self._lib.accmsm_device_ctx(self._h, C.c_int(index))
        if not p:
            raise AccmsmError(f"device_ctx({index}): out of range")
        return Context._borrowed(self._lib, p)

    def set_min_shard(self, min_points: int):
        self._check(self._lib.accmsm_set_min_shard(self._h, C.c_size_t(min_points)), "set_min_shard")

    def close(self):
        if getattr(self, "_h", None):
            if getattr(self, "_owned", True):
                self._lib.accmsm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- plumbing
    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self._lib.accmsm_last_error(self._h).decode()
            raise AccmsmError(f"{what}: {self._lib.accmsm_strerror(rc).decode()} ({msg})")

    def set_window_bits(self, c: int):
        self._check(self._lib.accmsm_set_window_bits(self._h, C.c_int(c)), "set_window_bits")

    def set_ipa_fold(self, rounds: int = 5, min_log_n: int = 11):
        """IpaPC::open: materialise the folded key every `rounds` rounds while the current key has >= 2^min_log_n
        points (0 = never); results are identical either way."""
        self._check(self._lib.accmsm_set_ipa_fold(self._h, C.c_int(rounds), C.c_int(min_log_n)), "set_ipa_fold")

    def kernel_launches(self) -> int:
        return int(self._lib.accmsm_kernel_launches(self._h))

    def last_timings(self) -> dict:
        buf = (C.c_float * 16)()
        k = self._lib.accmsm_last_timings(self._h, buf, C.c_int(16))
        return {self._lib.accmsm_stage_name(C.c_int(i)).decode(): float(buf[i]) for i in range(k)}

    # ---- keys
    def register_bases(self, curve: int, xy, infinity=None) -> "Bases":
        xy = _u64(xy).reshape(-1, 8)
        inf = None if infinity is None else np.ascontiguousarray(infinity, dtype=np.uint8)
        h = C.c_uint64(0)
        self._check(self._lib.accmsm_register_bases(self._h, C.c_int(curve), _p(xy), _p(inf), C.c_size_t(xy.shape[0]),
                                                    C.byref(h)), "register_bases")
        return Bases(self, curve, int(h.value), xy.shape[0])

    def register_synthetic_bases(self, curve: int, seed: int, n: int, first_index: int = 0) -> "Bases":
        h = C.c_uint64(0)
        self._check(self._lib.accmsm_register_synthetic_bases(self._h, C.c_int(curve), C.c_uint64(seed), C.c_uint64(first_index),
                                                              C.c_size_t(n), C.byref(h)), "register_synthetic_bases")
        return Bases(self, curve, int(h.value), n)

    def register_bases_compressed(self, curve: int, data) -> "Bases":
        """ark-serialize compressed points (n x 33 B, no length prefix) -> registered key, decompressed on the device"""
        buf = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        if buf.size % 33:
            raise ValueError("compressed points are 33 bytes each")
        n = buf.size // 33
        h = C.c_uint64(0)
        self._check(self._lib.accmsm_register_bases_compressed(self._h, C.c_int(curve), _p(buf) if n else None, C.c_size_t(n), C.byref(h)),
                    "register_bases_compressed")
        return Bases(self, curve, int(h.value), n)

    def serialize_bases(self, bases: "Bases", offset: int = 0, n: Optional[int] = None) -> bytes:
        n = bases.n - offset if n is None else n
        out = np.empty(n * 33, dtype=np.uint8)
        self._check(self._lib.accmsm_serialize_bases(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n), _p(out) if n else None),
                    "serialize_bases")
        return out.tobytes()

    def download_bases(self, bases: "Bases", offset: int = 0, n: Optional[int] = None):
        n = bases.n - offset if n is None else n
        out = np.empty((n, 8), dtype=np.uint64)
        self._check(self._lib.accmsm_download_bases(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n), _p(out)),
                    "download_bases")
        return out

    # ---- MSM
    def msm(self, bases: "Bases", scalars, montgomery: bool = True, offset: int = 0, n: Optional[int] = None):
        sc = _u64(scalars).reshape(-1, 4)
        n = sc.shape[0] if n is None else n
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_msm(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n), _p(sc),
                                         C.c_int(int(montgomery)), _p(out), C.byref(inf)), "msm")
        return out, int(inf.value)

    def msm_oneshot(self, curve: int, bases_xy, scalars, montgomery: bool = True, infinity=None):
        """VariableBaseMSM::multi_scalar_mul(&bases, &scalars).into_affine() for bases that are not a registered key"""
        xy, sc = _u64(bases_xy).reshape(-1, 8), _u64(scalars).reshape(-1, 4)
        n = min(xy.shape[0], sc.shape[0])                     # ark-ec truncates to the shorter slice
        inf_in = None if infinity is None else np.ascontiguousarray(infinity, dtype=np.uint8)
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_msm_oneshot(self._h, C.c_int(curve), _p(xy), _p(inf_in), _p(sc), C.c_int(int(montgomery)),
                                                 C.c_size_t(n), _p(out), C.byref(inf)), "msm_oneshot")
        return out, int(inf.value)

    def msm_oneshot_batch(self, curve: int, bases_xy, scalars, montgomery: bool = True, infinity=None):
        """m one-shot MSMs of equal length, each over its own bases, in shared passes: bases_xy (m, n, 8), scalars (m, n, 4),
        infinity (m, n) or None -> (xy (m, 8), inf (m,)).  The succinct-check equations of all inputs of one ipa-pc-as prove."""
        xy, sc = _u64(bases_xy), _u64(scalars)
        if xy.ndim != 3 or sc.ndim != 3 or xy.shape[0] != sc.shape[0]:
            raise ValueError("msm_oneshot_batch: bases (m, n, 8) and scalars (m, n, 4) expected")
        m, n = xy.shape[0], min(xy.shape[1], sc.shape[1])
        xy, sc = np.ascontiguousarray(xy[:, :n]), np.ascontiguousarray(sc[:, :n])
        inf_in = None if infinity is None else np.ascontiguousarray(np.asarray(infinity, dtype=np.uint8).reshape(m, -1)[:, :n])
        out = np.empty((m, 8), dtype=np.uint64)
        inf = np.zeros(m, dtype=np.uint8)
        self._check(self._lib.accmsm_msm_oneshot_batch(self._h, C.c_int(curve), _p(xy), _p(inf_in), _p(sc), C.c_int(int(montgomery)),
                                                       C.c_size_t(n), C.c_size_t(m), _p(out), _p(inf)), "msm_oneshot_batch")
        return out, inf

    def msm_ptr(self, bases: "Bases", host_ptr: int, n: int, montgomery: bool = True, offset: int = 0):
        """Same as msm() for a raw host pointer (e.g. a pinned torch tensor's data_ptr())."""
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_msm(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n),
                                         C.c_void_p(host_ptr), C.c_int(int(montgomery)), _p(out), C.byref(inf)), "msm")
        return out, int(inf.value)

    def msm_batch(self, bases: "Bases", scalars, montgomery: bool = True, offset: int = 0):
        sc = _u64(scalars)
        k, n = sc.shape[0], sc.shape[1]
        out = np.empty((k, 8), dtype=np.uint64)
        inf = np.zeros(k, dtype=np.uint8)
        self._check(self._lib.accmsm_msm_batch(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n),
                                               C.c_size_t(k), _p(sc), C.c_int(int(montgomery)), _p(out), _p(inf)), "msm_batch")
        return out, inf

    def commit(self, bases: "Bases", elems_mont, hiding_index: int = 0, randomizer_mont=None):
        el = _u64(elems_mont).reshape(-1, 4)
        r = None if randomizer_mont is None else _u64(randomizer_mont)
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_commit(self._h, C.c_uint64(bases.handle), C.c_size_t(el.shape[0]), _p(el),
                                            C.c_size_t(hiding_index), _p(r), _p(out), C.byref(inf)), "commit")
        return out, int(inf.value)

    def msm_dev(self, bases: "Bases", d_scalars_ptr: int, n: int, montgomery: bool = True, offset: int = 0, stream: int = 0):
        """MSM of scalars already resident in HBM (device pointer); blocks until the affine result is on the host."""
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_msm_dev(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n),
                                             C.c_void_p(d_scalars_ptr), C.c_int(int(montgomery)), _p(out), C.byref(inf),
                                             C.c_void_p(stream)), "msm_dev")
        return out, int(inf.value)

    def msm_partial_dev(self, bases: "Bases", d_scalars_ptr: int, n: int, d_out_ptr: int, montgomery: bool = True,
                        offset: int = 0, stream: int = 0):
        self._check(self._lib.accmsm_msm_partial_dev(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n),
                                                     C.c_void_p(d_scalars_ptr), C.c_int(int(montgomery)),
                                                     C.c_void_p(d_out_ptr), C.c_void_p(stream)), "msm_partial_dev")

    def msm_partial(self, bases: "Bases", scalars, d_out_ptr: int, montgomery: bool = True, offset: int = 0, n: Optional[int] = None):
        """one GPU's share of a sharded MSM from HOST scalars (numpy array or raw host pointer): the library uploads (large vectors
        pipelined behind the accumulation) and leaves the un-normalised partial in device memory at d_out_ptr"""
        if isinstance(scalars, int):
            ptr = C.c_void_p(scalars)
        else:
            sc = _u64(scalars).reshape(-1, 4)
            n = sc.shape[0] if n is None else n
            ptr = _p(sc)
        self._check(self._lib.accmsm_msm_partial(self._h, C.c_uint64(bases.handle), C.c_size_t(offset), C.c_size_t(n), C.c_size_t(1), ptr,
                                                 C.c_int(int(montgomery)), C.c_size_t(0), None, C.c_void_p(d_out_ptr)), "msm_partial")

    def combine_partials_dev(self, curve: int, d_partials_ptr: int, k: int, stream: int = 0):
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_combine_partials_dev(self._h, C.c_int(curve), C.c_void_p(d_partials_ptr), C.c_size_t(k),
                                                          _p(out), C.byref(inf), C.c_void_p(stream)), "combine_partials_dev")
        return out, int(inf.value)

    def combine_partials_batch_dev(self, curve: int, d_partials_ptr: int, k: int, m: int, stream: int = 0):
        """k x m gathered partials (rank-major) -> [(xy, inf)] * m"""
        out = np.empty((m, 8), dtype=np.uint64)
        inf = np.zeros(m, dtype=np.uint8)
        self._check(self._lib.accmsm_combine_partials_batch_dev(self._h, C.c_int(curve), C.c_void_p(d_partials_ptr), C.c_size_t(k),
                                                                C.c_size_t(m), _p(out), _p(inf), C.c_void_p(stream)),
                    "combine_partials_batch_dev")
        return [(out[j], int(inf[j])) for j in range(m)]

    # ---- IPA decider tail
    def ipa_final_key(self, bases: "Bases", challenges_mont):
        ch = _u64(challenges_mont).reshape(-1, 4)
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_ipa_final_key(self._h, C.c_uint64(bases.handle), _p(ch), C.c_int(ch.shape[0]), _p(out),
                                                   C.byref(inf)), "ipa_final_key")
        return out, int(inf.value)

    def ipa_check_final_key(self, bases: "Bases", challenges_mont, expected_xy, expected_inf: int = 0):
        ch = _u64(challenges_mont).reshape(-1, 4)
        exp = _u64(expected_xy)
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        acc = C.c_int(0)
        self._check(self._lib.accmsm_ipa_check_final_key(self._h, C.c_uint64(bases.handle), _p(ch), C.c_int(ch.shape[0]),
                                                         _p(exp), C.c_uint8(int(expected_inf)), C.byref(acc), _p(out),
                                                         C.byref(inf)), "ipa_check_final_key")
        return bool(acc.value), out, int(inf.value)

    def ipa_final_key_partial_dev(self, bases: "Bases", challenges_mont, coeff_offset: int, n: int, d_out_ptr: int,
                                  stream: int = 0):
        ch = _u64(challenges_mont).reshape(-1, 4)
        self._check(self._lib.accmsm_ipa_final_key_partial_dev(self._h, C.c_uint64(bases.handle), _p(ch), C.c_int(ch.shape[0]),
                                                               C.c_size_t(coeff_offset), C.c_size_t(n), C.c_void_p(d_out_ptr),
                                                               C.c_void_p(stream)), "ipa_final_key_partial_dev")

    # ---- IPA opening session
    def ipa_open_begin(self, bases: "Bases", coeffs_mont, k: int, point_mont, h_prime_xy=None) -> int:
        """h_prime_xy None: follow with ipa_open_use_hiding_generator(session, h_index, xi_0)"""
        cf = _u64(coeffs_mont).reshape(-1, 4)
        sess = C.c_uint64(0)
        hp = None if h_prime_xy is None else _u64(h_prime_xy)
        self._check(self._lib.accmsm_ipa_open_begin(self._h, C.c_uint64(bases.handle), _p(cf), C.c_size_t(cf.shape[0]), C.c_int(k),
                                                    _p(_u64(point_mont)), _p(hp), C.byref(sess)), "ipa_open_begin")
        return int(sess.value)

    def ipa_open_begin_shard(self, bases: "Bases", coeffs_mont, k: int, point_mont, h_prime_xy=None, shard_index: int = 0,
                             log_shards: int = 0, z_scale_mont=None) -> int:
        """session over ONE cyclic shard (indices = shard_index mod 2^log_shards) of a multi-GPU opening; k = log2 of
        the shard length; z-vector = z_scale * point^(shard_index + 2^log_shards i)"""
        cf = _u64(coeffs_mont).reshape(-1, 4)
        sess = C.c_uint64(0)
        hp = None if h_prime_xy is None else _u64(h_prime_xy)
        zs = None if z_scale_mont is None else _u64(z_scale_mont)
        self._check(self._lib.accmsm_ipa_open_begin_shard(self._h, C.c_uint64(bases.handle), _p(cf), C.c_size_t(cf.shape[0]), C.c_int(k),
                                                          _p(_u64(point_mont)), _p(hp), C.c_uint32(shard_index), C.c_uint32(log_shards),
                                                          _p(zs), C.byref(sess)), "ipa_open_begin_shard")
        return int(sess.value)

    def ipa_open_round_partial_dev(self, session: int, d_out_partials_ptr: int):
        """this shard's un-normalised shares of (l, r): 2 x 16 u64 written to device memory (blocking)"""
        self._check(self._lib.accmsm_ipa_open_round_partial_dev(self._h, C.c_uint64(session), C.c_void_p(d_out_partials_ptr)),
                    "ipa_open_round_partial_dev")

    def ipa_open_use_hiding_generator(self, session: int, h_index: int, xi0_mont):
        self._check(self._lib.accmsm_ipa_open_use_hiding_generator(self._h, C.c_uint64(session), C.c_size_t(h_index), _p(_u64(xi0_mont))),
                    "ipa_open_use_hiding_generator")

    def ipa_open_begin_combined(self, bases: "Bases", challenges_mont, alphas_mont, point_mont, h_prime_xy, random_poly_mont=None):
        """-> (session, P(point)) with P = [random poly] + sum_j alpha_j h_j(X) built on the device"""
        ch = _u64(challenges_mont)
        m, k = ch.shape[0], ch.shape[1]
        rp = None if random_poly_mont is None else _u64(random_poly_mont).reshape(-1, 4)
        sess = C.c_uint64(0)
        ev = np.empty(4, dtype=np.uint64)
        hp = None if h_prime_xy is None else _u64(h_prime_xy)
        self._check(self._lib.accmsm_ipa_open_begin_combined(self._h, C.c_uint64(bases.handle), _p(ch), C.c_int(m), C.c_int(k),
                                                             _p(_u64(alphas_mont)), _p(rp), C.c_size_t(0 if rp is None else rp.shape[0]),
                                                             _p(_u64(point_mont)), _p(hp), C.byref(sess), _p(ev)),
                    "ipa_open_begin_combined")
        return int(sess.value), ev

    def ipa_open_hide(self, session: int, hiding_coeffs_mont, s_index: int, hiding_rand_mont):
        """zk opening, before the first round: the random polynomial (shifted on the device to vanish at the point) and its
        commitment cm_commit(key, hiding') + rho * key[s_index] -> (hiding_comm_xy, inf)"""
        hc = _u64(hiding_coeffs_mont).reshape(-1, 4)
        out = np.empty(8, dtype=np.uint64)
        inf = C.c_uint8(0)
        self._check(self._lib.accmsm_ipa_open_hide(self._h, C.c_uint64(session), _p(hc) if hc.shape[0] else None, C.c_size_t(hc.shape[0]),
                                                   C.c_size_t(s_index), _p(_u64(hiding_rand_mont)), _p(out), C.byref(inf)),
                    "ipa_open_hide")
        return out, int(inf.value)

    def ipa_open_hiding_challenge(self, session: int, alpha_mont):
        """zk opening: coeffs += alpha * hiding' on the device (after ipa_open_hide, before the first round)"""
        self._check(self._lib.accmsm_ipa_open_hiding_challenge(self._h, C.c_uint64(session), _p(_u64(alpha_mont))),
                    "ipa_open_hiding_challenge")

    def ipa_open_round(self, session: int):
        l, r = np.empty(8, dtype=np.uint64), np.empty(8, dtype=np.uint64)
        li, ri = C.c_uint8(0), C.c_uint8(0)
        self._check(self._lib.accmsm_ipa_open_round(self._h, C.c_uint64(session), _p(l), C.byref(li), _p(r), C.byref(ri)),
                    "ipa_open_round")
        return (l, int(li.value)), (r, int(ri.value))

    def ipa_open_fold(self, session: int, xi_mont, xi_inv_mont):
        self._check(self._lib.accmsm_ipa_open_fold(self._h, C.c_uint64(session), _p(_u64(xi_mont)), _p(_u64(xi_inv_mont))),
                    "ipa_open_fold")

    def ipa_open_fold_round(self, session: int, xi_mont):
        """fold with xi (its inverse is computed in the library) and run the next round: -> ((l, inf), (r, inf)) or None when
        the opening is folded to length 1"""
        l, r = np.empty(8, dtype=np.uint64), np.empty(8, dtype=np.uint64)
        li, ri, done = C.c_uint8(0), C.c_uint8(0), C.c_int(0)
        self._check(self._lib.accmsm_ipa_open_fold_round(self._h, C.c_uint64(session), _p(_u64(xi_mont)), _p(l), C.byref(li), _p(r),
                                                         C.byref(ri), C.byref(done)), "ipa_open_fold_round")
        return None if done.value else ((l, int(li.value)), (r, int(ri.value)))

    def ipa_open_finish(self, session: int):
        fk, c = np.empty(8, dtype=np.uint64), np.empty(4, dtype=np.uint64)
        self._check(self._lib.accmsm_ipa_open_finish(self._h, C.c_uint64(session), _p(fk), _p(c)), "ipa_open_finish")
        return fk, c

    # ---- fused steps
    def hp_decide(self, bases: "Bases", a, b, expected_xy, expected_inf, hiding_index: int = 0, randomness=None):
        a, b = _u64(a).reshape(-1, 4), _u64(b).reshape(-1, 4)
        n = min(a.shape[0], b.shape[0])
        exp = _u64(expected_xy).reshape(3, 8)
        einf = np.ascontiguousarray(expected_inf, dtype=np.uint8).reshape(3)
        r = None if randomness is None else _u64(randomness).reshape(3, 4)
        out = np.empty((3, 8), dtype=np.uint64)
        oinf = np.zeros(3, dtype=np.uint8)
        acc = C.c_int(0)
        self._check(self._lib.accmsm_hp_decide(self._h, C.c_uint64(bases.handle), _p(a), _p(b), C.c_size_t(n), C.c_size_t(hiding_index),
                                               _p(r), _p(exp), _p(einf), C.byref(acc), _p(out), _p(oinf)), "hp_decide")
        return bool(acc.value), out, oinf

    def hp_product_poly_comm(self, bases: "Bases", a_vecs, b_vecs, mu, length: int, hiding_a=None, hiding_b=None, want_tvecs=False):
        a_vecs = [_u64(v).reshape(-1, 4) for v in a_vecs]
        b_vecs = [_u64(v).reshape(-1, 4) for v in b_vecs]
        n = len(a_vecs)
        al = np.array([v.shape[0] for v in a_vecs], dtype=np.uint64)
        bl = np.array([v.shape[0] for v in b_vecs], dtype=np.uint64)
        ha = None if hiding_a is None else _u64(hiding_a).reshape(-1, 4)
        hb = None if hiding_b is None else _u64(hiding_b).reshape(-1, 4)
        low, high = np.empty((max(n - 1, 0), 8), dtype=np.uint64), np.empty((max(n - 1, 0), 8), dtype=np.uint64)
        linf, hinf = np.zeros(max(n - 1, 0), dtype=np.uint8), np.zeros(max(n - 1, 0), dtype=np.uint8)
        tv = np.empty((2 * n - 1, length, 4), dtype=np.uint64) if want_tvecs else None
        self._check(self._lib.accmsm_hp_product_poly_comm(self._h, C.c_uint64(bases.handle), self._ptrs(a_vecs), _p(al), self._ptrs(b_vecs),
                                                          _p(bl), C.c_int(n), _p(_u64(mu)), C.c_size_t(length), _p(ha),
                                                          C.c_size_t(0 if ha is None else ha.shape[0]), _p(hb),
                                                          C.c_size_t(0 if hb is None else hb.shape[0]), _p(low), _p(linf), _p(high),
                                                          _p(hinf), _p(tv)), "hp_product_poly_comm")
        return (low, linf), (high, hinf), tv

    def register_csr(self, field: int, mats) -> int:
        rps = [np.ascontiguousarray(m[0], dtype=np.uint32) for m in mats]
        cls = [np.ascontiguousarray(m[1], dtype=np.uint32) for m in mats]
        cfs = [_u64(m[2]).reshape(-1, 4) for m in mats]
        h = C.c_uint64(0)
        self._check(self._lib.accmsm_register_csr(self._h, C.c_int(field), C.c_int(len(mats)), self._ptrs(rps), self._ptrs(cls),
                                                  self._ptrs(cfs), C.c_size_t(rps[0].size - 1), C.byref(h)), "register_csr")
        return int(h.value)

    def release_csr(self, handle: int):
        self._check(self._lib.accmsm_release_csr(self._h, C.c_uint64(handle)), "release_csr")

    def csr_matvec_commit(self, bases: "Bases", csr: int, n_mats: int, n_rows: int, inp, wit, hiding_index: int = 0, blinders=None,
                          want_vecs: bool = True):
        inp, wit = _u64(inp).reshape(-1, 4), _u64(wit).reshape(-1, 4)
        bl = None if blinders is None else _u64(blinders).reshape(n_mats, 4)
        vecs = [np.empty((n_rows, 4), dtype=np.uint64) for _ in range(n_mats)] if want_vecs else None
        out = np.empty((n_mats, 8), dtype=np.uint64)
        oinf = np.zeros(n_mats, dtype=np.uint8)
        self._check(self._lib.accmsm_csr_matvec_commit(self._h, C.c_uint64(bases.handle), C.c_uint64(csr), _p(inp), C.c_size_t(inp.shape[0]),
                                                       _p(wit), C.c_size_t(wit.shape[0]), C.c_size_t(hiding_index), _p(bl),
                                                       None if vecs is None else self._ptrs(vecs), _p(out), _p(oinf)), "csr_matvec_commit")
        return vecs, out, oinf

    def nark_prove_zk(self, bases: "Bases", csr: int, n_rows: int, inp, wit, r, blinders, hiding_index: int = 0, want_vecs: bool = True):
        """zk R1CSNark::prove first message: z_M, r_M, cross, rr and their 8 commitments (blinders: 8 x 4 in the order
        A, B, C, rA, rB, rC, 1, 2) in one vector launch and one pass -> (vecs | None, xy (8, 8), inf (8,))"""
        inp, wit, r = _u64(inp).reshape(-1, 4), _u64(wit).reshape(-1, 4), _u64(r).reshape(-1, 4)
        bl = _u64(blinders).reshape(8, 4)
        vecs = [np.empty((n_rows, 4), dtype=np.uint64) for _ in range(8)] if want_vecs else None
        out = np.empty((8, 8), dtype=np.uint64)
        oinf = np.zeros(8, dtype=np.uint8)
        self._check(self._lib.accmsm_nark_prove_zk(self._h, C.c_uint64(bases.handle), C.c_uint64(csr), _p(inp), C.c_size_t(inp.shape[0]),
                                                   _p(wit), C.c_size_t(wit.shape[0]), _p(r), C.c_size_t(hiding_index), _p(bl),
                                                   None if vecs is None else self._ptrs(vecs), _p(out), _p(oinf)), "nark_prove_zk")
        return vecs, out, oinf

    def nark_verify(self, bases: "Bases", csr: int, n_rows: int, inp, blinded_wit, expected_xy, expected_inf, hiding_index: int = 0,
                    sigmas=None, want_vecs: bool = False):
        """R1CSNark::verify: t_M = M (input || w'), Commit(t_M, sigma_M) and Commit(t_A o t_B, sigma_o) in one vector launch and
        one pass, compared with the 4 expected points -> (accept, [t_A, t_B, t_C] | None, xy (4, 8), inf (4,))"""
        inp, wit = _u64(inp).reshape(-1, 4), _u64(blinded_wit).reshape(-1, 4)
        exp = _u64(expected_xy).reshape(4, 8)
        einf = np.ascontiguousarray(expected_inf, dtype=np.uint8).reshape(4)
        sg = None if sigmas is None else _u64(sigmas).reshape(4, 4)
        vecs = [np.empty((n_rows, 4), dtype=np.uint64) for _ in range(3)] if want_vecs else None
        out = np.empty((4, 8), dtype=np.uint64)
        oinf = np.zeros(4, dtype=np.uint8)
        acc = C.c_int(0)
        self._check(self._lib.accmsm_nark_verify(self._h, C.c_uint64(bases.handle), C.c_uint64(csr), _p(inp), C.c_size_t(inp.shape[0]),
                                                 _p(wit), C.c_size_t(wit.shape[0]), C.c_size_t(hiding_index), _p(sg), _p(exp), _p(einf),
                                                 C.byref(acc), _p(out), _p(oinf), None if vecs is None else self._ptrs(vecs)), "nark_verify")
        return bool(acc.value), vecs, out, oinf

    def nark_as_decide(self, bases: "Bases", csr: int, inp, wit, hp_a, hp_b, expected_xy, expected_inf, hiding_index: int = 0,
                       sigmas=None, hp_randomness=None):
        """ASForR1CSNark::decide: t_M = M (input || w*), Commit(t_M, sigma_M*), Commit(a*, r1*), Commit(b*, r2*) and
        Commit(a* o b*, r3*) in one vector launch and one 6-job pass, compared with the 6 expected points (comm_A*, comm_B*,
        comm_C*, C1*, C2*, C3*) -> (accept, xy (6, 8), inf (6,))"""
        inp, wit = _u64(inp).reshape(-1, 4), _u64(wit).reshape(-1, 4)
        a, b = _u64(hp_a).reshape(-1, 4), _u64(hp_b).reshape(-1, 4)
        exp = _u64(expected_xy).reshape(6, 8)
        einf = np.ascontiguousarray(expected_inf, dtype=np.uint8).reshape(6)
        sg = None if sigmas is None else _u64(sigmas).reshape(3, 4)
        hr = None if hp_randomness is None else _u64(hp_randomness).reshape(3, 4)
        out = np.empty((6, 8), dtype=np.uint64)
        oinf = np.zeros(6, dtype=np.uint8)
        acc = C.c_int(0)
        self._check(self._lib.accmsm_nark_as_decide(self._h, C.c_uint64(bases.handle), C.c_uint64(csr), _p(inp), C.c_size_t(inp.shape[0]),
                                                    _p(wit), C.c_size_t(wit.shape[0]), _p(a), C.c_size_t(a.shape[0]), _p(b),
                                                    C.c_size_t(b.shape[0]), C.c_size_t(hiding_index), _p(sg), _p(hr), _p(exp), _p(einf),
                                                    C.byref(acc), _p(out), _p(oinf)), "nark_as_decide")
        return bool(acc.value), out, oinf

    def hp_prove_begin(self, bases: "Bases", a_vecs, b_vecs, length: int, hiding_a=None, hiding_b=None, hiding_index: int = 0,
                       hiding_rand=None):
        """ASForHadamardProducts::prove, first step: the n pairs (a_i, b_i) go to HBM once and stay there until
        hp_prove_finish.  With hiding (ha, hb of `length` elements, hiding_rand = (r1, r2, r3)) the three hiding commitments
        Commit(ha, r1), Commit(hb, r2), Commit(ha o b_0 + a_{n-1} o hb, r3) come from one pass -> (session, (xy (3, 8),
        inf (3,)) | None)"""
        a_vecs = [_u64(v).reshape(-1, 4) for v in a_vecs]
        b_vecs = [_u64(v).reshape(-1, 4) for v in b_vecs]
        n = len(a_vecs)
        al = np.array([v.shape[0] for v in a_vecs], dtype=np.uint64)
        bl = np.array([v.shape[0] for v in b_vecs], dtype=np.uint64)
        ha = None if hiding_a is None else _u64(hiding_a).reshape(-1, 4)
        hb = None if hiding_b is None else _u64(hiding_b).reshape(-1, 4)
        hr = None if hiding_rand is None else _u64(hiding_rand).reshape(3, 4)
        out, oinf = np.zeros((3, 8), dtype=np.uint64), np.zeros(3, dtype=np.uint8)
        sess = C.c_uint64(0)
        self._check(self._lib.accmsm_hp_prove_begin(self._h, C.c_uint64(bases.handle), self._ptrs(a_vecs), _p(al), self._ptrs(b_vecs),
                                                    _p(bl), C.c_int(n), C.c_size_t(length), _p(ha), _p(hb), C.c_size_t(hiding_index),
                                                    _p(hr), _p(out), _p(oinf), C.byref(sess)), "hp_prove_begin")
        return int(sess.value), (None if ha is None else (out, oinf))

    def hp_prove_product_poly_comm(self, session: int, n: int, mu):
        """second step: t-vectors of the resident pairs and their 2n - 2 commitments; mu has n entries (n + 1 with hiding:
        mu_n = mu_1 mu_{n-1}) -> ((low xy (n-1, 8), inf), (high xy (n-1, 8), inf))"""
        mu = _u64(mu).reshape(-1, 4)
        low, high = np.empty((max(n - 1, 0), 8), dtype=np.uint64), np.empty((max(n - 1, 0), 8), dtype=np.uint64)
        linf, hinf = np.zeros(max(n - 1, 0), dtype=np.uint8), np.zeros(max(n - 1, 0), dtype=np.uint8)
        self._check(self._lib.accmsm_hp_prove_product_poly_comm(self._h, C.c_uint64(session), _p(mu), C.c_size_t(mu.shape[0]), _p(low),
                                                                _p(linf), _p(high), _p(hinf)), "hp_prove_product_poly_comm")
        return (low, linf), (high, hinf)

    def hp_prove_finish(self, session: int, nu, capacity: int):
        """last step: a* = mu_n ha + sum_i mu_i nu^i a_i, b* = mu_1 hb + sum_j nu^j b_{n-1-j}; releases the session (on error
        too) -> (a*, b*)"""
        a, b = np.empty((capacity, 4), dtype=np.uint64), np.empty((capacity, 4), dtype=np.uint64)
        olen = (C.c_size_t * 2)()
        self._check(self._lib.accmsm_hp_prove_finish(self._h, C.c_uint64(session), _p(_u64(nu)), _p(a), _p(b), C.c_size_t(capacity), olen),
                    "hp_prove_finish")
        return a[: olen[0]], b[: olen[1]]

    def hp_prove_abort(self, session: int):
        self._check(self._lib.accmsm_hp_prove_abort(self._h, C.c_uint64(session)), "hp_prove_abort")

    def nark_as_prove_begin(self, bases: "Bases", csr: int, inputs, blinded_witnesses, acc_witnesses, acc_a, acc_b, zk=None,
                            hiding_index: int = 0, n_input: Optional[int] = None):
        """ASForR1CSNark::prove, first step (SURVEY App. C.12): an hp_prove session whose first pairs are A (x_i || w'_i),
        B (x_i || w'_i) of the fresh inputs (one row-kernel launch), then the accumulators' (a*_j, b*_j).  zk = (r_x, r_w, ha, hb,
        rand) with rand = (sigma_rA, sigma_rB, sigma_rC, r1, r2, r3): the same launch forms M (r_x || r_w) and one 6-job pass
        returns H1, H2, H3, comm_rA, comm_rB, comm_rC.  Continue with hp_prove_product_poly_comm and nark_as_prove_finish
        n_input: the index's input length, needed (for the column check) when there is neither a fresh input nor zk
        -> (session, (xy (6, 8), inf (6,)) | None)"""
        xs = [_u64(v).reshape(-1, 4) for v in inputs]
        ws = [_u64(v).reshape(-1, 4) for v in blinded_witnesses]
        aw = [_u64(v).reshape(-1, 4) for v in acc_witnesses]
        aa = [_u64(v).reshape(-1, 4) for v in acc_a]
        bb = [_u64(v).reshape(-1, 4) for v in acc_b]
        if n_input is None:
            n_input = xs[0].shape[0] if xs else (_u64(zk[0]).reshape(-1, 4).shape[0] if zk is not None else 0)
        n_witness = ws[0].shape[0] if ws else (aw[0].shape[0] if aw else 0)
        al = np.array([v.shape[0] for v in aa] or [0], dtype=np.uint64)
        bl = np.array([v.shape[0] for v in bb] or [0], dtype=np.uint64)
        rx, rw, ha, hb, rand = (None,) * 5 if zk is None else (_u64(zk[0]).reshape(-1, 4), _u64(zk[1]).reshape(-1, 4), _u64(zk[2]).reshape(-1, 4),
                                                            _u64(zk[3]).reshape(-1, 4), _u64(zk[4]).reshape(6, 4))
        out, oinf = np.zeros((6, 8), dtype=np.uint64), np.zeros(6, dtype=np.uint8)
        sess = C.c_uint64(0)
        self._check(self._lib.accmsm_nark_as_prove_begin(
            self._h, C.c_uint64(bases.handle), C.c_uint64(csr), C.c_int(len(xs)), self._ptrs(xs), C.c_size_t(n_input), self._ptrs(ws),
            C.c_size_t(n_witness), C.c_int(len(aa)), self._ptrs(aw), self._ptrs(aa), _p(al), self._ptrs(bb), _p(bl), _p(rx), _p(rw), _p(ha),
            _p(hb), C.c_size_t(hiding_index), _p(rand), _p(out), _p(oinf), C.byref(sess)), "nark_as_prove_begin")
        return int(sess.value), (None if zk is None else (out, oinf))

    def nark_as_prove_finish(self, session: int, nu, beta, capacity: int, n_witness: int):
        """last step: a*, b* as hp_prove_finish and w* = sum_k beta_k w_k (w'_i, then w*_j, then r_w with zk; beta_0 = 1
        included); releases the session (on error too) -> (a*, b*, w*)"""
        beta = _u64(beta).reshape(-1, 4)
        a, b = np.empty((capacity, 4), dtype=np.uint64), np.empty((capacity, 4), dtype=np.uint64)
        w = np.empty((n_witness, 4), dtype=np.uint64)
        olen = (C.c_size_t * 2)()
        self._check(self._lib.accmsm_nark_as_prove_finish(self._h, C.c_uint64(session), _p(_u64(nu)), _p(beta), C.c_size_t(beta.shape[0]),
                                                          _p(a), _p(b), C.c_size_t(capacity), olen, _p(w)), "nark_as_prove_finish")
        return a[: olen[0]], b[: olen[1]], w

    # ---- field-vector kernels
    def compute_coeffs(self, field: int, challenges_mont):
        ch = _u64(challenges_mont).reshape(-1, 4)
        out = np.empty((1 << ch.shape[0], 4), dtype=np.uint64)
        self._check(self._lib.accmsm_compute_coeffs(self._h, C.c_int(field), _p(ch), C.c_int(ch.shape[0]), _p(out)), "compute_coeffs")
        return out

    def combine_check_polys(self, field: int, challenges_mont, alphas_mont, random_poly_mont=None):
        ch = _u64(challenges_mont)
        m, k = ch.shape[0], ch.shape[1]
        al = _u64(alphas_mont)
        rp = None if random_poly_mont is None else _u64(random_poly_mont).reshape(-1, 4)
        out = np.empty((1 << k, 4), dtype=np.uint64)
        self._check(self._lib.accmsm_combine_check_polys(self._h, C.c_int(field), _p(ch), C.c_int(m), C.c_int(k), _p(al), _p(rp),
                                                         C.c_size_t(0 if rp is None else rp.shape[0]), _p(out)), "combine_check_polys")
        return out

    def poly_evaluate(self, field: int, coeffs_mont, point_mont):
        cf = _u64(coeffs_mont).reshape(-1, 4)
        z = _u64(point_mont)
        out = np.empty(4, dtype=np.uint64)
        self._check(self._lib.accmsm_poly_evaluate(self._h, C.c_int(field), _p(cf), C.c_size_t(cf.shape[0]), _p(z), _p(out)), "poly_evaluate")
        return out

    def hadamard(self, field: int, a, b):
        a, b = _u64(a).reshape(-1, 4), _u64(b).reshape(-1, 4)
        n = min(a.shape[0], b.shape[0])
        out = np.empty((n, 4), dtype=np.uint64)
        self._check(self._lib.accmsm_vec_hadamard(self._h, C.c_int(field), _p(a), _p(b), C.c_size_t(n), _p(out)), "vec_hadamard")
        return out

    def scale(self, field: int, v, coeff):
        v, c = _u64(v).reshape(-1, 4), _u64(coeff)
        out = np.empty_like(v)
        self._check(self._lib.accmsm_vec_scale(self._h, C.c_int(field), _p(v), C.c_size_t(v.shape[0]), _p(c), _p(out)), "vec_scale")
        return out

    @staticmethod
    def _ptrs(vecs):
        arr = (C.c_void_p * max(len(vecs), 1))()
        for i, v in enumerate(vecs):
            arr[i] = v.ctypes.data if v.size else None
        return arr

    def lincomb(self, field: int, vecs: Sequence, challenges, hiding=None):
        vecs = [_u64(v).reshape(-1, 4) for v in vecs]
        lens = np.array([v.shape[0] for v in vecs], dtype=np.uint64)
        ch = _u64(challenges)
        hid = None if hiding is None else _u64(hiding).reshape(-1, 4)
        cap = max([int(x) for x in lens] + [0 if hid is None else hid.shape[0]])
        out = np.empty((cap, 4), dtype=np.uint64)
        olen = C.c_size_t(0)
        self._check(self._lib.accmsm_vec_lincomb(self._h, C.c_int(field), self._ptrs(vecs), _p(lens), C.c_int(len(vecs)), _p(ch),
                                                 _p(hid), C.c_size_t(0 if hid is None else hid.shape[0]), _p(out),
                                                 C.c_size_t(cap), C.byref(olen)), "vec_lincomb")
        return out[: olen.value]

    def tvecs(self, field: int, a_vecs, b_vecs, mu, length: int, hiding_a=None, hiding_b=None):
        a_vecs = [_u64(v).reshape(-1, 4) for v in a_vecs]
        b_vecs = [_u64(v).reshape(-1, 4) for v in b_vecs]
        n = len(a_vecs)
        al = np.array([v.shape[0] for v in a_vecs], dtype=np.uint64)
        bl = np.array([v.shape[0] for v in b_vecs], dtype=np.uint64)
        mu = _u64(mu)
        ha = None if hiding_a is None else _u64(hiding_a).reshape(-1, 4)
        hb = None if hiding_b is None else _u64(hiding_b).reshape(-1, 4)
        out = np.empty((2 * n - 1, length, 4), dtype=np.uint64)
        self._check(self._lib.accmsm_vec_tvecs(self._h, C.c_int(field), self._ptrs(a_vecs), _p(al), self._ptrs(b_vecs), _p(bl),
                                               C.c_int(n), _p(mu), C.c_size_t(length), _p(ha),
                                               C.c_size_t(0 if ha is None else ha.shape[0]), _p(hb),
                                               C.c_size_t(0 if hb is None else hb.shape[0]), _p(out)), "vec_tvecs")
        return out

    def csr_matvec(self, field: int, mats, inp, wit):
        """mats: list of (row_ptr u32, cols u32, coeffs_mont u64) sharing z = input || witness."""
        rps = [np.ascontiguousarray(m[0], dtype=np.uint32) for m in mats]
        cls = [np.ascontiguousarray(m[1], dtype=np.uint32) for m in mats]
        cfs = [_u64(m[2]).reshape(-1, 4) for m in mats]
        n_rows = rps[0].size - 1
        inp, wit = _u64(inp).reshape(-1, 4), _u64(wit).reshape(-1, 4)
        outs = [np.empty((n_rows, 4), dtype=np.uint64) for _ in mats]
        self._check(self._lib.accmsm_csr_matvec(self._h, C.c_int(field), C.c_int(len(mats)), self._ptrs(rps), self._ptrs(cls),
                                                self._ptrs(cfs), C.c_size_t(n_rows), _p(inp), C.c_size_t(inp.shape[0]), _p(wit),
                                                C.c_size_t(wit.shape[0]), self._ptrs(outs)), "csr_matvec")
        return outs


@dataclass
class Bases:
    """A commitment key resident in HBM (ipa_pc::CommitterKey.comm_key / trivial_pc::CommitterKey.generators)."""
    ctx: Context
    curve: int
    handle: int
    n: int

    def precompute(self, window_bits: int = 0) -> "Bases":
        """build the window table (accmsm_precompute_bases); later MSMs on this key use a single bucket set"""
        self.ctx._check(self.ctx._lib.accmsm_precompute_bases(self.ctx._h, C.c_uint64(self.handle), C.c_int(window_bits)),
                        "precompute_bases")
        return self

    def release(self):
        if self.handle:
            self.ctx._check(self.ctx._lib.accmsm_release_bases(self.ctx._h, C.c_uint64(self.handle)), "release_bases")
            self.handle = 0


from .mirror import (  # noqa: E402
    AccumulatorInstance, AccumulatorWitness, ASForHadamardProducts, ASForR1CSNark, CommitterKey, InnerProductArgPC, NarkProof, PedersenCommitment,
    R1CSNark, SuccinctCheckPolynomial, ZkHiding, matrix_vec_mul,
)

__all__ = ["Context", "Bases", "pinned_array", "release_pinned", "AccmsmError", "PALLAS", "VESTA", "FP", "FQ", "scalar_field", "PedersenCommitment",
           "CommitterKey", "InnerProductArgPC", "SuccinctCheckPolynomial", "ZkHiding", "ASForHadamardProducts", "R1CSNark", "NarkProof", "ASForR1CSNark",
           "AccumulatorInstance", "AccumulatorWitness", "matrix_vec_mul"]
