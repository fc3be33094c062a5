"""ctypes mirror of include/curdle_b200.h.  Buffers are raw bytes in gnark's
memory layout (see the header); no arithmetic happens on this side."""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "..", "include", "curdle_b200.h")

FP_BYTES = 48
FR_BYTES = 32
G1_AFFINE_BYTES = 96
G1_JAC_BYTES = 144


class CdlError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"curdle_b200 error {code}: {msg}")
        self.code = code
        self.msg = msg


def lib_path() -> str:
    # CDL_LIB: an alternative build of the same library (A/B experiments of kernel variants)
    return os.environ.get("CDL_LIB") or os.path.join(HERE, "libcurdle_b200.so")


def declared_symbols():
    """Every function the public header declares."""
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(cdl_[a-z0-9_]+)\s*\(", txt)))


_LIB = None


def load_library():
    """dlopen libcurdle_b200.so; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not os.path.exists(p):
        raise RuntimeError(
            f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(p)
    vp, sz, i32, u32p = C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_uint32)
    lib.cdl_abi_version.restype = C.c_uint32
    lib.cdl_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.cdl_create_devices.argtypes = [C.POINTER(C.c_int32), sz, C.POINTER(vp)]
    lib.cdl_context_devices.argtypes = [vp, C.POINTER(C.c_int32), sz, C.POINTER(sz)]
    lib.cdl_destroy.argtypes = [vp]
    lib.cdl_destroy.restype = None
    lib.cdl_last_error.argtypes = [vp]
    lib.cdl_last_error.restype = C.c_char_p
    lib.cdl_device_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.c_char_p, sz]
    lib.cdl_g1_msm.argtypes = [vp, vp, vp, sz, vp]
    lib.cdl_g1_msm_batch.argtypes = [vp, vp, vp, u32p, sz, vp]
    lib.cdl_g1_msm_batch_device.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp, vp]
    lib.cdl_g1_scalar_mul_affine.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.cdl_g1_fold.argtypes = [vp, vp, vp, vp, sz]
    lib.cdl_g1_batch_scalar_mul_base.argtypes = [vp, vp, vp, sz, vp, vp]
    lib.cdl_g1_batch_to_affine.argtypes = [vp, vp, sz, vp]
    lib.cdl_g1_sum_affine.argtypes = [vp, vp, sz, vp]
    lib.cdl_g1_compress.argtypes = [vp, vp, sz, vp]
    lib.cdl_g1_decompress.argtypes = [vp, vp, sz, vp, vp]
    lib.cdl_fp_mul.argtypes = [vp, vp, vp, sz, vp]
    lib.cdl_int_peak.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.cdl_int_peak_cfg.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    u64, i32p = C.c_uint64, C.POINTER(C.c_int32)
    lib.cdl_rand_new.argtypes = [u64, C.POINTER(vp)]
    lib.cdl_rand_free.argtypes = [vp]
    lib.cdl_rand_free.restype = None
    lib.cdl_rand_get_frs.argtypes = [vp, sz, vp]
    lib.cdl_rand_get_g1_affines.argtypes = [vp, vp, sz, vp]
    lib.cdl_rand_generate_permutation.argtypes = [vp, sz, u32p]
    lib.cdl_crs_generate.argtypes = [vp, sz, vp, C.POINTER(vp)]
    lib.cdl_crs_from_points.argtypes = [vp, sz, vp, C.POINTER(vp)]
    lib.cdl_crs_export.argtypes = [vp, vp, vp]
    lib.cdl_crs_ell.argtypes = [vp]
    lib.cdl_crs_ell.restype = sz
    lib.cdl_crs_free.argtypes = [vp]
    lib.cdl_crs_free.restype = None
    lib.cdl_shuffle_permute_commit.argtypes = [vp, vp, vp, vp, u32p, vp, vp, vp, vp, vp, vp]
    lib.cdl_prove.argtypes = [vp, vp, vp, vp, vp, vp, vp, u32p, vp, vp, vp, vp, sz, C.POINTER(sz)]
    lib.cdl_verify.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, vp, vp, i32p]
    szp = C.POINTER(sz)
    lib.cdl_shuffle_permute_commit_batch.argtypes = [vp, vp, sz, vp, vp, u32p, vp, C.POINTER(vp), vp, vp, vp, vp, i32p]
    lib.cdl_prove_batch.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp, u32p, vp, vp, C.POINTER(vp), vp, sz, szp, i32p]
    lib.cdl_verify_batch.argtypes = [vp, vp, sz, vp, sz, szp, vp, vp, vp, vp, vp, C.POINTER(vp), i32p, i32p]
    lib.cdl_whisk_generate_shuffle_proof.argtypes = [vp, vp, vp, vp, vp, vp, sz]
    lib.cdl_whisk_is_valid_shuffle_proof.argtypes = [vp, vp, vp, vp, sz, sz, vp, sz, vp, i32p]
    lib.cdl_whisk_generate_shuffle_proof_batch.argtypes = [vp, vp, sz, vp, C.POINTER(vp), vp, vp, sz, i32p]
    lib.cdl_whisk_is_valid_shuffle_proof_batch.argtypes = [vp, vp, sz, vp, vp, vp, sz, C.POINTER(vp), i32p, i32p]
    lib.cdl_whisk_generate_tracker_proof_batch.argtypes = [vp, sz, vp, vp, C.POINTER(vp), vp, i32p]
    lib.cdl_whisk_is_valid_tracker_proof_batch.argtypes = [vp, sz, vp, vp, vp, i32p, i32p]
    lib.cdl_whisk_generate_registration_batch.argtypes = [vp, sz, vp, C.POINTER(vp), vp, vp, vp, i32p]
    lib.cdl_whisk_match_trackers.argtypes = [vp, sz, vp, sz, vp, i32p, i32p]
    lib.cdl_host_selftest.argtypes = [vp, vp, vp, vp]
    lib.cdl_host_selftest_fibers.argtypes = [C.c_uint32, C.c_uint32, vp, C.POINTER(C.c_int32)]
    lib.cdl_engine_stats.argtypes = [vp, vp, vp, vp, vp, C.c_int]
    lib.cdl_engine_busy_ms.argtypes = [vp, C.POINTER(C.c_double)]
    lib.cdl_engine_busy_ms_device.argtypes = [vp, sz, C.POINTER(C.c_double)]
    lib.cdl_set_lanes.argtypes = [vp, i32]
    lib.cdl_launch_count.argtypes = [vp]
    lib.cdl_launch_count.restype = u64
    f32p = C.POINTER(C.c_float)
    lib.cdl_dev_alloc.argtypes = [vp, sz, C.POINTER(vp)]
    lib.cdl_dev_free.argtypes = [vp, vp]
    lib.cdl_dev_upload.argtypes = [vp, vp, vp, sz]
    lib.cdl_dev_download.argtypes = [vp, vp, vp, sz]
    lib.cdl_g1_scalar_mul_affine_device.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.cdl_g1_fold_device.argtypes = [vp, vp, vp, vp, sz]
    lib.cdl_g1_msm_device.argtypes = [vp, vp, vp, sz, C.c_uint32, C.c_uint32, i32, vp, f32p]
    lib.cdl_set_msm_window.argtypes = [vp, i32]
    lib.cdl_set_msm_batch_affine.argtypes = [vp, i32]
    lib.cdl_set_fixed_base_min_batch.argtypes = [vp, i32]
    lib.cdl_set_batch_verify_min.argtypes = [vp, i32]
    lib.cdl_comm_unique_id.argtypes = [vp]
    lib.cdl_comm_init.argtypes = [vp, vp, i32, i32]
    lib.cdl_comm_destroy.argtypes = [vp]
    lib.cdl_comm_partition.argtypes = [sz, i32, i32, i32, i32p, i32p, i32p, i32p]
    lib.cdl_comm_partition.restype = None
    lib.cdl_g1_msm_sharded_device.argtypes = [vp, vp, vp, sz, vp, f32p]
    lib.cdl_g1_msm_sharded.argtypes = [vp, vp, vp, sz, vp]
    no_status = ("cdl_comm_partition", "cdl_destroy", "cdl_last_error", "cdl_abi_version", "cdl_rand_free", "cdl_crs_free", "cdl_crs_ell",
                 "cdl_launch_count")
    for name in declared_symbols():
        fn = getattr(lib, name)  # AttributeError if the build lost a symbol
        if name not in no_status:
            fn.restype = i32
    _LIB = lib
    return lib


class Context:
    """One CUDA device, or with `devices` a list of them whose batched calls are split over the GPUs
    (cdl_create_devices); mirrors cdl_ctx."""

    def __init__(self, device: int = 0, devices=None):
        self.lib = load_library()
        h = C.c_void_p()
        if devices is None:
            rc = self.lib.cdl_create(device, C.byref(h))
        else:
            devs = list(devices)
            rc = self.lib.cdl_create_devices((C.c_int32 * max(1, len(devs)))(*devs), len(devs), C.byref(h))
        if rc != 0:
            raise CdlError(rc, "cdl_create failed (no CUDA device? this library has no CPU fallback)")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.cdl_destroy(self.h)
            self.h = None

    __del__ = close

    def _chk(self, rc: int):
        if rc != 0:
            raise CdlError(rc, (self.lib.cdl_last_error(self.h) or b"").decode())

    def device_info(self):
        sm, khz = C.c_int32(), C.c_int32()
        name = C.create_string_buffer(128)
        self._chk(self.lib.cdl_device_info(self.h, C.byref(sm), C.byref(khz), name, 128))
        return {"sm_count": sm.value, "clock_khz": khz.value, "name": name.value.decode()}

    # --- 1:1 gnark replacements; all arguments/results are bytes -------------
    def g1_msm(self, points: bytes, scalars: bytes) -> bytes:
        n = len(points) // G1_AFFINE_BYTES
        if len(scalars) != n * FR_BYTES:
            raise CdlError(-3, "len(points) != len(scalars)")
        out = C.create_string_buffer(G1_JAC_BYTES)
        self._chk(self.lib.cdl_g1_msm(self.h, points, scalars, n, out))
        return out.raw

    def g1_msm_batch(self, points: bytes, scalars: bytes, offsets) -> bytes:
        k = len(offsets) - 1
        offs = (C.c_uint32 * (k + 1))(*offsets)
        out = C.create_string_buffer(max(1, k) * G1_AFFINE_BYTES)
        self._chk(self.lib.cdl_g1_msm_batch(self.h, points, scalars, offs, k, out))
        return out.raw[: k * G1_AFFINE_BYTES]

    def g1_scalar_mul_affine(self, points: bytes, scalars: bytes, broadcast: bool) -> bytes:
        n = len(points) // G1_AFFINE_BYTES
        out = C.create_string_buffer(max(1, n) * G1_AFFINE_BYTES)
        self._chk(self.lib.cdl_g1_scalar_mul_affine(self.h, points, scalars, n, 0 if broadcast else 1, out))
        return out.raw[: n * G1_AFFINE_BYTES]

    def g1_fold(self, L: bytes, R: bytes, x: bytes) -> bytes:
        n = len(L) // G1_AFFINE_BYTES
        buf = C.create_string_buffer(L, max(1, len(L)))
        self._chk(self.lib.cdl_g1_fold(self.h, buf, R, x, n))
        return buf.raw[: len(L)]

    def g1_batch_scalar_mul_base(self, base: bytes, scalars: bytes, affine: bool = True, compressed: bool = False):
        """bls12381.BatchScalarMultiplicationG1: scalars[i] * base for n scalars (n x 32 bytes, gnark fr.Element)
        and one affine base (96 bytes, in G1) -> n x 96 affine bytes if `affine`, n x 48 compressed bytes if
        `compressed`, or the pair (affine, compressed) when both are asked for."""
        if not (affine or compressed):
            raise CdlError(-3, "ask for affine or compressed results")
        n = len(scalars) // FR_BYTES
        out = C.create_string_buffer(max(1, n) * G1_AFFINE_BYTES) if affine else None
        out48 = C.create_string_buffer(max(1, n) * 48) if compressed else None
        self._chk(self.lib.cdl_g1_batch_scalar_mul_base(self.h, base, scalars, n, out, out48))
        a = out.raw[: n * G1_AFFINE_BYTES] if affine else None
        z = out48.raw[: n * 48] if compressed else None
        if affine and compressed:
            return a, z
        return a if affine else z

    def g1_batch_to_affine(self, jac: bytes) -> bytes:
        n = len(jac) // G1_JAC_BYTES
        out = C.create_string_buffer(max(1, n) * G1_AFFINE_BYTES)
        self._chk(self.lib.cdl_g1_batch_to_affine(self.h, jac, n, out))
        return out.raw[: n * G1_AFFINE_BYTES]

    def g1_sum_affine(self, points: bytes) -> bytes:
        n = len(points) // G1_AFFINE_BYTES
        out = C.create_string_buffer(G1_AFFINE_BYTES)
        self._chk(self.lib.cdl_g1_sum_affine(self.h, points, n, out))
        return out.raw

    def g1_compress(self, points: bytes) -> bytes:
        n = len(points) // G1_AFFINE_BYTES
        out = C.create_string_buffer(max(1, n) * 48)
        self._chk(self.lib.cdl_g1_compress(self.h, points, n, out))
        return out.raw[: n * 48]

    def g1_decompress(self, enc: bytes, check: bool = True):
        """Returns (affine bytes, status list).  Raises CdlError(CDL_ERR_DECODE)
        when `check` and any point was rejected."""
        n = len(enc) // 48
        out = C.create_string_buffer(max(1, n) * G1_AFFINE_BYTES)
        st = C.create_string_buffer(max(1, n))
        rc = self.lib.cdl_g1_decompress(self.h, enc, n, out, st)
        if rc != 0 and (check or rc != -4):
            self._chk(rc)
        return out.raw[: n * G1_AFFINE_BYTES], list(st.raw[:n])

    def fp_mul(self, a: bytes, b: bytes) -> bytes:
        n = len(a) // FP_BYTES
        out = C.create_string_buffer(max(1, n) * FP_BYTES)
        self._chk(self.lib.cdl_fp_mul(self.h, a, b, n, out))
        return out.raw[: n * FP_BYTES]

    def int_peak(self, kind: int, iters: int):
        ops, ms = C.c_double(), C.c_double()
        self._chk(self.lib.cdl_int_peak(self.h, kind, iters, C.byref(ops), C.byref(ms)))
        return ops.value, ms.value


def _ctx_int_peak_cfg(self, kind: int, iters: int, blocks_per_sm: int, tpb: int):
    ops, ms = C.c_double(), C.c_double()
    self._chk(self.lib.cdl_int_peak_cfg(self.h, kind, iters, blocks_per_sm, tpb, C.byref(ops), C.byref(ms)))
    return ops.value, ms.value


class DeviceBuffer:
    """Raw device memory owned by a Context (cdl_dev_alloc)."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx = ctx
        self.nbytes = nbytes
        p = C.c_void_p()
        ctx._chk(ctx.lib.cdl_dev_alloc(ctx.h, nbytes, C.byref(p)))
        self.ptr = p

    def upload(self, data: bytes, offset: int = 0):
        if offset + len(data) > self.nbytes:
            raise ValueError("upload past the end of the device buffer")
        self.ctx._chk(self.ctx.lib.cdl_dev_upload(self.ctx.h, C.c_void_p(self.ptr.value + offset), data, len(data)))

    def download(self, nbytes: int | None = None, offset: int = 0) -> bytes:
        nbytes = self.nbytes - offset if nbytes is None else nbytes
        out = C.create_string_buffer(max(1, nbytes))
        self.ctx._chk(self.ctx.lib.cdl_dev_download(self.ctx.h, out, C.c_void_p(self.ptr.value + offset), nbytes))
        return out.raw[:nbytes]

    def close(self):
        if getattr(self, "ptr", None) and getattr(self.ctx, "h", None):
            self.ctx.lib.cdl_dev_free(self.ctx.h, self.ptr)
        self.ptr = None

    __del__ = close


def comm_unique_id() -> bytes:
    """128-byte NCCL unique id (rank 0 creates it, the host application ships it to every rank)."""
    lib = load_library()
    out = C.create_string_buffer(128)
    rc = lib.cdl_comm_unique_id(out)
    if rc != 0:
        raise CdlError(rc, "cdl_comm_unique_id (NCCL unavailable?)")
    return out.raw


def comm_partition(n: int, world: int, rank: int, window_bits: int = 0):
    """Windows owned by `rank`: (first_window, window_step, n_windows, my_windows).  Pure host logic."""
    lib = load_library()
    a, b, c, d = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    lib.cdl_comm_partition(n, world, rank, window_bits, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    return a.value, b.value, c.value, d.value


def _ctx_dev_buffer(self, nbytes: int) -> DeviceBuffer:
    return DeviceBuffer(self, nbytes)


def _ctx_g1_scalar_mul_affine_device(self, d_in: DeviceBuffer, d_s: DeviceBuffer, n: int, broadcast: bool,
                                     d_out: DeviceBuffer):
    self._chk(self.lib.cdl_g1_scalar_mul_affine_device(self.h, d_in.ptr, d_s.ptr, n, 0 if broadcast else 1, d_out.ptr))


def _ctx_g1_msm_batch_device(self, d_pool: "DeviceBuffer", idx, scalars: bytes, offsets, out_slot=None, want_affine=True,
                             want_enc=True):
    """Batched MSM over a device-resident pool; returns (affine bytes | None, 48-byte encodings | None)."""
    k = len(offsets) - 1
    ia = (C.c_uint32 * max(1, len(idx)))(*idx)
    oa = (C.c_uint32 * (k + 1))(*offsets)
    sa = (C.c_uint32 * k)(*out_slot) if out_slot is not None else None
    out = C.create_string_buffer(max(1, k) * G1_AFFINE_BYTES) if want_affine else None
    o48 = C.create_string_buffer(max(1, k) * 48) if want_enc else None
    self._chk(self.lib.cdl_g1_msm_batch_device(self.h, d_pool.ptr, ia, scalars, oa, k, sa, out, o48))
    return (out.raw[:k * G1_AFFINE_BYTES] if out else None), (o48.raw[:k * 48] if o48 else None)


def _ctx_g1_fold_device(self, d_L: DeviceBuffer, d_R: DeviceBuffer, d_x: DeviceBuffer, n: int):
    self._chk(self.lib.cdl_g1_fold_device(self.h, d_L.ptr, d_R.ptr, d_x.ptr, n))


def _ctx_g1_msm_device(self, d_points, d_scalars, n: int, part_index: int = 0, part_count: int = 1,
                       normalize: bool = True, d_out: DeviceBuffer | None = None):
    """MultiExp on device vectors -> (G1Jac bytes, kernel ms).  d_points / d_scalars are DeviceBuffers or raw ints."""
    own = d_out is None
    if own:
        d_out = DeviceBuffer(self, G1_JAC_BYTES)
    ms = C.c_float()
    pp = d_points.ptr if isinstance(d_points, DeviceBuffer) else C.c_void_p(int(d_points))
    ps = d_scalars.ptr if isinstance(d_scalars, DeviceBuffer) else C.c_void_p(int(d_scalars))
    self._chk(self.lib.cdl_g1_msm_device(self.h, pp, ps, n, part_index, part_count, 1 if normalize else 0, d_out.ptr,
                                         C.byref(ms)))
    res = d_out.download(G1_JAC_BYTES)
    if own:
        d_out.close()
    return res, ms.value


def _ctx_set_msm_window(self, bits: int):
    self._chk(self.lib.cdl_set_msm_window(self.h, bits))


def _ctx_set_fixed_base_min_batch(self, instances: int):
    self._chk(self.lib.cdl_set_fixed_base_min_batch(self.h, instances))


def _ctx_set_batch_verify_min(self, proofs: int):
    self._chk(self.lib.cdl_set_batch_verify_min(self.h, proofs))


def _ctx_set_msm_batch_affine(self, rounds: int):
    self._chk(self.lib.cdl_set_msm_batch_affine(self.h, rounds))


def _ctx_comm_init(self, uid: bytes, rank: int, world: int):
    self._chk(self.lib.cdl_comm_init(self.h, uid, rank, world))


def _ctx_comm_destroy(self):
    self._chk(self.lib.cdl_comm_destroy(self.h))


def _ctx_g1_msm_sharded_device(self, d_points: DeviceBuffer, d_scalars: DeviceBuffer, n: int):
    d_out = DeviceBuffer(self, G1_JAC_BYTES)
    ms = C.c_float()
    self._chk(self.lib.cdl_g1_msm_sharded_device(self.h, d_points.ptr, d_scalars.ptr, n, d_out.ptr, C.byref(ms)))
    res = d_out.download(G1_JAC_BYTES)
    d_out.close()
    return res, ms.value


def _ctx_g1_msm_sharded(self, points: bytes, scalars: bytes) -> bytes:
    n = len(points) // G1_AFFINE_BYTES
    if len(scalars) != n * FR_BYTES:
        raise CdlError(-3, "len(points) != len(scalars)")
    out = C.create_string_buffer(G1_JAC_BYTES)
    self._chk(self.lib.cdl_g1_msm_sharded(self.h, points, scalars, n, out))
    return out.raw


class Rand:
    """common.Rand (common/rand.go): deterministic SHAKE256 RNG."""

    def __init__(self, seed: int):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.cdl_rand_new(seed, C.byref(h))
        if rc != 0:
            raise CdlError(rc, "cdl_rand_new")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.cdl_rand_free(self.h)
            self.h = None

    __del__ = close

    def get_frs(self, n: int) -> bytes:
        out = C.create_string_buffer(max(1, n) * FR_BYTES)
        rc = self.lib.cdl_rand_get_frs(self.h, n, out)
        if rc != 0:
            raise CdlError(rc, "cdl_rand_get_frs")
        return out.raw[: n * FR_BYTES]

    def get_fr(self) -> bytes:
        return self.get_frs(1)

    def generate_permutation(self, n: int):
        out = (C.c_uint32 * max(1, n))()
        rc = self.lib.cdl_rand_generate_permutation(self.h, n, out)
        if rc != 0:
            raise CdlError(rc, "cdl_rand_generate_permutation")
        return list(out[:n])


class CRS:
    """curdleproof.CRS (crs.go:10-18), device resident."""

    def __init__(self, ctx: "Context", handle):
        self.ctx = ctx
        self.h = handle

    @property
    def ell(self) -> int:
        return self.ctx.lib.cdl_crs_ell(self.h)

    def export(self) -> bytes:
        """Gs[ell] | Hs[4] | H | Gt | Gu | Gsum | Hsum as affine points."""
        out = C.create_string_buffer((self.ell + 9) * G1_AFFINE_BYTES)
        self.ctx._chk(self.ctx.lib.cdl_crs_export(self.ctx.h, self.h, out))
        return out.raw

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.lib.cdl_crs_free(self.h)
        self.h = None

    __del__ = close


def _ctx_rand_get_g1_affines(self, rand: Rand, n: int) -> bytes:
    out = C.create_string_buffer(max(1, n) * G1_AFFINE_BYTES)
    self._chk(self.lib.cdl_rand_get_g1_affines(self.h, rand.h, n, out))
    return out.raw[: n * G1_AFFINE_BYTES]


def _ctx_generate_crs(self, ell: int, rand: Rand) -> CRS:
    """curdleproof.GenerateCRS (crs.go:20-59)."""
    h = C.c_void_p()
    self._chk(self.lib.cdl_crs_generate(self.h, ell, rand.h, C.byref(h)))
    return CRS(self, h)


def _ctx_crs_from_points(self, ell: int, points: bytes) -> CRS:
    h = C.c_void_p()
    self._chk(self.lib.cdl_crs_from_points(self.h, ell, points, C.byref(h)))
    return CRS(self, h)


def _ctx_shuffle_permute_commit(self, crs: CRS, Rs: bytes, Ss: bytes, perm, k: bytes, rand: Rand):
    """common.ShufflePermuteCommit -> (Ts, Us, M jac, rs_m)."""
    ell = crs.ell
    Ts = C.create_string_buffer(ell * G1_AFFINE_BYTES)
    Us = C.create_string_buffer(ell * G1_AFFINE_BYTES)
    M = C.create_string_buffer(G1_JAC_BYTES)
    rs_m = C.create_string_buffer(4 * FR_BYTES)
    p = (C.c_uint32 * ell)(*perm)
    self._chk(self.lib.cdl_shuffle_permute_commit(self.h, crs.h, Rs, Ss, p, k, rand.h, Ts, Us, M, rs_m))
    return Ts.raw, Us.raw, M.raw, rs_m.raw


def _ctx_prove(self, crs: CRS, Rs, Ss, Ts, Us, M, perm, k, rs_m, rand: Rand) -> bytes:
    """curdleproof.Prove + Proof.Serialize."""
    ell = crs.ell
    cap = PROOF_CAP
    out = C.create_string_buffer(cap)
    n = C.c_size_t()
    p = (C.c_uint32 * ell)(*perm)
    self._chk(self.lib.cdl_prove(self.h, crs.h, Rs, Ss, Ts, Us, M, p, k, rs_m, rand.h, out, cap, C.byref(n)))
    return out.raw[: n.value]


def _ctx_verify(self, crs: CRS, proof: bytes, Rs, Ss, Ts, Us, M, rand: Rand) -> bool:
    """Proof.FromReader + curdleproof.Verify; raises CdlError where the reference returns an error."""
    ok = C.c_int32()
    self._chk(self.lib.cdl_verify(self.h, crs.h, proof, len(proof), Rs, Ss, Ts, Us, M, rand.h, C.byref(ok)))
    return bool(ok.value)


PROOF_CAP = 48 * (18 + 10 * 32) + 32 * 7 + 40  # the largest proof Prove serializes (lg n < 32)


def _split(buf, n: int, size: int):
    return [bytes(buf[i * size:(i + 1) * size]) for i in range(n)]


def _perms(perms, B: int, ell: int):
    flat = [p for perm in perms for p in perm]
    if len(perms) != B or len(flat) != B * ell:
        raise CdlError(-3, "every instance needs a permutation of ell entries")
    return (C.c_uint32 * (B * ell))(*flat)


def _ctx_shuffle_permute_commit_batch(self, crs: CRS, Rs, Ss, perms, ks, rands):
    """common.ShufflePermuteCommit for B = len(rands) instances.  Rs, Ss and ks are lists of per-instance
    byte strings (ell affine points, one fr.Element), perms a list of permutations.  Returns per-instance
    lists (Ts, Us, M jac, rs_m, status); an instance whose status is not 0 has zero-filled outputs."""
    B, ell = len(rands), crs.ell
    pb = ell * G1_AFFINE_BYTES
    Ts, Us = bytearray(B * pb), bytearray(B * pb)
    M, rs_m = bytearray(B * G1_JAC_BYTES), bytearray(B * 4 * FR_BYTES)
    status = (C.c_int32 * max(1, B))()
    rh = (C.c_void_p * max(1, B))(*[r.h for r in rands])
    self._chk(self.lib.cdl_shuffle_permute_commit_batch(
        self.h, crs.h, B, b"".join(Rs), b"".join(Ss), _perms(perms, B, ell), b"".join(ks), rh, _inbuf(Ts), _inbuf(Us),
        _inbuf(M), _inbuf(rs_m), status))
    return (_split(Ts, B, pb), _split(Us, B, pb), _split(M, B, G1_JAC_BYTES), _split(rs_m, B, 4 * FR_BYTES),
            list(status)[:B])


def _ctx_prove_batch(self, crs: CRS, Rs, Ss, Ts, Us, Ms, perms, ks, rs_ms, rands, proof_cap: int = PROOF_CAP):
    """curdleproof.Prove + Proof.Serialize for B = len(rands) instances (lists of per-instance byte strings as
    in shuffle_permute_commit_batch).  Returns (proofs, proof lengths, status): proofs[b] is b"" unless
    status[b] == 0; the length is also reported when the proof did not fit proof_cap."""
    B, ell = len(rands), crs.ell
    out = bytearray(max(1, B) * proof_cap)
    lens = (C.c_size_t * max(1, B))()
    status = (C.c_int32 * max(1, B))()
    rh = (C.c_void_p * max(1, B))(*[r.h for r in rands])
    self._chk(self.lib.cdl_prove_batch(
        self.h, crs.h, B, b"".join(Rs), b"".join(Ss), b"".join(Ts), b"".join(Us), b"".join(Ms), _perms(perms, B, ell),
        b"".join(ks), b"".join(rs_ms), rh, _inbuf(out), proof_cap, lens, status))
    proofs = [bytes(out[b * proof_cap:b * proof_cap + lens[b]]) if status[b] == 0 else b"" for b in range(B)]
    return proofs, list(lens)[:B], list(status)[:B]


def _ctx_verify_batch(self, crs: CRS, proofs, Rs, Ss, Ts, Us, Ms, rands):
    """Proof.FromReader + curdleproof.Verify for B = len(rands) instances: proofs is a list of proof byte
    strings, the instance arguments lists as in prove_batch.  Returns (ok, status) lists; status[b] is
    what cdl_verify would have returned for instance b."""
    B = len(rands)
    stride = max([len(p) for p in proofs] + [1])
    buf = b"".join(p.ljust(stride, b"\0") for p in proofs)
    lens = (C.c_size_t * max(1, B))(*[len(p) for p in proofs])
    ok = (C.c_int32 * max(1, B))()
    status = (C.c_int32 * max(1, B))()
    rh = (C.c_void_p * max(1, B))(*[r.h for r in rands])
    self._chk(self.lib.cdl_verify_batch(self.h, crs.h, B, buf, stride, lens, b"".join(Rs), b"".join(Ss), b"".join(Ts),
                                        b"".join(Us), b"".join(Ms), rh, ok, status))
    return list(ok)[:B], list(status)[:B]


def _ctx_whisk_generate(self, crs: CRS, pre: bytes, rand: Rand, proof_size: int = 4576):
    """whisk.GenerateWhiskShuffleProof -> (post_trackers, proof)."""
    ell = crs.ell
    post = C.create_string_buffer(ell * 96)
    proof = C.create_string_buffer(proof_size)
    self._chk(self.lib.cdl_whisk_generate_shuffle_proof(self.h, crs.h, pre, rand.h, post, proof, proof_size))
    return post.raw, proof.raw


def _ctx_whisk_is_valid(self, crs: CRS, pre: bytes, post: bytes, proof: bytes, rand: Rand) -> bool:
    """whisk.IsValidWhiskShuffleProof."""
    ok = C.c_int32()
    self._chk(self.lib.cdl_whisk_is_valid_shuffle_proof(self.h, crs.h, pre, post, len(pre) // 96, len(post) // 96,
                                                        proof, len(proof), rand.h, C.byref(ok)))
    return bool(ok.value)


def _inbuf(x):
    """bytes pass through; writable bytes-likes (bytearray, memoryview) are wrapped without a copy."""
    if isinstance(x, bytes):
        return x
    return (C.c_char * len(x)).from_buffer(x)


def _ctx_whisk_generate_batch(self, crs: CRS, pre, rands, proof_size: int = 4576):
    """Returns (post_trackers, proofs, status); the two buffers are bytearrays the library wrote
    into directly (no intermediate copies: they are tens of MB for a few thousand instances)."""
    B = len(rands)
    ell = crs.ell
    post = bytearray(B * ell * 96)
    proofs = bytearray(B * proof_size)
    status = (C.c_int32 * B)()
    rh = (C.c_void_p * B)(*[r.h for r in rands])
    self._chk(self.lib.cdl_whisk_generate_shuffle_proof_batch(self.h, crs.h, B, _inbuf(pre), rh, _inbuf(post), _inbuf(proofs),
                                                              proof_size, status))
    return post, proofs, list(status)


def _ctx_whisk_is_valid_batch(self, crs: CRS, pre, post, proofs, rands, proof_size: int = 4576):
    B = len(rands)
    ok = (C.c_int32 * B)()
    status = (C.c_int32 * B)()
    rh = (C.c_void_p * B)(*[r.h for r in rands])
    self._chk(self.lib.cdl_whisk_is_valid_shuffle_proof_batch(self.h, crs.h, B, _inbuf(pre), _inbuf(post), _inbuf(proofs),
                                                              proof_size, rh, ok, status))
    return list(ok), list(status)


def _ctx_whisk_generate_tracker_proof_batch(self, trackers: bytes, ks: bytes, rands):
    """whisk.GenerateWhiskTrackerProof for B trackers -> (B x 128 proof bytes, status list)."""
    B = len(rands)
    proofs = C.create_string_buffer(B * 128)
    status = (C.c_int32 * B)()
    rh = (C.c_void_p * B)(*[r.h for r in rands])
    self._chk(self.lib.cdl_whisk_generate_tracker_proof_batch(self.h, B, trackers, ks, rh, proofs, status))
    return proofs.raw, list(status)


def _ctx_whisk_is_valid_tracker_proof_batch(self, trackers: bytes, k_comms: bytes, proofs: bytes):
    """whisk.IsValidWhiskTrackerProof for B trackers -> (ok list, status list)."""
    B = len(trackers) // 96
    ok = (C.c_int32 * B)()
    status = (C.c_int32 * B)()
    self._chk(self.lib.cdl_whisk_is_valid_tracker_proof_batch(self.h, B, trackers, k_comms, proofs, ok, status))
    return list(ok), list(status)


def _ctx_whisk_generate_registration_batch(self, ks: bytes, rands):
    """Whisk registration for B = len(rands) validators with secrets ks (B x 32 bytes, gnark fr.Element): r is
    drawn from each Rand, then one blinder -> (B x 96 tracker bytes {rG, krG}, B x 48 k-commitment bytes kG,
    B x 128 opening-proof bytes, status list).  A validator whose status is not 0 (r = 0 or 1) has zero bytes.
    rands must be distinct Rand objects, one per validator: the validators draw concurrently."""
    B = len(rands)
    trackers = C.create_string_buffer(max(1, B) * 96)
    k_comms = C.create_string_buffer(max(1, B) * 48)
    proofs = C.create_string_buffer(max(1, B) * 128)
    status = (C.c_int32 * max(1, B))()
    rh = (C.c_void_p * max(1, B))(*[r.h for r in rands])
    self._chk(self.lib.cdl_whisk_generate_registration_batch(self.h, B, _inbuf(ks), rh, trackers, k_comms, proofs,
                                                             status))
    return trackers.raw[:96 * B], k_comms.raw[:48 * B], proofs.raw[:128 * B], list(status)[:B]


def _ctx_whisk_match_trackers(self, trackers: bytes, ks: bytes):
    """Which of the V secrets in ks (V x 32 bytes, gnark fr.Element) own which of the T trackers
    (T x 96 bytes) -> (owner list, status list); owner[t] is the smallest owning key index or -1."""
    T = len(trackers) // 96
    V = len(ks) // 32
    owner = (C.c_int32 * max(T, 1))()
    status = (C.c_int32 * max(T, 1))()
    self._chk(self.lib.cdl_whisk_match_trackers(self.h, T, _inbuf(trackers), V, _inbuf(ks), owner, status))
    return list(owner)[:T], list(status)[:T]


def _ctx_engine_stats(self, reset: bool = False):
    """Per kernel class (msm, elem, decompress, compress): launches, event ms, algorithmic modmul / bytes."""
    n = (C.c_uint64 * 4)()
    ms = (C.c_double * 4)()
    mm = (C.c_double * 4)()
    by = (C.c_double * 4)()
    self._chk(self.lib.cdl_engine_stats(self.h, n, ms, mm, by, 1 if reset else 0))
    names = ("msm_small", "elem_scalar_mul", "decompress", "compress")
    return {names[i]: {"launches": int(n[i]), "ms": ms[i], "modmul": mm[i], "bytes": by[i]} for i in range(4)}


def _ctx_engine_busy_ms(self) -> float:
    v = C.c_double()
    self._chk(self.lib.cdl_engine_busy_ms(self.h, C.byref(v)))
    return v.value


def _ctx_engine_busy_ms_device(self, slot: int) -> float:
    """Busy time of device slot `slot` since the last stats reset."""
    v = C.c_double()
    self._chk(self.lib.cdl_engine_busy_ms_device(self.h, slot, C.byref(v)))
    return v.value


def _ctx_devices(self):
    """The context's device list (one entry per device slot)."""
    n = C.c_size_t()
    self._chk(self.lib.cdl_context_devices(self.h, None, 0, C.byref(n)))
    out = (C.c_int32 * max(1, n.value))()
    self._chk(self.lib.cdl_context_devices(self.h, out, n.value, C.byref(n)))
    return list(out)[:n.value]


def _ctx_set_lanes(self, lanes: int):
    self._chk(self.lib.cdl_set_lanes(self.h, lanes))


def _ctx_launch_count(self) -> int:
    return int(self.lib.cdl_launch_count(self.h))


Context.int_peak_cfg = _ctx_int_peak_cfg
Context.dev_buffer = _ctx_dev_buffer
Context.g1_scalar_mul_affine_device = _ctx_g1_scalar_mul_affine_device
Context.g1_fold_device = _ctx_g1_fold_device
Context.g1_msm_batch_device = _ctx_g1_msm_batch_device
Context.g1_msm_device = _ctx_g1_msm_device
Context.set_msm_window = _ctx_set_msm_window
Context.set_msm_batch_affine = _ctx_set_msm_batch_affine
Context.set_fixed_base_min_batch = _ctx_set_fixed_base_min_batch
Context.set_batch_verify_min = _ctx_set_batch_verify_min
Context.comm_init = _ctx_comm_init
Context.comm_destroy = _ctx_comm_destroy
Context.g1_msm_sharded_device = _ctx_g1_msm_sharded_device
Context.g1_msm_sharded = _ctx_g1_msm_sharded
Context.rand_get_g1_affines = _ctx_rand_get_g1_affines
Context.generate_crs = _ctx_generate_crs
Context.crs_from_points = _ctx_crs_from_points
Context.shuffle_permute_commit = _ctx_shuffle_permute_commit
Context.prove = _ctx_prove
Context.verify = _ctx_verify
Context.shuffle_permute_commit_batch = _ctx_shuffle_permute_commit_batch
Context.prove_batch = _ctx_prove_batch
Context.verify_batch = _ctx_verify_batch
Context.whisk_generate_shuffle_proof = _ctx_whisk_generate
Context.whisk_is_valid_shuffle_proof = _ctx_whisk_is_valid
Context.whisk_generate_shuffle_proof_batch = _ctx_whisk_generate_batch
Context.whisk_is_valid_shuffle_proof_batch = _ctx_whisk_is_valid_batch
Context.whisk_generate_tracker_proof_batch = _ctx_whisk_generate_tracker_proof_batch
Context.whisk_is_valid_tracker_proof_batch = _ctx_whisk_is_valid_tracker_proof_batch
Context.whisk_generate_registration_batch = _ctx_whisk_generate_registration_batch
Context.whisk_match_trackers = _ctx_whisk_match_trackers
Context.launch_count = _ctx_launch_count
Context.engine_busy_ms = _ctx_engine_busy_ms
Context.engine_busy_ms_device = _ctx_engine_busy_ms_device
Context.devices = _ctx_devices
Context.set_lanes = _ctx_set_lanes
Context.engine_stats = _ctx_engine_stats
