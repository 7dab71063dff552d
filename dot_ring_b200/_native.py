"""ctypes binding of ``libdotring_b200.so`` (C ABI declared in ``include/dot_ring_b200.h``).

The product always loads the CUDA build that sits next to this file and raises if it is missing
or is not a CUDA build; there is no CPU fallback.  ``Library(path)`` exists so that the CPU
test-suite can bind the *test-only* emulation build of the same sources (``tests/host``)
explicitly; nothing in this package ever selects it.
"""

from __future__ import annotations

import ctypes
import itertools
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_size_t, c_uint8, c_uint32, c_uint64, c_void_p
from pathlib import Path

import numpy as np

DR_OK, DR_EINVAL, DR_ECUDA, DR_ENOMEM, DR_ESTATE = 0, -1, -2, -3, -4

_HERE = Path(__file__).resolve().parent
DEFAULT_LIBRARY = _HERE / "libdotring_b200.so"
FR_MODULUS = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
BANDERSNATCH_ORDER = 0x1CFB69D4CA675F520CCE760202687600FF8F87007419047174FD06B52876E7E1


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"dot_ring_b200 native error {code}: {message}")
        self.code = code
        self.message = message


def _u8(buf) -> ctypes.Array:
    return (c_uint8 * len(buf)).from_buffer_copy(bytes(buf))


class Library:
    """One loaded shared library + typed entry points."""

    def __init__(self, path: os.PathLike | str | None = None, require_cuda: bool = True):
        path = Path(path) if path is not None else DEFAULT_LIBRARY
        if not path.exists():
            raise ImportError(
                f"{path} is missing: build it with ./build.sh (nvcc, sm_100a). dot_ring_b200 has no CPU fallback."
            )
        self.path = path
        self.lib = ctypes.CDLL(str(path))
        self._declare()
        if require_cuda and not self.lib.dr_is_cuda_build():
            raise ImportError(f"{path} is not a CUDA build; refusing to run the product path on the CPU")

    # ---- prototypes ---------------------------------------------------------------------------
    def _declare(self) -> None:
        L = self.lib
        L.dr_last_error.restype = c_char_p
        L.dr_version.restype = c_char_p
        L.dr_is_cuda_build.restype = c_int
        L.dr_launch_count.restype = c_uint64
        L.dr_ctx_create.argtypes = [c_int, POINTER(c_void_p)]
        L.dr_ctx_destroy.argtypes = [c_void_p]
        L.dr_ctx_destroy.restype = None
        L.dr_ctx_sync.argtypes = [c_void_p]
        L.dr_ctx_trim.argtypes = [c_void_p]
        L.dr_ctx_timer_start.argtypes = [c_void_p]
        L.dr_ctx_timer_stop.argtypes = [c_void_p, POINTER(c_float)]
        L.dr_ctx_device_info.argtypes = [c_void_p, c_char_p, c_size_t, POINTER(c_int), POINTER(c_int), POINTER(c_size_t), POINTER(c_size_t)]
        L.dr_srs_load.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_int, POINTER(c_void_p)]
        L.dr_srs_destroy.argtypes = [c_void_p]
        L.dr_srs_destroy.restype = None
        L.dr_srs_size.argtypes = [c_void_p]
        L.dr_srs_size.restype = c_size_t
        L.dr_srs_table_bytes.argtypes = [c_void_p]
        L.dr_srs_table_bytes.restype = c_size_t
        L.dr_srs_geometry.argtypes = [c_void_p, POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32)]
        L.dr_srs_geometry.restype = None
        L.dr_kzg_commit.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_size_t, c_void_p]
        L.dr_kzg_open.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_void_p, c_void_p]
        L.dr_kzg_pairing_check.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, POINTER(c_int)]
        L.dr_kzg_commit_bench.argtypes = [c_void_p, c_void_p, c_size_t, c_size_t, c_int, c_uint64, POINTER(c_float), c_void_p]
        L.dr_g1_msm.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
        L.dr_g1_synthetic_srs.argtypes = [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p]
        L.dr_fr_ntt_bench.argtypes = [c_void_p, c_size_t, c_size_t, c_int, c_void_p, POINTER(c_float), c_void_p]
        L.dr_g1_msm_bench.argtypes = [c_void_p, c_size_t, c_int, c_uint64, c_int, c_void_p, POINTER(c_float), POINTER(ctypes.c_uint32), c_void_p]
        L.dr_g1_compress.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p]
        L.dr_g1_decompress.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]
        L.dr_fr_ntt.argtypes = [c_void_p, c_void_p, c_size_t, c_size_t, c_int, c_void_p]
        L.dr_field_op.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t]
        L.dr_microbench.argtypes = [c_void_p, c_int, c_int, POINTER(ctypes.c_double), POINTER(c_float)]

        L.dr_ring_create.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, POINTER(c_void_p)]
        L.dr_ring_destroy.argtypes = [c_void_p]
        L.dr_ring_destroy.restype = None
        L.dr_ring_root.argtypes = [c_void_p, c_void_p]
        L.dr_ring_fixed_commitments.argtypes = [c_void_p, c_void_p]
        L.dr_ring_points.argtypes = [c_void_p, c_void_p, c_size_t]
        L.dr_ring_prove_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 10
        L.dr_ring_prove_multi.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t] + [c_void_p] * 10
        L.dr_ring_proof_prove_multi.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]
        L.dr_ring_prove_phase_ms.argtypes = [c_void_p, POINTER(c_float * 6)]
        L.dr_ring_prove_commit_kernel_ms.argtypes = [c_void_p, POINTER(c_float), POINTER(c_uint32)]
        L.dr_ring_witness_table_bits.argtypes = [c_void_p]
        L.dr_ring_witness_table_bits.restype = c_uint32
        L.dr_ctx_set_prove_chunk.argtypes = [c_void_p, c_size_t]
        L.dr_ctx_set_dense_witness_commit.argtypes = [c_void_p, c_int]
        L.dr_ctx_set_commit_mode.argtypes = [c_void_p, c_int]
        L.dr_ctx_set_generic_ntt_path.argtypes = [c_void_p, c_int]

        L.dr_pedersen_verify_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 7
        L.dr_tiny_verify_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 8
        L.dr_pedersen_prove_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 7
        L.dr_tiny_prove_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 7
        L.dr_pedersen_prove_batch_ex.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 8
        L.dr_thin_prove_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 7
        L.dr_thin_verify_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 8
        L.dr_ring_proof_verify_batch.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_int, c_void_p, POINTER(c_int)]
        L.dr_ring_verify_batch.argtypes = [c_void_p, c_void_p, c_size_t] + [c_void_p] * 7 + [c_int, c_void_p, POINTER(c_int)]
        L.dr_ring_verify_set_msm_threshold.argtypes = [c_size_t]
        L.dr_ring_roots_from_keys.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]
        L.dr_ring_root_update.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]
        L.dr_ring_verifier_create.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_void_p)]
        L.dr_ring_verifier_destroy.argtypes = [c_void_p]
        L.dr_ring_verifier_destroy.restype = None
        L.dr_ring_verify_multi.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t] + [c_void_p] * 7 + [c_int, c_void_p, POINTER(c_int)]
        L.dr_vrf_verify_set_coop_threshold.argtypes = [c_size_t]
        L.dr_pairing_check_batch.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
        L.dr_te_decode_batch.argtypes = [c_void_p, c_void_p, c_size_t, c_int, c_void_p, c_void_p]
        L.dr_te_msm.argtypes = [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
        L.dr_te_mul_batch.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p, c_void_p]

    def check(self, code: int) -> None:
        if code == DR_OK:
            return
        msg = (self.lib.dr_last_error() or b"").decode("utf-8", "replace")
        if code == DR_EINVAL:
            raise ValueError(msg)
        if code == DR_ENOMEM:
            raise MemoryError(msg)
        raise NativeError(code, msg)

    @property
    def is_cuda(self) -> bool:
        return bool(self.lib.dr_is_cuda_build())

    def launch_count(self) -> int:
        return int(self.lib.dr_launch_count())

    def device_count(self) -> int:
        return int(self.lib.dr_device_count())


_default: Library | None = None


def default_library() -> Library:
    """The CUDA library next to this package (loaded once); raises ImportError when absent."""
    global _default
    if _default is None:
        _default = Library()
    return _default


def set_default_library(lib: Library | None) -> None:
    """Test hook: inject an explicitly constructed Library (e.g. the tests/host emulation build)."""
    global _default
    _default = lib


class VrfSuiteStruct(ctypes.Structure):
    """dr_vrf_suite (include/dot_ring_b200.h)."""

    _fields_ = [
        ("suite_id_len", ctypes.c_uint32),
        ("h2c_dst_len", ctypes.c_uint32),
        ("hash_id", ctypes.c_uint32),
        ("pad", ctypes.c_uint32),
        ("suite_id", c_uint8 * 32),
        ("h2c_dst", c_uint8 * 64),
        ("generator", c_uint8 * 64),
        ("blinding_base", c_uint8 * 64),
    ]


class VerifierKeyStruct(ctypes.Structure):
    """dr_verifier_key (include/dot_ring_b200.h)."""

    _fields_ = [
        ("domain_size", ctypes.c_uint32),
        ("label_len", ctypes.c_uint32),
        ("label", c_uint8 * 32),
        ("omega", c_uint8 * 32),
        ("seed", c_uint8 * 64),
        ("g1_0_be96", c_uint8 * 96),
        ("g2_be192", c_uint8 * 384),
        ("fixed_be96", c_uint8 * 288),
    ]


def _put(arr, data: bytes) -> None:
    data = bytes(data)
    if len(data) > ctypes.sizeof(arr):
        raise ValueError(f"value of {len(data)} bytes does not fit a {ctypes.sizeof(arr)}-byte field")
    ctypes.memmove(arr, data, len(data))


def _xy64(pt) -> bytes:
    return int(pt[0]).to_bytes(32, "little") + int(pt[1]).to_bytes(32, "little")


HASH_IDS = {"sha512": 0, "shake128": 1}


def make_suite(suite_id: bytes, h2c_dst: bytes, generator, blinding_base, hash_name: str = "sha512") -> VrfSuiteStruct:
    s = VrfSuiteStruct()
    s.suite_id_len, s.h2c_dst_len = len(suite_id), len(h2c_dst)
    s.hash_id = HASH_IDS[hash_name]
    _put(s.suite_id, suite_id)
    _put(s.h2c_dst, h2c_dst)
    _put(s.generator, _xy64(generator))
    _put(s.blinding_base, _xy64(blinding_base))
    return s


def pack_items(inputs: list[bytes], ads: list[bytes]):
    """(blob, in_off, in_len, ad_off, ad_len) ctypes arrays for the batched entry points."""
    n = len(inputs)
    if len(ads) != n:
        raise ValueError("inputs and additional data must have the same length")
    if n == 0:
        U32 = ctypes.c_uint32 * 1
        return None, U32(), U32(), U32(), U32()
    in_len = np.fromiter(map(len, inputs), dtype=np.uint32, count=n)
    ad_len = np.fromiter(map(len, ads), dtype=np.uint32, count=n)
    ends = np.cumsum(in_len.astype(np.uint64) + ad_len)
    if int(ends[-1]) >> 32:
        raise ValueError("a batch carries at most 4 GiB of input and additional data")
    in_off = (ends - in_len - ad_len).astype(np.uint32)
    ad_off = in_off + in_len
    blob = b"".join(itertools.chain.from_iterable(zip(inputs, ads)))
    return (blob or None, *[np.ctypeslib.as_ctypes(a) for a in (in_off, in_len, ad_off, ad_len)])


class Context:
    """One per GPU (dr_ctx)."""

    def __init__(self, device: int = 0, library: Library | None = None):
        self.library = library or default_library()
        self.handle = c_void_p()
        self.library.check(self.library.lib.dr_ctx_create(device, ctypes.byref(self.handle)))
        self.device = device

    def close(self) -> None:
        if self.handle:
            self.library.lib.dr_ctx_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def sync(self) -> None:
        self.library.check(self.library.lib.dr_ctx_sync(self.handle))

    def set_commit_mode(self, mode: int) -> None:
        """0: XYZZ accumulation, 1: batched-affine pairing rounds (same commitments, cheaper additions)."""
        self.library.check(self.library.lib.dr_ctx_set_commit_mode(self.handle, mode))

    def set_prove_chunk(self, chunk: int) -> None:
        """Proofs per internal pass of dr_ring_prove_batch (0 = automatic, 4096 or what the free memory allows)."""
        self.library.check(self.library.lib.dr_ctx_set_prove_chunk(self.handle, chunk))

    def set_generic_ntt_path(self, enabled: bool) -> None:
        """Force the large-domain route (element-wise twists around the batched NTT) at any domain size (tests)."""
        self.library.check(self.library.lib.dr_ctx_set_generic_ntt_path(self.handle, 1 if enabled else 0))

    def set_dense_witness_commit(self, enabled: bool) -> None:
        """Commit witness columns from interpolated coefficients (the reference's route) instead of the sparse Lagrange form."""
        self.library.check(self.library.lib.dr_ctx_set_dense_witness_commit(self.handle, 1 if enabled else 0))

    def trim(self) -> None:
        """Return cached device scratch to the driver."""
        self.library.check(self.library.lib.dr_ctx_trim(self.handle))

    def timer_start(self) -> None:
        self.library.check(self.library.lib.dr_ctx_timer_start(self.handle))

    def timer_stop(self) -> float:
        ms = c_float()
        self.library.check(self.library.lib.dr_ctx_timer_stop(self.handle, ctypes.byref(ms)))
        return float(ms.value)

    def device_info(self) -> dict:
        name = ctypes.create_string_buffer(128)
        sm, khz, free, total = c_int(), c_int(), c_size_t(), c_size_t()
        self.library.check(
            self.library.lib.dr_ctx_device_info(self.handle, name, 128, ctypes.byref(sm), ctypes.byref(khz), ctypes.byref(free), ctypes.byref(total))
        )
        return {"name": name.value.decode(), "sm_count": sm.value, "sm_clock_khz": khz.value, "free_bytes": free.value, "total_bytes": total.value}

    # ---- Fr NTT ---------------------------------------------------------------------------------
    def fr_ntt(self, values: list[int], n: int, omega: int, inverse: bool = False) -> list[int]:
        """Batched transform of len(values)/n vectors; ints in, ints out (fft.py:87-144 semantics)."""
        if len(values) % n:
            raise ValueError("values length must be a multiple of n")
        batch = len(values) // n
        buf = ctypes.create_string_buffer(b"".join(int(v).to_bytes(32, "little") for v in values), 32 * len(values))
        self.library.check(self.library.lib.dr_fr_ntt(self.handle, buf, n, batch, 1 if inverse else 0, int(omega).to_bytes(32, "little")))
        raw = buf.raw
        return [int.from_bytes(raw[32 * i : 32 * i + 32], "little") for i in range(len(values))]

    def field_op(self, field: str, op: str, a: list[int], b: list[int] | None = None) -> list[int]:
        """Element-wise device arithmetic in 'fq' | 'fr' | 'fn' (self-test of the Montgomery kernels)."""
        fidx = {"fq": 0, "fr": 1, "fn": 2}[field]
        oidx = {"mul": 0, "add": 1, "sub": 2, "inv": 3, "sqr": 4, "neg": 5}[op]
        b = b if b is not None else [0] * len(a)
        size, order = (48, "big") if fidx == 0 else (32, "little")
        out = ctypes.create_string_buffer(size * len(a))
        abuf = b"".join(int(x).to_bytes(size, order) for x in a)
        bbuf = b"".join(int(x).to_bytes(size, order) for x in b)
        self.library.check(self.library.lib.dr_field_op(self.handle, fidx, oidx, abuf, bbuf, out, len(a)))
        raw = out.raw
        return [int.from_bytes(raw[size * i : size * i + size], order) for i in range(len(a))]

    def microbench(self, kind: str, iters: int) -> tuple[float, float]:
        """(ops per second over the chip, elapsed ms) for 'imad' | 'imad_wide' | 'fq_mul' | 'fr_mul' | 'g1_madd'."""
        k = {"imad": 0, "imad_wide": 1, "fq_mul": 2, "fr_mul": 3, "g1_madd": 4, "dfma": 5, "imad_dfma": 6, "fr_chain": 7, "fq_chain": 8, "fr_inv_chain": 9, "fq_inv_chain": 10, "fq_sqr": 11, "fr_sqr": 12}[kind]
        ops, ms = ctypes.c_double(), c_float()
        self.library.check(self.library.lib.dr_microbench(self.handle, k, iters, ctypes.byref(ops), ctypes.byref(ms)))
        return float(ops.value), float(ms.value)

    def te_decode(self, encoded: list[bytes], checked: bool = True) -> list[tuple[int, int] | None]:
        """Batch `dec_point`: affine (x, y) per item, None where the reference would raise ValueError."""
        n = len(encoded)
        if any(len(e) != 32 for e in encoded):
            raise ValueError("point must be exactly 32 bytes")
        out = ctypes.create_string_buffer(64 * max(n, 1))
        ok = ctypes.create_string_buffer(max(n, 1))
        self.library.check(self.library.lib.dr_te_decode_batch(self.handle, b"".join(encoded), n, 1 if checked else 0, out, ok))
        raw, okr = out.raw, ok.raw
        return [
            (int.from_bytes(raw[64 * i : 64 * i + 32], "little"), int.from_bytes(raw[64 * i + 32 : 64 * i + 64], "little")) if okr[i] else None
            for i in range(n)
        ]

    def te_mul(self, points: list[bytes], scalars: list[int]) -> list[bytes | None]:
        """Batch scalar multiplication on 32-byte encodings; one shared base when len(points) == 1."""
        n = len(scalars)
        out = ctypes.create_string_buffer(32 * max(n, 1))
        ok = ctypes.create_string_buffer(max(n, 1))
        ks = b"".join((int(k) % BANDERSNATCH_ORDER).to_bytes(32, "little") for k in scalars)
        self.library.check(self.library.lib.dr_te_mul_batch(self.handle, b"".join(points), len(points), ks, n, out, ok))
        raw, okr = out.raw, ok.raw
        return [raw[32 * i : 32 * i + 32] if okr[i] else None for i in range(n)]

    # ---- verification ---------------------------------------------------------------------------
    def pedersen_verify(self, suite: VrfSuiteStruct, inputs: list[bytes], ads: list[bytes], proofs: list[bytes]) -> list[int]:
        """Per item: 1 valid, 0 invalid, 2 malformed (PedersenVRF.decode would raise ValueError)."""
        n = len(proofs)
        if any(len(p) != 192 for p in proofs):
            raise ValueError("invalid Pedersen VRF proof length: expected 192")
        blob, a, b, c, d = pack_items(inputs, ads)
        out = ctypes.create_string_buffer(max(n, 1))
        self.library.check(self.library.lib.dr_pedersen_verify_batch(self.handle, ctypes.byref(suite), n, blob, a, b, c, d, b"".join(proofs), out))
        return list(out.raw[:n])

    def thin_verify(self, suite: VrfSuiteStruct, public_keys: list[bytes], inputs: list[bytes], ads: list[bytes], proofs: list[bytes]) -> list[int]:
        return self.tiny_verify(suite, public_keys, inputs, ads, proofs, thin=True)

    def tiny_verify(self, suite: VrfSuiteStruct, public_keys: list[bytes], inputs: list[bytes], ads: list[bytes], proofs: list[bytes], thin: bool = False) -> list[int]:
        n = len(proofs)
        size = 96 if thin else 80
        if any(len(p) != size for p in proofs):
            raise ValueError(f"invalid {'Thin' if thin else 'Tiny'} VRF proof length: expected {size}")
        if len(public_keys) != n or any(len(k) != 32 for k in public_keys):
            raise ValueError("public keys must be 32 bytes, one per proof")
        blob, a, b, c, d = pack_items(inputs, ads)
        out = ctypes.create_string_buffer(max(n, 1))
        fn = self.library.lib.dr_thin_verify_batch if thin else self.library.lib.dr_tiny_verify_batch
        self.library.check(fn(self.handle, ctypes.byref(suite), n, blob, a, b, c, d, b"".join(public_keys), b"".join(proofs), out))
        return list(out.raw[:n])

    def vrf_prove(self, scheme: str, suite: VrfSuiteStruct, inputs: list[bytes], ads: list[bytes], secret_keys: list[bytes]) -> list[bytes]:
        """Batched `PedersenVRF.prove` ('pedersen', 192-byte proofs) / `TinyVRF.prove` ('tiny', 80 bytes)."""
        n = len(inputs)
        if len(secret_keys) != n or any(len(k) != 32 for k in secret_keys):
            raise ValueError("secret keys must be 32 bytes, one per item")
        size = {"pedersen": 192, "tiny": 80, "thin": 96}[scheme]
        fn = {"pedersen": self.library.lib.dr_pedersen_prove_batch, "tiny": self.library.lib.dr_tiny_prove_batch, "thin": self.library.lib.dr_thin_prove_batch}[scheme]
        blob, a, b, c, d = pack_items(inputs, ads)
        out = ctypes.create_string_buffer(size * max(n, 1))
        self.library.check(fn(self.handle, ctypes.byref(suite), n, blob, a, b, c, d, b"".join(secret_keys), out))
        raw = out.raw
        return [raw[size * i : size * i + size] for i in range(n)]

    def pedersen_prove_with_blinding(self, suite: VrfSuiteStruct, inputs: list[bytes], ads: list[bytes], secret_keys: list[bytes]):
        """(192-byte proofs, blinding factors) -- `PedersenVRF.prove` keeping `_blinding_factor`."""
        n = len(inputs)
        if len(secret_keys) != n or any(len(k) != 32 for k in secret_keys):
            raise ValueError("secret keys must be 32 bytes, one per item")
        blob, a, b, c, d = pack_items(inputs, ads)
        out = ctypes.create_string_buffer(192 * max(n, 1))
        bl = ctypes.create_string_buffer(32 * max(n, 1))
        self.library.check(self.library.lib.dr_pedersen_prove_batch_ex(self.handle, ctypes.byref(suite), n, blob, a, b, c, d, b"".join(secret_keys), out, bl))
        raw, braw = out.raw, bl.raw
        return [raw[192 * i : 192 * i + 192] for i in range(n)], [int.from_bytes(braw[32 * i : 32 * i + 32], "little") for i in range(n)]

    def ring_proof_verify(self, key: VerifierKeyStruct, relations: list[tuple[int, int]], payloads: list[bytes], coeffs: list[int], aggregate: bool = False):
        """`Verify(...).is_valid()` for a batch under an explicit verifier key -> (verdicts, all_ok)."""
        n = len(payloads)
        if any(len(p) != 592 for p in payloads) or len(relations) != n or len(coeffs) != 2 * n:
            raise ValueError("bad ring-proof verification batch")
        out = ctypes.create_string_buffer(max(n, 1))
        all_ok = c_int(0)
        self.library.check(
            self.library.lib.dr_ring_proof_verify_batch(
                self.handle, ctypes.byref(key), n, b"".join(_xy64(r) for r in relations), b"".join(payloads),
                b"".join(int(v).to_bytes(32, "little") for v in coeffs), 1 if aggregate else 0, out, ctypes.byref(all_ok),
            )
        )
        return list(out.raw[:n]), bool(all_ok.value)

    def pairing_check(self, a1_be96: bytes, b1_be192: bytes, a2_be96: bytes, b2_be192: bytes) -> list[bool]:
        """[e(a1_i, b1_i) == e(a2_i, b2_i)] for concatenated uncompressed encodings (pairing.py:24-31)."""
        n = len(a1_be96) // 96
        if not (len(a2_be96) == 96 * n and len(b1_be192) == 192 * n and len(b2_be192) == 192 * n):
            raise ValueError("mismatched pairing operand lengths")
        out = ctypes.create_string_buffer(max(n, 1))
        self.library.check(self.library.lib.dr_pairing_check_batch(self.handle, a1_be96, b1_be192, a2_be96, b2_be192, n, out))
        return [bool(b) for b in out.raw[:n]]

    def te_msm(self, points: list[bytes], scalars: list[int]) -> bytes:
        """`BandersnatchPoint.msm`: sum_i k_i * P_i on 32-byte encodings (ValueError on an undecodable point)."""
        if len(points) != len(scalars) or any(len(p) != 32 for p in points):
            raise ValueError("points and scalars must have the same length; points are 32 bytes")
        out = ctypes.create_string_buffer(32)
        ks = b"".join((int(k) % BANDERSNATCH_ORDER).to_bytes(32, "little") for k in scalars)
        self.library.check(self.library.lib.dr_te_msm(self.handle, b"".join(points), ks, len(points), out))
        return out.raw

    def g1_msm(self, points_be96: bytes, scalars: list[int]) -> bytes:
        """`KZG.msm_g1` (kzg.py:147-149) over arbitrary points: 96-byte uncompressed result."""
        count = len(points_be96) // 96
        if isinstance(scalars, (bytes, bytearray)):  # already 32-byte little-endian each
            ks = bytes(scalars)
            if len(ks) != 32 * count:
                raise ValueError("points and scalars must have the same length")
        else:
            if len(scalars) != count:
                raise ValueError("points and scalars must have the same length")
            ks = b"".join((int(k) % FR_MODULUS).to_bytes(32, "little") for k in scalars)
        out = ctypes.create_string_buffer(96)
        self.library.check(self.library.lib.dr_g1_msm(self.handle, points_be96, ks, count, out))
        return out.raw

    def g1_synthetic_srs(self, tau: int, offset: int, n: int) -> bytes:
        """n x 96 bytes: tau^(offset + i) * G."""
        out = ctypes.create_string_buffer(96 * max(n, 1))
        self.library.check(self.library.lib.dr_g1_synthetic_srs(self.handle, int(tau).to_bytes(32, "little"), offset, n, out))
        return out.raw[: 96 * n]

    def fr_ntt_bench(self, n: int, batch: int, iters: int, omega: int) -> tuple[float, int]:
        """(ms per batched forward transform, first output element) with operands resident on the device."""
        ms = c_float()
        first = ctypes.create_string_buffer(32)
        self.library.check(self.library.lib.dr_fr_ntt_bench(self.handle, n, batch, iters, int(omega).to_bytes(32, "little"), ctypes.byref(ms), first))
        return float(ms.value), int.from_bytes(first.raw, "little")

    def g1_msm_bench(self, n: int, iters: int, seed: int, distribution: int, tau: int) -> tuple[float, int, bytes]:
        """(ms per MSM, window bits, result) of an n-point MSM over the synthetic SRS tau^i * G, operands on the device."""
        ms, c = c_float(), ctypes.c_uint32()
        out = ctypes.create_string_buffer(96)
        self.library.check(
            self.library.lib.dr_g1_msm_bench(self.handle, n, iters, seed, distribution, int(tau).to_bytes(32, "little"), ctypes.byref(ms), ctypes.byref(c), out)
        )
        return float(ms.value), int(c.value), out.raw

    def g1_compress(self, points_be96: bytes) -> bytes:
        count = len(points_be96) // 96
        out = ctypes.create_string_buffer(48 * count)
        self.library.check(self.library.lib.dr_g1_compress(self.handle, points_be96, count, out))
        return out.raw

    def g1_decompress(self, points_be48: bytes) -> tuple[bytes, bytes]:
        count = len(points_be48) // 48
        out = ctypes.create_string_buffer(96 * count)
        ok = ctypes.create_string_buffer(count)
        self.library.check(self.library.lib.dr_g1_decompress(self.handle, points_be48, count, out, ok))
        return out.raw, ok.raw


class NativeSrs:
    """dr_srs: SRS points + fixed-base window table resident on the device."""

    def __init__(self, ctx: Context, g1_be96: bytes, g2_be192: bytes, window_bits: int = 0, wide_windows: int = 0, glv: bool = False):
        self.ctx = ctx
        self.handle = c_void_p()
        n = len(g1_be96) // 96
        if len(g2_be192) != 384:
            raise ValueError("expected two 192-byte G2 points")
        lib = ctx.library
        if not 0 <= window_bits < 256 or not 0 <= wide_windows < 256 or ((wide_windows or glv) and not window_bits):
            raise ValueError("bad window geometry")
        lib.check(lib.lib.dr_srs_load(ctx.handle, g1_be96, n, g2_be192, window_bits | (wide_windows << 8) | (int(bool(glv)) << 16), ctypes.byref(self.handle)))
        self.size = n

    def close(self) -> None:
        if self.handle:
            self.ctx.library.lib.dr_srs_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def geometry(self) -> tuple[int, int, int, int]:
        """(window bits c, number of (c + 1)-bit windows, GLV split 0 / 1, table additions per coefficient)."""
        c, k, g, a = c_uint32(), c_uint32(), c_uint32(), c_uint32()
        self.ctx.library.lib.dr_srs_geometry(self.handle, ctypes.byref(c), ctypes.byref(k), ctypes.byref(g), ctypes.byref(a))
        return c.value, k.value, g.value, a.value

    @property
    def table_bytes(self) -> int:
        return int(self.ctx.library.lib.dr_srs_table_bytes(self.handle))

    def commit(self, coeff_vectors: list[list[int]]) -> list[bytes]:
        """KZG.commit for a batch of equal-length coefficient vectors -> 96-byte uncompressed points."""
        if not coeff_vectors:
            return []
        n = len(coeff_vectors[0])
        if any(len(v) != n for v in coeff_vectors):
            raise ValueError("all coefficient vectors in a batch must have the same length")
        batch = len(coeff_vectors)
        out = ctypes.create_string_buffer(96 * batch)
        data = b"".join((int(c) % FR_MODULUS).to_bytes(32, "little") for v in coeff_vectors for c in v)
        lib = self.ctx.library
        lib.check(lib.lib.dr_kzg_commit(self.ctx.handle, self.handle, data, n, batch, out))
        raw = out.raw
        return [raw[96 * i : 96 * i + 96] for i in range(batch)]

    def open(self, coeff_vectors: list[list[int]], points: list[int]) -> list[tuple[bytes, int]]:
        """KZG.open for a batch of equal-length coefficient vectors: [(proof 96 bytes, value)]."""
        if not coeff_vectors:
            return []
        n, batch = len(coeff_vectors[0]), len(coeff_vectors)
        if any(len(v) != n for v in coeff_vectors) or len(points) != batch:
            raise ValueError("all coefficient vectors in a batch must have the same length, one point per vector")
        proofs, values = ctypes.create_string_buffer(96 * batch), ctypes.create_string_buffer(32 * batch)
        data = b"".join((int(c) % FR_MODULUS).to_bytes(32, "little") for v in coeff_vectors for c in v)
        xs = b"".join((int(x) % FR_MODULUS).to_bytes(32, "little") for x in points)
        lib = self.ctx.library
        lib.check(lib.lib.dr_kzg_open(self.ctx.handle, self.handle, data, n, batch, xs, proofs, values))
        return [(proofs.raw[96 * i : 96 * i + 96], int.from_bytes(values.raw[32 * i : 32 * i + 32], "little")) for i in range(batch)]

    def pairing_check(self, lhs_points: list[bytes], lhs_scalars: list[int], rhs_points: list[bytes], rhs_scalars: list[int]) -> bool:
        """e(sum lhs_scalars[i] * lhs_points[i], [1]_2) == e(sum rhs_scalars[j] * rhs_points[j], [tau]_2)  (pcs/kzg.py:194-338)."""
        if len(lhs_points) != len(lhs_scalars) or len(rhs_points) != len(rhs_scalars):
            raise ValueError("points and scalars must have the same length")
        if any(len(p) != 96 for p in lhs_points) or any(len(p) != 96 for p in rhs_points):
            raise ValueError("expected 96-byte uncompressed G1 points")
        le = lambda ks: b"".join((int(k) % FR_MODULUS).to_bytes(32, "little") for k in ks)  # noqa: E731
        ok = c_int(0)
        lib = self.ctx.library
        lib.check(lib.lib.dr_kzg_pairing_check(self.ctx.handle, self.handle, b"".join(lhs_points) or None, le(lhs_scalars) or None, len(lhs_points),
                                               b"".join(rhs_points) or None, le(rhs_scalars) or None, len(rhs_points), ctypes.byref(ok)))
        return bool(ok.value)

    def commit_bench(self, n: int, batch: int, iters: int, seed: int = 1) -> tuple[float, bytes]:
        ms = c_float()
        first = ctypes.create_string_buffer(96)
        lib = self.ctx.library
        lib.check(lib.lib.dr_kzg_commit_bench(self.ctx.handle, self.handle, n, batch, iters, seed, ctypes.byref(ms), first))
        return float(ms.value), first.raw


class RingParamsStruct(ctypes.Structure):
    """dr_ring_params (include/dot_ring_b200.h)."""

    _fields_ = [
        ("domain_size", ctypes.c_uint32),
        ("max_ring_size", ctypes.c_uint32),
        ("padding_rows", ctypes.c_uint32),
        ("suite_id_len", ctypes.c_uint32),
        ("h2c_dst_len", ctypes.c_uint32),
        ("hash_id", ctypes.c_uint32),
        ("omega", c_uint8 * 32),
        ("radix_omega", c_uint8 * 32),
        ("seed", c_uint8 * 64),
        ("blinding_base", c_uint8 * 64),
        ("padding_point", c_uint8 * 64),
        ("generator", c_uint8 * 64),
        ("suite_id", c_uint8 * 32),
        ("h2c_dst", c_uint8 * 64),
    ]


def make_ring_params(*, domain_size: int, omega: int, seed, blinding_base, generator, suite_id: bytes, h2c_dst: bytes, hash_name: str = "sha512", max_ring_size: int = 0,
                     padding_rows: int = 0, radix_omega: int = 0, padding_point=(0, 0)) -> RingParamsStruct:
    p = RingParamsStruct()
    p.domain_size, p.max_ring_size, p.padding_rows = domain_size, max_ring_size, padding_rows
    p.suite_id_len, p.h2c_dst_len = len(suite_id), len(h2c_dst)
    p.hash_id = HASH_IDS[hash_name]
    _put(p.omega, int(omega).to_bytes(32, "little"))
    _put(p.radix_omega, int(radix_omega).to_bytes(32, "little"))
    _put(p.seed, _xy64(seed))
    _put(p.blinding_base, _xy64(blinding_base))
    _put(p.padding_point, _xy64(padding_point))
    _put(p.generator, _xy64(generator))
    _put(p.suite_id, suite_id)
    _put(p.h2c_dst, h2c_dst)
    return p


def ring_roots_from_keys(srs: NativeSrs, params: RingParamsStruct, key_sets: list[list[bytes]]) -> list[bytes]:
    """dr_ring_roots_from_keys: the 144-byte root of every key set (32-byte keys), all under one params, in one call."""
    if any(len(k) != 32 for keys in key_sets for k in keys):
        raise ValueError("ring keys must be 32 bytes")
    n = len(key_sets)
    counts = np.array([len(keys) for keys in key_sets] or [0], dtype=np.int64)
    if counts.max() >> 32:
        raise ValueError("ring size exceeds max supported size")
    blob = b"".join(k for keys in key_sets for k in keys)
    out = ctypes.create_string_buffer(144 * max(n, 1))
    lib = srs.ctx.library
    lib.check(lib.lib.dr_ring_roots_from_keys(srs.ctx.handle, srs.handle, ctypes.byref(params), n, blob or None, np.ctypeslib.as_ctypes(counts.astype(np.uint32)), out))
    return [out.raw[144 * i : 144 * i + 144] for i in range(n)]


def ring_root_update(srs: NativeSrs, params: RingParamsStruct, root144: bytes, rows: list[int], new_keys: list[bytes], old_keys: list[bytes] | None = None) -> bytes:
    """dr_ring_root_update: the root after row rows[j] went from old_keys[j] (None: padding everywhere) to new_keys[j]."""
    n = len(rows)
    if len(root144) != 144:
        raise ValueError(f"invalid ring root length: ring root must be exactly 144 bytes, got {len(root144)}")
    if len(new_keys) != n or (old_keys is not None and len(old_keys) != n):
        raise ValueError("one new key (and one old key, when given) per row is required")
    if any(len(k) != 32 for k in list(new_keys) + list(old_keys or [])):
        raise ValueError("ring keys must be 32 bytes")
    if any(not 0 <= int(r) < 1 << 32 for r in rows):
        raise ValueError("row out of range")
    out = ctypes.create_string_buffer(144)
    idx = np.ctypeslib.as_ctypes(np.array([int(r) for r in rows] or [0], dtype=np.uint32))
    lib = srs.ctx.library
    lib.check(lib.lib.dr_ring_root_update(srs.ctx.handle, srs.handle, ctypes.byref(params), bytes(root144), n, idx, b"".join(old_keys) if old_keys is not None else None,
                                          b"".join(new_keys) or None, out))
    return out.raw


class NativeRing:
    """dr_ring: decoded keys, fixed columns (coefficients + 4x LDE), ring root, transcript prefix."""

    def __init__(self, srs: NativeSrs, keys: list[bytes], *, domain_size: int, max_ring_size: int, padding_rows: int, omega: int, radix_omega: int,
                 seed, blinding_base, padding_point, generator, suite_id: bytes, h2c_dst: bytes, hash_name: str = "sha512"):
        self.srs = srs
        self.ctx = srs.ctx
        p = make_ring_params(domain_size=domain_size, max_ring_size=max_ring_size, padding_rows=padding_rows, omega=omega, radix_omega=radix_omega, seed=seed,
                             blinding_base=blinding_base, padding_point=padding_point, generator=generator, suite_id=suite_id, h2c_dst=h2c_dst, hash_name=hash_name)
        for key in keys:
            if len(key) != 32:
                raise ValueError("ring keys must be 32 bytes")
        self.handle = c_void_p()
        self.domain_size = domain_size
        self.time_calls = False
        self.last_call_ms = 0.0
        lib = self.ctx.library
        lib.check(lib.lib.dr_ring_create(self.ctx.handle, srs.handle, ctypes.byref(p), b"".join(keys), len(keys), ctypes.byref(self.handle)))

    def close(self) -> None:
        if self.handle:
            self.ctx.library.lib.dr_ring_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def root(self) -> bytes:
        out = ctypes.create_string_buffer(144)
        self.ctx.library.check(self.ctx.library.lib.dr_ring_root(self.handle, out))
        return out.raw

    def fixed_commitments(self) -> bytes:
        out = ctypes.create_string_buffer(288)
        self.ctx.library.check(self.ctx.library.lib.dr_ring_fixed_commitments(self.handle, out))
        return out.raw

    def points(self) -> list[tuple[int, int]]:
        n = self.domain_size
        out = ctypes.create_string_buffer(64 * n)
        self.ctx.library.check(self.ctx.library.lib.dr_ring_points(self.handle, out, n))
        raw = out.raw
        return [(int.from_bytes(raw[64 * i : 64 * i + 32], "little"), int.from_bytes(raw[64 * i + 32 : 64 * i + 64], "little")) for i in range(n)]

    @staticmethod
    def pack_prove_inputs(alphas: list[bytes], ads: list[bytes], secret_keys: list[bytes], producer_index: list[int], zk_rows=None, ring_index=None) -> dict:
        """Host-side packing of a prove batch into the flat buffers of dr_ring_prove_batch (done once per batch, also when the batch
        is then sharded over several devices: the offsets are absolute, so a shard is just a sub-range of every array).
        `ring_index` (dr_ring_prove_multi): the ring of every item, an index into the call's list of rings."""
        n = len(alphas)
        if not (len(ads) == len(secret_keys) == len(producer_index) == n) or (ring_index is not None and len(ring_index) != n):
            raise ValueError("batch inputs must have equal length")
        blob, a_off, a_len, d_off, d_len = pack_items(alphas, ads)
        rows = np.ctypeslib.as_ctypes(np.array(producer_index if n else [0], dtype=np.uint32))
        ring = None if ring_index is None else NativeRing._pack_ring_index(ring_index, n)
        return {"n": n, "blob": blob, "a_off": a_off, "a_len": a_len, "d_off": d_off, "d_len": d_len, "sk": b"".join(secret_keys), "rows": rows,
                "zk": NativeRing._pack_zk_rows(zk_rows, n), "ring": ring, "proofs": ctypes.create_string_buffer(784 * max(n, 1)),
                "status": (ctypes.c_uint32 * max(n, 1))()}

    @staticmethod
    def _pack_zk_rows(zk_rows, n: int) -> bytes | None:
        """12 blinding rows per proof as 32-byte little-endian values (None: zeros)."""
        if isinstance(zk_rows, (bytes, bytearray)):  # already 12 x 32-byte little-endian values per proof
            if len(zk_rows) != 12 * 32 * n:
                raise ValueError("zk_rows must hold 12 field elements per proof")
            return bytes(zk_rows)
        if zk_rows is not None:
            if len(zk_rows) != 12 * n:
                raise ValueError("zk_rows must hold 12 field elements per proof")
            return b"".join(int(v).to_bytes(32, "little") for v in zk_rows)
        return None

    @staticmethod
    def _pack_ring_index(ring_index, n: int):
        idx = np.array(ring_index if n else [0], dtype=np.int64)
        if idx.min() < 0 or idx.max() >> 32:
            raise ValueError("ring index out of range")
        return np.ctypeslib.as_ctypes(idx.astype(np.uint32))

    @staticmethod
    def _packed_args(pk: dict, lo: int, hi: int) -> list:
        """The batch arguments (blob ... status) of items [lo, hi) of a packed batch, as dr_ring_prove_batch / _multi take them."""
        u32 = lambda arr: ctypes.byref(arr, 4 * lo)  # noqa: E731
        sk = (ctypes.c_char * (32 * (hi - lo))).from_buffer_copy(pk["sk"], 32 * lo) if lo or hi != pk["n"] else pk["sk"]
        zk = None if pk["zk"] is None else (pk["zk"] if not lo and hi == pk["n"] else (ctypes.c_char * (384 * (hi - lo))).from_buffer_copy(pk["zk"], 384 * lo))
        return [pk["blob"], u32(pk["a_off"]), u32(pk["a_len"]), u32(pk["d_off"]), u32(pk["d_len"]), sk, u32(pk["rows"]), zk, ctypes.byref(pk["proofs"], 784 * lo),
                ctypes.byref(pk["status"], 4 * lo)]

    def prove_packed(self, pk: dict, lo: int = 0, hi: int | None = None) -> None:
        """Prove items [lo, hi) of a packed batch; proofs and status words land in the batch's own output buffers."""
        hi = pk["n"] if hi is None else hi
        if hi <= lo:
            return
        args = self._packed_args(pk, lo, hi)
        lib = self.ctx.library
        if self.time_calls:  # one CUDA event pair on the ctx stream around the whole call (bench.py); every argument is ready by now
            self.ctx.timer_start()
        lib.check(lib.lib.dr_ring_prove_batch(self.ctx.handle, self.handle, hi - lo, *args))
        if self.time_calls:
            self.last_call_ms = self.ctx.timer_stop()

    @staticmethod
    def prove_multi_packed(rings: list["NativeRing"], pk: dict, lo: int = 0, hi: int | None = None) -> None:
        """dr_ring_prove_multi over items [lo, hi) of a batch packed with a ring-index column (indices into `rings`)."""
        hi = pk["n"] if hi is None else hi
        if hi <= lo:
            return
        if not rings:
            raise ValueError("at least one ring is required")
        ctx = rings[0].ctx
        handles = (c_void_p * len(rings))(*[r.handle for r in rings])
        ctx.library.check(ctx.library.lib.dr_ring_prove_multi(ctx.handle, handles, len(rings), ctypes.byref(pk["ring"], 4 * lo), hi - lo, *NativeRing._packed_args(pk, lo, hi)))

    @staticmethod
    def prove_multi(rings: list["NativeRing"], index: list[int], alphas: list[bytes], ads: list[bytes], secret_keys: list[bytes], producer_index: list[int],
                    zk_rows=None):
        """Item i against rings[index[i]] in one call (dr_ring_prove_multi) -> (list of 784-byte proofs, list of status words)."""
        pk = NativeRing.pack_prove_inputs(alphas, ads, secret_keys, producer_index, zk_rows, ring_index=index)
        NativeRing.prove_multi_packed(rings, pk)
        return NativeRing.unpack_proofs(pk)

    @staticmethod
    def pack_ring_proof_inputs(index: list[int], producer_index: list[int], blindings: list[int], zk_rows=None, label: bytes | None = None) -> dict:
        """Host-side packing of a bare ring-proof batch (dr_ring_proof_prove_multi), once per batch: a shard is a sub-range of every array."""
        n = len(index)
        if not (len(producer_index) == len(blindings) == n):
            raise ValueError("batch inputs must have equal length")
        if any(int(t) < 0 or int(t) >> 256 for t in blindings):
            raise ValueError("blinding factor out of range")
        rows = np.array(producer_index if n else [0], dtype=np.int64)
        if rows.min() < 0 or rows.max() >> 32:
            raise ValueError("producer row out of range")
        label = b"" if label is None else bytes(label)
        return {"n": n, "ring": NativeRing._pack_ring_index(index, n), "rows": np.ctypeslib.as_ctypes(rows.astype(np.uint32)),
                "t": b"".join(int(t).to_bytes(32, "little") for t in blindings), "zk": NativeRing._pack_zk_rows(zk_rows, n), "label": label,
                "relations": ctypes.create_string_buffer(64 * max(n, 1)), "payloads": ctypes.create_string_buffer(592 * max(n, 1))}

    @staticmethod
    def proof_prove_multi_packed(rings: list["NativeRing"], pk: dict, lo: int = 0, hi: int | None = None) -> None:
        """dr_ring_proof_prove_multi over items [lo, hi) of a packed bare ring-proof batch."""
        hi = pk["n"] if hi is None else hi
        if hi <= lo:
            return
        if not rings:
            raise ValueError("at least one ring is required")
        ctx = rings[0].ctx
        handles = (c_void_p * len(rings))(*[r.handle for r in rings])
        t = (ctypes.c_char * (32 * (hi - lo))).from_buffer_copy(pk["t"], 32 * lo)
        zk = None if pk["zk"] is None else (ctypes.c_char * (384 * (hi - lo))).from_buffer_copy(pk["zk"], 384 * lo)
        label = pk["label"]
        ctx.library.check(
            ctx.library.lib.dr_ring_proof_prove_multi(
                ctx.handle, handles, len(rings), ctypes.byref(pk["ring"], 4 * lo), hi - lo, ctypes.byref(pk["rows"], 4 * lo), t, zk, label or None, len(label),
                ctypes.byref(pk["relations"], 64 * lo), ctypes.byref(pk["payloads"], 592 * lo),
            )
        )
        ctypes.memset(t, 0, ctypes.sizeof(t))

    @staticmethod
    def unpack_ring_proofs(pk: dict):
        """-> (relations as (x, y), 592-byte payloads)."""
        n, rel, pay = pk["n"], pk["relations"].raw, pk["payloads"].raw
        relations = [(int.from_bytes(rel[64 * i : 64 * i + 32], "little"), int.from_bytes(rel[64 * i + 32 : 64 * i + 64], "little")) for i in range(n)]
        return relations, [pay[592 * i : 592 * i + 592] for i in range(n)]

    @staticmethod
    def proof_prove_multi(rings: list["NativeRing"], index: list[int], producer_index: list[int], blindings: list[int], zk_rows=None, label: bytes | None = None):
        """Bare ring proofs (RingProofBuilder.build): item i proves row producer_index[i] of rings[index[i]] with blinding factor blindings[i],
        under `label` (None: the suite id) -> (relations PK_k + t * B as (x, y), 592-byte payloads)."""
        pk = NativeRing.pack_ring_proof_inputs(index, producer_index, blindings, zk_rows, label)
        NativeRing.proof_prove_multi_packed(rings, pk)
        return NativeRing.unpack_ring_proofs(pk)

    @staticmethod
    def unpack_proofs(pk: dict):
        n, raw = pk["n"], pk["proofs"].raw
        return [raw[784 * i : 784 * i + 784] for i in range(n)], pk["status"][:n]

    def prove_batch(self, alphas: list[bytes], ads: list[bytes], secret_keys: list[bytes], producer_index: list[int], zk_rows: list[int] | None = None):
        """-> (list of 784-byte proofs, list of status words)."""
        pk = self.pack_prove_inputs(alphas, ads, secret_keys, producer_index, zk_rows)
        self.prove_packed(pk)
        return self.unpack_proofs(pk)

    def verify_batch(self, inputs: list[bytes], ads: list[bytes], proofs: list[bytes], coeffs: list[int], aggregate: bool = False):
        """RingVRF decode + verify for 784-byte proofs -> (per-item verdicts 1 / 0 / 2, all_ok)."""
        n = len(proofs)
        if any(len(p) != 784 for p in proofs):
            raise ValueError("invalid Ring VRF proof length: Ring VRF proof must be exactly 784 bytes")
        if len(coeffs) != 2 * n:
            raise ValueError("two batching coefficients per proof are required")
        blob, a, b, c, d = pack_items(inputs, ads)
        out = ctypes.create_string_buffer(max(n, 1))
        all_ok = c_int(0)
        lib = self.ctx.library
        lib.check(
            lib.lib.dr_ring_verify_batch(
                self.ctx.handle, self.handle, n, blob, a, b, c, d, b"".join(proofs), b"".join(int(v).to_bytes(32, "little") for v in coeffs),
                1 if aggregate else 0, out, ctypes.byref(all_ok),
            )
        )
        return list(out.raw[:n]), bool(all_ok.value)

    def witness_table_bits(self) -> int:
        return int(self.ctx.library.lib.dr_ring_witness_table_bits(self.handle))

    def commit_kernel_ms(self) -> tuple[float, int]:
        """(device ms, launches) of the dense commit kernel `CommitBodyT` within the last prove call (CUDA events around the launches)."""
        ms, n = c_float(), c_uint32()
        self.ctx.library.check(self.ctx.library.lib.dr_ring_prove_commit_kernel_ms(self.ctx.handle, ctypes.byref(ms), ctypes.byref(n)))
        return float(ms.value), int(n.value)

    def prove_phase_ms(self) -> list[float]:
        arr = (c_float * 6)()
        self.ctx.library.check(self.ctx.library.lib.dr_ring_prove_phase_ms(self.ctx.handle, ctypes.byref(arr)))
        return [float(x) for x in arr]


class NativeRingVerifier:
    """dr_ring_verifier: the verifier key of one ring built from its 144-byte root alone (no keys, no SRS window table)."""

    def __init__(self, ctx: Context, root144: bytes, g1_0_be96: bytes, g2_be192: bytes, *, domain_size: int, omega: int, seed, blinding_base, generator,
                 suite_id: bytes, h2c_dst: bytes, hash_name: str = "sha512"):
        if len(root144) != 144:
            raise ValueError(f"invalid ring root length: ring root must be exactly 144 bytes, got {len(root144)}")
        if len(g1_0_be96) != 96 or len(g2_be192) != 384:
            raise ValueError("expected [1]_1 (96 bytes) and [1]_2 | [tau]_2 (384 bytes)")
        self.ctx = ctx
        self.domain_size = domain_size
        self.handle = c_void_p()
        p = make_ring_params(domain_size=domain_size, omega=omega, seed=seed, blinding_base=blinding_base, generator=generator, suite_id=suite_id, h2c_dst=h2c_dst,
                             hash_name=hash_name)
        lib = ctx.library
        lib.check(lib.lib.dr_ring_verifier_create(ctx.handle, ctypes.byref(p), bytes(g1_0_be96), bytes(g2_be192), bytes(root144), ctypes.byref(self.handle)))

    def close(self) -> None:
        if self.handle:
            self.ctx.library.lib.dr_ring_verifier_destroy(self.handle)
            self.handle = c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def verify_multi(verifiers: list["NativeRingVerifier"], index: list[int], inputs: list[bytes], ads: list[bytes], proofs: list[bytes], coeffs: list[int],
                     aggregate: bool = False):
        """Item i against verifiers[index[i]] (one call, one context) -> (per-item verdicts 1 / 0 / 2, all_ok); aggregate folds every item
        into one pairing check."""
        n = len(proofs)
        if not verifiers:
            raise ValueError("at least one ring verifier is required")
        if any(len(p) != 784 for p in proofs):
            raise ValueError("invalid Ring VRF proof length: Ring VRF proof must be exactly 784 bytes")
        if len(coeffs) != 2 * n or len(index) != n:
            raise ValueError("one ring index and two batching coefficients per proof are required")
        if any(not 0 <= int(k) < len(verifiers) for k in index):
            raise ValueError("ring index out of range")
        ctx = verifiers[0].ctx
        blob, a, b, c, d = pack_items(inputs, ads)
        handles = (c_void_p * len(verifiers))(*[v.handle for v in verifiers])
        idx = np.ctypeslib.as_ctypes(np.array(index if n else [0], dtype=np.uint32))
        out = ctypes.create_string_buffer(max(n, 1))
        all_ok = c_int(0)
        lib = ctx.library
        lib.check(
            lib.lib.dr_ring_verify_multi(
                ctx.handle, handles, len(verifiers), idx, n, blob, a, b, c, d, b"".join(proofs), b"".join(int(v).to_bytes(32, "little") for v in coeffs),
                1 if aggregate else 0, out, ctypes.byref(all_ok),
            )
        )
        return list(out.raw[:n]), bool(all_ok.value)
