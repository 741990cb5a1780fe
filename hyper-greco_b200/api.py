"""ctypes harness over the C ABI (include/hg_b200.h). It plays the role of the Rust caller in this container
(no Rust toolchain here, SURVEY.md F2): same object names and call order as the reference

    LassoPreprocessing::preprocess      /root/reference/lasso/src/lasso.rs:527-627
    LassoNode::new / prove_claim_reduction   /root/reference/lasso/src/lasso.rs:143-154, :57-114
    Keccak256Transcript                 /root/reference/bfv-gkr/src/transcript.rs:117-203

There is NO CPU fallback: if the CUDA library is missing or no GPU is present every compute call raises.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

GOLDILOCKS, BN254 = 0, 1
MODE_PREFETCH, MODE_INTERACTIVE = 0, 1
OPT_A3_WIRE, OPT_A3_H1, OPT_A5_ASCENDING = 3, 31, 5
LIMBS = {GOLDILOCKS: 1, BN254: 4}
DEGREE = {GOLDILOCKS: 2, BN254: 1}
GL_P = 2**64 - 2**32 + 1                                                          # Goldilocks prime
BN_R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001  # BN254 scalar field order

# every symbol include/hg_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "hg_last_error", "hg_version", "hg_ctx_create", "hg_ctx_destroy", "hg_ctx_set_option", "hg_ctx_synchronize", "hg_ctx_launch_count",
    "hg_ctx_stream", "hg_ctx_profile", "hg_ctx_profile_read", "hg_kernel_class_count", "hg_kernel_class_name", "hg_buf_alloc", "hg_buf_upload", "hg_buf_upload_async", "hg_buf_download", "hg_device_download", "hg_buf_device_ptr", "hg_buf_size", "hg_buf_free", "hg_field_base_bytes", "hg_field_encode", "hg_field_decode",
    "hg_transcript_new", "hg_transcript_from_proof", "hg_transcript_from_callbacks", "hg_transcript_free", "hg_transcript_squeeze_challenge", "hg_transcript_squeeze_challenges", "hg_transcript_write_felt_ext",
    "hg_transcript_read_felt_ext", "hg_transcript_proof_len", "hg_transcript_proof_copy", "hg_transcript_num_squeezed",
    "hg_lasso_preprocess", "hg_lasso_preprocess_lookups", "hg_lasso_pp_lookup_index_by_id", "hg_lasso_node_new_ids", "hg_lasso_pp_free", "hg_lasso_pp_num_lookups", "hg_lasso_pp_num_subtables", "hg_lasso_pp_num_memories",
    "hg_lasso_pp_lookup_index", "hg_lasso_pp_memory_maps", "hg_lasso_pp_subtable_id", "hg_lasso_node_new", "hg_lasso_node_free",
    "hg_lasso_node_log2_input_size", "hg_lasso_node_device_bytes", "hg_lasso_node_prove", "hg_lasso_node_download_polys",
    "hg_lasso_node_num_chunks", "hg_lasso_node_timing", "hg_lasso_node_shard_words", "hg_lasso_node_prove_shard", "hg_lasso_node_emit_shard",
    "hg_shard_merge", "hg_lasso_node_prove_shard_dev", "hg_lasso_node_emit_shard_dev", "hg_shard_merge_device", "hg_gkr_shard_words", "hg_gkr_prove_shard_dev", "hg_gkr_emit_shard_dev", "hg_gkr_emit_shard_part_dev", "hg_transcript_append_bytes",
    "hg_circuit_new_host", "hg_circuit_insert_lasso_host", "hg_gkr_verify", "hg_mle_eval_host", "hg_bfv_witness_generate", "hg_lasso_node_verify", "hg_sumcheck_prove", "hg_mle_eval_batch", "hg_ntt", "hg_bfv_configure", "hg_field_selftest",
    "hg_bfv_pk_configure", "hg_bfv_pk_witness_generate",
    "hg_circuit_new", "hg_circuit_free", "hg_circuit_insert_input", "hg_circuit_insert_fft", "hg_circuit_insert_lasso", "hg_circuit_insert_vanilla",
    "hg_circuit_connect", "hg_circuit_evaluate", "hg_circuit_evaluate_host", "hg_circuit_node_value", "hg_gkr_prove", "hg_gkr_timing", "hg_gkr_num_challenges", "hg_gkr_num_inputs", "hg_gkr_num_input_claims",
    "hg_gkr_input_claim_num_vars", "hg_gkr_input_claim", "hg_verifier_new", "hg_verifier_free", "hg_gkr_verify_batch", "hg_verifier_reason", "hg_mle_eval_multi",
    "hg_verifier_num_inputs", "hg_verifier_input_len", "hg_verifier_timing",
]

# callback types of hg_transcript_from_callbacks (include/hg_b200.h)
SQUEEZE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64))
WRITE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64))
READ_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64))

_lib = None


class HgError(RuntimeError):
    pass


def lib():
    """Loads hyper-greco_b200/lib/libhg_b200.so (built by build.py). Raises if it is missing: no fallback."""
    global _lib
    if _lib is None:
        path = _build.LIB
        if not os.path.exists(path):
            raise HgError(f"{path} is missing: run __graft_entry__.build() (nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(path)
        vp, sz, i32, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
        L.hg_last_error.restype = C.c_char_p
        L.hg_ctx_create.argtypes = [i32, i32, C.POINTER(vp)]
        L.hg_ctx_destroy.argtypes = [vp]
        L.hg_ctx_set_option.argtypes = [vp, i32, i32]
        L.hg_ctx_synchronize.argtypes = [vp]
        L.hg_ctx_launch_count.argtypes = [vp]
        L.hg_ctx_launch_count.restype = u64
        L.hg_ctx_profile.argtypes = [vp, i32]
        L.hg_ctx_profile_read.argtypes = [vp, i32, vp, vp, vp]
        L.hg_kernel_class_name.argtypes = [i32]
        L.hg_kernel_class_name.restype = C.c_char_p
        L.hg_ctx_stream.argtypes = [vp]
        L.hg_ctx_stream.restype = vp
        L.hg_buf_alloc.argtypes = [vp, sz, C.POINTER(vp)]
        L.hg_buf_upload.argtypes = [vp, vp, sz, vp, sz]
        L.hg_buf_download.argtypes = [vp, vp, sz, vp, sz]
        L.hg_device_download.argtypes = [vp, vp, vp, sz]
        L.hg_buf_upload_async.argtypes = [vp, vp, sz, vp, sz]
        L.hg_buf_device_ptr.argtypes = [vp]
        L.hg_buf_device_ptr.restype = vp
        L.hg_buf_size.argtypes = [vp]
        L.hg_buf_size.restype = sz
        L.hg_buf_free.argtypes = [vp]
        L.hg_field_base_bytes.argtypes = [i32]
        L.hg_field_base_bytes.restype = sz
        L.hg_field_encode.argtypes = [vp, vp, sz]
        L.hg_field_decode.argtypes = [vp, vp, sz]
        L.hg_transcript_new.argtypes = [i32, C.POINTER(vp)]
        L.hg_transcript_from_proof.argtypes = [i32, vp, sz, C.POINTER(vp)]
        L.hg_transcript_free.argtypes = [vp]
        L.hg_transcript_from_callbacks.argtypes = [i32, vp, SQUEEZE_FN, WRITE_FN, READ_FN, i32, C.POINTER(vp)]
        L.hg_transcript_squeeze_challenge.argtypes = [vp, vp]
        L.hg_transcript_squeeze_challenges.argtypes = [vp, sz, vp]
        L.hg_transcript_write_felt_ext.argtypes = [vp, vp]
        L.hg_transcript_read_felt_ext.argtypes = [vp, vp]
        L.hg_transcript_proof_len.argtypes = [vp]
        L.hg_transcript_proof_len.restype = sz
        L.hg_transcript_proof_copy.argtypes = [vp, vp, sz]
        L.hg_transcript_num_squeezed.argtypes = [vp]
        L.hg_transcript_num_squeezed.restype = sz
        L.hg_verifier_new.argtypes = [vp, vp, sz, C.POINTER(vp)]
        L.hg_verifier_free.argtypes = [vp]
        L.hg_verifier_free.restype = None
        L.hg_gkr_verify_batch.argtypes = [vp, sz, vp, sz, vp, vp, vp, vp, i32, vp, vp]
        L.hg_verifier_reason.argtypes = [vp, sz]
        L.hg_verifier_reason.restype = C.c_char_p
        L.hg_verifier_num_inputs.argtypes = [vp]
        L.hg_verifier_num_inputs.restype = sz
        L.hg_verifier_input_len.argtypes = [vp, sz]
        L.hg_verifier_input_len.restype = sz
        L.hg_verifier_timing.argtypes = [vp, vp]
        L.hg_verifier_timing.restype = None
        L.hg_mle_eval_multi.argtypes = [vp, sz, vp, vp, vp, i32, vp]
        L.hg_lasso_preprocess.argtypes = [vp, sz, sz, sz, C.POINTER(vp)]
        L.hg_lasso_pp_free.argtypes = [vp]
        L.hg_lasso_preprocess_lookups.argtypes = [vp, sz, sz, sz, C.POINTER(vp)]
        L.hg_lasso_pp_lookup_index_by_id.argtypes = [vp, C.c_char_p]
        L.hg_lasso_node_new_ids.argtypes = [vp, vp, sz, vp, vp, sz, C.POINTER(vp)]
        for f in ("hg_lasso_pp_num_lookups", "hg_lasso_pp_num_subtables", "hg_lasso_pp_num_memories"):
            getattr(L, f).argtypes = [vp]
            getattr(L, f).restype = sz
        L.hg_lasso_pp_lookup_index.argtypes = [vp, u64]
        L.hg_lasso_pp_memory_maps.argtypes = [vp, vp, vp]
        L.hg_lasso_pp_subtable_id.argtypes = [vp, sz, vp, sz]
        L.hg_lasso_node_new.argtypes = [vp, vp, sz, vp, vp, sz, C.POINTER(vp)]
        L.hg_lasso_node_free.argtypes = [vp]
        for f in ("hg_lasso_node_log2_input_size", "hg_lasso_node_device_bytes", "hg_lasso_node_num_chunks"):
            getattr(L, f).argtypes = [vp]
            getattr(L, f).restype = sz
        L.hg_lasso_node_timing.argtypes = [vp, vp]
        L.hg_lasso_node_timing.restype = None
        L.hg_lasso_node_prove.argtypes = [vp, vp, sz, i32, vp, i32, vp, vp]
        L.hg_lasso_node_download_polys.argtypes = [vp, vp, vp, vp, vp]
        L.hg_lasso_node_shard_words.argtypes = [vp]
        L.hg_lasso_node_shard_words.restype = sz
        L.hg_lasso_node_prove_shard.argtypes = [vp, vp, sz, i32, vp, i32, i32, vp, sz, C.POINTER(sz)]
        L.hg_lasso_node_emit_shard.argtypes = [vp, vp, sz, vp, vp]
        L.hg_shard_merge.argtypes = [i32, vp, vp, sz]
        L.hg_lasso_node_prove_shard_dev.argtypes = [vp, vp, sz, i32, vp, i32, i32, vp, sz, C.POINTER(sz)]
        L.hg_lasso_node_emit_shard_dev.argtypes = [vp, vp, sz, vp, vp]
        L.hg_shard_merge_device.argtypes = [vp, vp, i32, sz, vp]
        L.hg_gkr_shard_words.argtypes = [vp]
        L.hg_gkr_shard_words.restype = sz
        L.hg_gkr_prove_shard_dev.argtypes = [vp, sz, vp, vp, vp, vp, i32, i32, vp, sz, C.POINTER(sz)]
        L.hg_gkr_emit_shard_dev.argtypes = [vp, vp, sz]
        L.hg_gkr_emit_shard_part_dev.argtypes = [vp, vp, sz, i32, i32, vp, sz, vp]
        L.hg_transcript_append_bytes.argtypes = [vp, vp, sz]
        L.hg_circuit_new_host.argtypes = [i32, C.POINTER(vp)]
        L.hg_circuit_insert_lasso_host.argtypes = [vp, vp, sz, C.POINTER(i32)]
        L.hg_gkr_verify.argtypes = [vp, sz, vp, vp, vp, vp, vp]
        L.hg_mle_eval_host.argtypes = [i32, vp, sz, sz, vp, vp]
        L.hg_bfv_witness_generate.argtypes = [vp, sz, sz] + [vp] * 15
        L.hg_lasso_node_verify.argtypes = [vp, sz, vp, vp, vp, vp]
        L.hg_sumcheck_prove.argtypes = [vp, i32, sz, sz, vp, vp, vp, vp, i32, vp, vp]
        L.hg_mle_eval_batch.argtypes = [vp, vp, sz, sz, sz, vp, vp]
        L.hg_field_selftest.argtypes = [vp, i32, vp, vp, sz, vp]
        L.hg_ntt.argtypes = [vp, vp, sz, i32, sz]
        L.hg_circuit_new.argtypes = [vp, C.POINTER(vp)]
        L.hg_circuit_free.argtypes = [vp]
        L.hg_circuit_insert_input.argtypes = [vp, sz, sz, C.POINTER(i32)]
        L.hg_circuit_insert_fft.argtypes = [vp, sz, i32, C.POINTER(i32)]
        L.hg_circuit_insert_lasso.argtypes = [vp, vp, C.POINTER(i32)]
        L.hg_circuit_insert_vanilla.argtypes = [vp, sz, sz, sz, sz] + [vp] * 12 + [C.POINTER(i32)]
        L.hg_circuit_connect.argtypes = [vp, i32, i32]
        L.hg_circuit_evaluate.argtypes = [vp, vp, sz]
        L.hg_circuit_evaluate_host.argtypes = [vp, vp, vp, sz]
        L.hg_circuit_node_value.argtypes = [vp, i32, C.POINTER(vp), C.POINTER(sz)]
        L.hg_gkr_prove.argtypes = [vp, sz, vp, vp, vp, vp, i32]
        for f in ("hg_gkr_num_inputs",):
            getattr(L, f).argtypes = [vp]
            getattr(L, f).restype = sz
        L.hg_gkr_timing.argtypes = [vp, vp]
        L.hg_gkr_timing.restype = None
        L.hg_gkr_num_challenges.argtypes = [vp]
        L.hg_gkr_num_challenges.restype = sz
        L.hg_gkr_num_input_claims.argtypes = [vp, sz]
        L.hg_gkr_num_input_claims.restype = sz
        L.hg_gkr_input_claim_num_vars.argtypes = [vp, sz, sz]
        L.hg_gkr_input_claim_num_vars.restype = sz
        L.hg_gkr_input_claim.argtypes = [vp, sz, sz, vp, vp]
        L.hg_bfv_configure.argtypes = [vp, sz, sz, vp, vp, vp, vp, u64, u64, u64, vp, vp, sz, vp]
        L.hg_bfv_pk_configure.argtypes = [vp, sz, sz, vp, vp, vp, vp, vp, vp, u64, u64, u64, vp, vp, sz, vp]
        L.hg_bfv_pk_witness_generate.argtypes = [vp, sz, sz] + [vp] * 24
        _lib = L
    return _lib


def _chk(rc):
    if rc != 0:
        raise HgError(lib().hg_last_error().decode())


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Context:
    """One device + one stream (hg_ctx)."""

    def __init__(self, device=0, field=GOLDILOCKS):
        self.field = field
        self.device = device
        self.h = C.c_void_p()
        _chk(lib().hg_ctx_create(device, field, C.byref(self.h)))

    def set_option(self, option, value):
        _chk(lib().hg_ctx_set_option(self.h, option, value))

    def synchronize(self):
        _chk(lib().hg_ctx_synchronize(self.h))

    @property
    def launch_count(self):
        return int(lib().hg_ctx_launch_count(self.h))

    @property
    def stream(self):
        return lib().hg_ctx_stream(self.h)

    def profile(self, enable: bool):
        _chk(lib().hg_ctx_profile(self.h, 1 if enable else 0))

    def profile_read(self):
        """{class name: (launches, device ms, algorithmic bytes)} accumulated since profile(True)."""
        out = {}
        for k in range(lib().hg_kernel_class_count()):
            n, ms, by = C.c_uint64(0), C.c_double(0), C.c_uint64(0)
            _chk(lib().hg_ctx_profile_read(self.h, k, C.byref(n), C.byref(ms), C.byref(by)))
            out[lib().hg_kernel_class_name(k).decode()] = (n.value, ms.value, by.value)
        return out

    def close(self):
        if self.h:
            lib().hg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceBuffer:
    """hg_buf: device memory owned by the caller through a handle."""

    def __init__(self, ctx: Context, nbytes: int):
        self.ctx = ctx
        self.h = C.c_void_p()
        _chk(lib().hg_buf_alloc(ctx.h, nbytes, C.byref(self.h)))
        self.nbytes = nbytes

    @classmethod
    def from_numpy(cls, ctx, arr):
        arr = np.ascontiguousarray(arr)
        b = cls(ctx, arr.nbytes)
        b.upload(arr)
        return b

    @classmethod
    def from_field(cls, ctx, limbs):
        """Upload base-field elements given as canonical little-endian u64 limbs ([n] for Goldilocks, [n, 4] for BN254) and
        convert them to the device representation (Montgomery form for BN254)."""
        limbs = np.ascontiguousarray(limbs, np.uint64)
        b = cls.from_numpy(ctx, limbs)
        _chk(lib().hg_field_encode(ctx.h, b.ptr, limbs.size // LIMBS[ctx.field]))
        return b

    def to_field(self, count):
        """Inverse of from_field: canonical limbs of `count` base elements."""
        k = LIMBS[self.ctx.field]
        tmp = DeviceBuffer(self.ctx, count * 8 * k)
        out = self.download(np.uint64, count * k)
        if k > 1:
            tmp.upload(out)
            _chk(lib().hg_field_decode(self.ctx.h, tmp.ptr, count))
            out = tmp.download(np.uint64, count * k)
        tmp.free()
        return out.reshape(count, k) if k > 1 else out

    def upload(self, arr, offset=0):
        arr = np.ascontiguousarray(arr)
        _chk(lib().hg_buf_upload(self.ctx.h, self.h, offset, _p(arr), arr.nbytes))

    def upload_async(self, arr, offset=0):
        """No wait: `arr` (contiguous, ideally pinned) must stay alive until the next synchronising call."""
        if not arr.flags["C_CONTIGUOUS"]:
            raise HgError("upload_async needs a contiguous array")
        self._keepalive = arr
        _chk(lib().hg_buf_upload_async(self.ctx.h, self.h, offset, _p(arr), arr.nbytes))

    def download(self, dtype, count, offset=0):
        out = np.zeros(count, dtype)
        _chk(lib().hg_buf_download(self.ctx.h, self.h, offset, _p(out), out.nbytes))
        return out

    @property
    def ptr(self):
        return lib().hg_buf_device_ptr(self.h)

    def free(self):
        if self.h:
            lib().hg_buf_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceView:
    """A slice of a DeviceBuffer (no ownership): what Circuit.evaluate needs is .ptr"""

    def __init__(self, base: DeviceBuffer, offset: int, nbytes: int):
        self.base, self.offset, self.nbytes, self.ctx = base, offset, nbytes, base.ctx

    @property
    def ptr(self):
        return self.base.ptr + self.offset

    def download(self, dtype, count):
        return self.base.download(dtype, count, self.offset)

    def to_field(self, count):
        k = LIMBS[self.ctx.field]
        tmp = DeviceBuffer(self.ctx, count * 8 * k)
        tmp.upload(self.base.download(np.uint64, count * k, self.offset))
        out = tmp.to_field(count)
        tmp.free()
        return out


class Keccak256Transcript:
    """transcript.rs:117-203."""

    def __init__(self, field=GOLDILOCKS, proof: bytes = None):
        self.field = field
        self.h = C.c_void_p()
        self._el = LIMBS[field] * DEGREE[field]
        if proof is None:
            _chk(lib().hg_transcript_new(field, C.byref(self.h)))
        else:
            buf = np.frombuffer(proof, np.uint8)
            _chk(lib().hg_transcript_from_proof(field, _p(np.ascontiguousarray(buf)), buf.size, C.byref(self.h)))

    @classmethod
    def from_proof(cls, proof: bytes, field=GOLDILOCKS):
        return cls(field, proof)

    def squeeze_challenge(self):
        out = np.zeros(self._el, np.uint64)
        _chk(lib().hg_transcript_squeeze_challenge(self.h, _p(out)))
        return out

    def squeeze_challenges(self, n):
        out = np.zeros((n, self._el), np.uint64)
        if n:
            _chk(lib().hg_transcript_squeeze_challenges(self.h, n, _p(out)))
        return out

    def write_felt_ext(self, e):
        _chk(lib().hg_transcript_write_felt_ext(self.h, _p(np.ascontiguousarray(e, np.uint64))))

    def read_felt_ext(self):
        out = np.zeros(self._el, np.uint64)
        _chk(lib().hg_transcript_read_felt_ext(self.h, _p(out)))
        return out

    def append_bytes(self, data: bytes):
        """bytes serialised elsewhere (the per-rank parts of a sharded proof)"""
        buf = np.frombuffer(data, np.uint8)
        if buf.size:
            _chk(lib().hg_transcript_append_bytes(self.h, _p(np.ascontiguousarray(buf)), buf.size))

    def into_proof(self) -> bytes:
        n = lib().hg_transcript_proof_len(self.h)
        out = np.zeros(max(n, 1), np.uint8)
        _chk(lib().hg_transcript_proof_copy(self.h, _p(out), n))
        return out[:n].tobytes()

    @property
    def num_squeezed(self):
        return int(lib().hg_transcript_num_squeezed(self.h))

    def __del__(self):
        try:
            if self.h:
                lib().hg_transcript_free(self.h)
                self.h = None
        except Exception:
            pass


class CallbackTranscript(Keccak256Transcript):
    """A transcript owned by the CALLER, handed to the library as callbacks (hg_transcript_from_callbacks): what the Rust shim
    does with the `&mut dyn TranscriptWrite<F, E>` it receives in Node::prove_claim_reduction (lasso.rs:58-63). `inner` is any
    object with squeeze_challenge() / write_felt_ext(e) / read_felt_ext(); every call the library makes is forwarded to it and
    recorded in `log` as ("squeeze" | "write" | "read", limbs). A callback that raises makes the library call fail."""

    def __init__(self, inner, field=GOLDILOCKS, message_independent=False):
        self.field, self.inner, self.log = field, inner, []
        self._el = LIMBS[field] * DEGREE[field]
        el = self._el

        def squeeze(_user, out):
            try:
                v = np.asarray(self.inner.squeeze_challenge(), np.uint64)
                for i in range(el):
                    out[i] = int(v[i])
                self.log.append(("squeeze", tuple(int(x) for x in v)))
                return 0
            except Exception:
                return 1

        def write(_user, ext):
            try:
                v = np.array([ext[i] for i in range(el)], np.uint64)
                self.inner.write_felt_ext(v)
                self.log.append(("write", tuple(int(x) for x in v)))
                return 0
            except Exception:
                return 1

        def read(_user, out):
            try:
                v = np.asarray(self.inner.read_felt_ext(), np.uint64)
                for i in range(el):
                    out[i] = int(v[i])
                self.log.append(("read", tuple(int(x) for x in v)))
                return 0
            except Exception:
                return 1

        self._cbs = (SQUEEZE_FN(squeeze), WRITE_FN(write), READ_FN(read))  # keep the trampolines alive
        self.h = C.c_void_p()
        _chk(lib().hg_transcript_from_callbacks(field, None, self._cbs[0], self._cbs[1], self._cbs[2], 1 if message_independent else 0, C.byref(self.h)))

    def into_proof(self) -> bytes:
        return self.inner.into_proof()


class HgLookupDesc(C.Structure):
    """hg_lookup_desc (include/hg_b200.h)"""
    _fields_ = [("lookup_id", C.c_char_p), ("n_subtables", C.c_size_t), ("subtable_ids", C.POINTER(C.c_char_p)), ("tables", C.POINTER(C.c_void_p)),
                ("dimension_masks", C.POINTER(C.c_uint64)), ("n_chunk_bits", C.c_size_t), ("chunk_bits", C.POINTER(C.c_uint32)), ("combine_weight", C.c_uint64)]


class TableLookup:
    """A LookupType given by data (table.rs:35-67 through hg_lookup_desc): lookup_id, subtables [(subtable_id, table of M u64, dimensions)],
    chunk_bits (low chunk first) and the weight w of combine_lookups = sum_t w^t operand_t."""

    def __init__(self, lookup_id, subtables, chunk_bits, combine_weight):
        self.lookup_id, self.subtables, self.chunk_bits, self.combine_weight = lookup_id, subtables, list(chunk_bits), int(combine_weight)


def range_lookup_as_table(bound, M=1 << 16):
    """RangeLookup::new_boxed(bound) (range.rs:177-274) written out as a TableLookup: the same subtables, indices, chunk bits and weight."""
    log2M = M.bit_length() - 1
    bits = bound.bit_length() - 1
    full = ("full", np.arange(M, dtype=np.uint64))
    cutoff = (1 << (bits % log2M)) + bound % M                      # range.rs:58-62 (Q5)
    rem_t = np.arange(M, dtype=np.uint64)
    rem_t[min(cutoff, M):] = 0
    rem = (f"bound_{bound}", rem_t)
    nch = bits // log2M
    if bound % M == 0:
        subs, cb = [(full[0], full[1], list(range(nch)))], [log2M] * nch
    elif bound < M:
        subs, cb = [(rem[0], rem[1], [0])], [cutoff.bit_length() - 1]
    else:
        subs, cb = [(full[0], full[1], list(range(nch))), (rem[0], rem[1], [nch])], [log2M] * nch + [cutoff.bit_length() - 1]
    return TableLookup(f"range_{bound}", subs, cb, M)


class LassoPreprocessing:
    """lasso.rs:513-651: LassoPreprocessing::preprocess::<C, M>. `bounds`: RangeLookup types given by their bounds; or
    LassoPreprocessing.preprocess_lookups([TableLookup, ...]) for plug-in lookup types."""

    def __init__(self, bounds, C_=4, M=1 << 16, _lookups=None):
        self.h = C.c_void_p()
        self.C, self.M = C_, M
        if _lookups is None:
            b = np.array([int(x) for x in bounds], np.uint64)
            _chk(lib().hg_lasso_preprocess(_p(b), b.size, C_, M, C.byref(self.h)))
            return
        descs = (HgLookupDesc * len(_lookups))()
        keep = []
        for d, lk in zip(descs, _lookups):
            n = len(lk.subtables)
            ids = (C.c_char_p * n)(*[sid.encode() for sid, _, _ in lk.subtables])
            tabs = [np.ascontiguousarray(t, np.uint64) for _, t, _ in lk.subtables]
            for t in tabs:
                if t.size != M:
                    raise HgError(f"subtable of lookup {lk.lookup_id} has {t.size} entries, M = {M}")
            tp = (C.c_void_p * n)(*[t.ctypes.data for t in tabs])
            masks = (C.c_uint64 * n)(*[sum(1 << int(x) for x in dims) for _, _, dims in lk.subtables])
            cb = (C.c_uint32 * len(lk.chunk_bits))(*lk.chunk_bits)
            d.lookup_id, d.n_subtables, d.subtable_ids, d.tables = lk.lookup_id.encode(), n, ids, tp
            d.dimension_masks, d.n_chunk_bits, d.chunk_bits, d.combine_weight = masks, len(lk.chunk_bits), cb, lk.combine_weight
            keep += [ids, tabs, tp, masks, cb]
        _chk(lib().hg_lasso_preprocess_lookups(descs, len(_lookups), C_, M, C.byref(self.h)))

    @classmethod
    def preprocess(cls, bounds, C_=4, M=1 << 16):
        return cls(bounds, C_, M)

    @classmethod
    def preprocess_lookups(cls, lookups, C_=4, M=1 << 16):
        return cls(None, C_, M, _lookups=list(lookups))

    def lookup_index_by_id(self, lookup_id: str):
        return int(lib().hg_lasso_pp_lookup_index_by_id(self.h, lookup_id.encode()))

    @property
    def num_lookups(self):
        return int(lib().hg_lasso_pp_num_lookups(self.h))

    @property
    def num_subtables(self):
        return int(lib().hg_lasso_pp_num_subtables(self.h))

    @property
    def num_memories(self):
        return int(lib().hg_lasso_pp_num_memories(self.h))

    def lookup_index(self, bound):
        return int(lib().hg_lasso_pp_lookup_index(self.h, int(bound)))

    def memory_maps(self):
        m = self.num_memories
        a, b = np.zeros(m, np.uint32), np.zeros(m, np.uint32)
        _chk(lib().hg_lasso_pp_memory_maps(self.h, _p(a), _p(b)))
        return [int(x) for x in a], [int(x) for x in b]

    def subtable_id(self, idx):
        buf = C.create_string_buffer(64)
        _chk(lib().hg_lasso_pp_subtable_id(self.h, idx, buf, 64))
        return buf.value.decode()

    def memory_names(self):
        sub, dim = self.memory_maps()
        return [f"{self.subtable_id(s)}@{d}" for s, d in zip(sub, dim)]

    def __del__(self):
        try:
            if self.h:
                lib().hg_lasso_pp_free(self.h)
                self.h = None
        except Exception:
            pass


class LassoNode:
    """LassoNode<F, E, C, M> (lasso.rs:32-154) on one device."""

    def __init__(self, ctx: Context, preprocessing: LassoPreprocessing, num_vars: int, lookup_segments):
        """lookup_segments: [(bound | lookup id string, run_length), ...] = the node's `lookups: Vec<LookupId>` run-length encoded."""
        self.ctx, self.pp, self.num_vars = ctx, preprocessing, num_vars
        sl = np.array([int(l) for _, l in lookup_segments], np.uint64)
        self.h = C.c_void_p()
        if lookup_segments and isinstance(lookup_segments[0][0], str):
            ids = (C.c_char_p * len(lookup_segments))(*[b.encode() for b, _ in lookup_segments])
            _chk(lib().hg_lasso_node_new_ids(ctx.h, preprocessing.h, num_vars, ids, _p(sl), sl.size, C.byref(self.h)))
        else:
            sb = np.array([int(b) for b, _ in lookup_segments], np.uint64)
            _chk(lib().hg_lasso_node_new(ctx.h, preprocessing.h, num_vars, _p(sb), _p(sl), sb.size, C.byref(self.h)))
        self._el = LIMBS[ctx.field] * DEGREE[ctx.field]

    def is_input(self):
        return False  # lasso.rs:41-43

    def log2_input_size(self):
        return int(lib().hg_lasso_node_log2_input_size(self.h))  # lasso.rs:45-47

    def log2_output_size(self):
        return 0  # lasso.rs:49-51

    @property
    def device_bytes(self):
        return int(lib().hg_lasso_node_device_bytes(self.h))

    @property
    def num_chunks(self):
        return int(lib().hg_lasso_node_num_chunks(self.h))

    def prove_claim_reduction(self, inputs, transcript: Keccak256Transcript, mode=MODE_PREFETCH, n_inputs=None):
        """inputs: numpy uint64 array of canonical limbs (host; copied inside the call) or a DeviceBuffer.
        Returns the node's single EvalClaim (point limbs [num_vars, el], value limbs [el])."""
        pt = np.zeros((self.num_vars, self._el), np.uint64)
        val = np.zeros(self._el, np.uint64)
        if hasattr(inputs, "ptr"):   # DeviceBuffer, DeviceView, NodeValueView: device memory
            n = n_inputs if n_inputs is not None else inputs.nbytes // (8 * LIMBS[self.ctx.field])
            _chk(lib().hg_lasso_node_prove(self.h, inputs.ptr, n, 1, transcript.h, mode, _p(pt), _p(val)))
        else:
            arr = np.ascontiguousarray(inputs, np.uint64)
            n = arr.size // LIMBS[self.ctx.field]
            _chk(lib().hg_lasso_node_prove(self.h, _p(arr), n, 0, transcript.h, mode, _p(pt), _p(val)))
        return pt, val

    # ---- one proof over several GPUs (include/hg_b200.h, "one proof over several GPUs")
    def prove_shard(self, inputs, transcript: Keccak256Transcript, rank: int, world: int, n_inputs=None):
        """This rank's part of the node's message buffer (uint64 words, device representation; slots of other ranks are 0)."""
        cap = int(lib().hg_lasso_node_shard_words(self.h))
        out = np.zeros(cap, np.uint64)
        nw = C.c_size_t(0)
        if hasattr(inputs, "ptr"):   # DeviceBuffer, DeviceView, NodeValueView: device memory
            n = n_inputs if n_inputs is not None else inputs.nbytes // (8 * LIMBS[self.ctx.field])
            _chk(lib().hg_lasso_node_prove_shard(self.h, inputs.ptr, n, 1, transcript.h, rank, world, _p(out), cap, C.byref(nw)))
        else:
            arr = np.ascontiguousarray(inputs, np.uint64)
            n = arr.size // LIMBS[self.ctx.field]
            _chk(lib().hg_lasso_node_prove_shard(self.h, _p(arr), n, 0, transcript.h, rank, world, _p(out), cap, C.byref(nw)))
        return out[: nw.value]

    def emit_shard(self, merged):
        """Rank 0, after prove_shard on this node: serialise the merged message buffer into the transcript given to prove_shard."""
        merged = np.ascontiguousarray(merged, np.uint64)
        pt = np.zeros((self.num_vars, self._el), np.uint64)
        val = np.zeros(self._el, np.uint64)
        _chk(lib().hg_lasso_node_emit_shard(self.h, _p(merged), merged.size, _p(pt), _p(val)))
        return pt, val

    @property
    def shard_words(self):
        return int(lib().hg_lasso_node_shard_words(self.h))

    def prove_shard_dev(self, inputs, transcript: Keccak256Transcript, rank: int, world: int, d_out_ptr: int, cap_words: int, n_inputs=None):
        """prove_shard without leaving the device: this rank's partial message buffer is copied to device memory at d_out_ptr
        (stream-ordered on the context's stream). Returns the number of 64-bit words written."""
        nw = C.c_size_t(0)
        if hasattr(inputs, "ptr"):   # DeviceBuffer, DeviceView, NodeValueView: device memory
            n = n_inputs if n_inputs is not None else inputs.nbytes // (8 * LIMBS[self.ctx.field])
            _chk(lib().hg_lasso_node_prove_shard_dev(self.h, inputs.ptr, n, 1, transcript.h, rank, world, C.c_void_p(d_out_ptr), cap_words, C.byref(nw)))
        else:
            arr = np.ascontiguousarray(inputs, np.uint64)
            n = arr.size // LIMBS[self.ctx.field]
            _chk(lib().hg_lasso_node_prove_shard_dev(self.h, _p(arr), n, 0, transcript.h, rank, world, C.c_void_p(d_out_ptr), cap_words, C.byref(nw)))
        return int(nw.value)

    def emit_shard_dev(self, d_merged_ptr: int, n_words: int):
        pt = np.zeros((self.num_vars, self._el), np.uint64)
        val = np.zeros(self._el, np.uint64)
        _chk(lib().hg_lasso_node_emit_shard_dev(self.h, C.c_void_p(d_merged_ptr), n_words, _p(pt), _p(val)))
        return pt, val

    def prove_claim_reduction_sharded(self, inputs, transcript: Keccak256Transcript, group=None, n_inputs=None):
        """prove_claim_reduction with the node's grand-product terms split over the ranks of a torch.distributed group
        (one process per GPU, every rank holds the inputs and a transcript in the same state). The only exchange is one
        gather of the message buffers to rank 0, which sums them and writes the proof; other ranks return None."""
        import torch
        import torch.distributed as dist

        rank, world = dist.get_rank(group), dist.get_world_size(group)
        part = self.prove_shard(inputs, transcript, rank, world, n_inputs)
        merged = gather_and_merge(self.ctx.field, part, group)
        if rank != 0:
            return None
        return self.emit_shard(merged)

    def timing(self):
        """Host phases of the last prove in microseconds: squeeze+upload challenges, enqueue, wait for GPU, serialise."""
        out = np.zeros(4, np.float64)
        lib().hg_lasso_node_timing(self.h, _p(out))
        return dict(zip(("challenges_us", "enqueue_us", "gpu_wait_us", "serialise_us"), (float(x) for x in out)))

    def download_polys(self):
        R, M, m, nc = 1 << self.num_vars, self.pp.M, self.pp.num_memories, self.num_chunks
        dims = np.zeros((self.pp.C, R), np.uint16)
        rd = np.zeros((nc, R), np.uint32)
        fc = np.zeros((nc, M), np.uint32)
        e = np.zeros((m, R, LIMBS[self.ctx.field]), np.uint64)
        _chk(lib().hg_lasso_node_download_polys(self.h, _p(dims), _p(rd), _p(fc), _p(e)))
        return dims, rd, fc, e

    def free(self):
        if self.h:
            lib().hg_lasso_node_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def lasso_node_verify(preprocessing: "LassoPreprocessing", num_vars: int, transcript: "Keccak256Transcript", options=None):
    """Node::verify_claim_reduction on the host (no GPU): reads the node's messages from a transcript built with
    Keccak256Transcript(field, proof=...). Returns (point [num_vars, el], claimed_sum [el]); raises HgError when the reference
    would return Err / panic. options = (a3_wire, a3_h1, a5_ascending) or None."""
    el = LIMBS[transcript.field] * DEGREE[transcript.field]
    pt = np.zeros((num_vars, el), np.uint64)
    val = np.zeros(el, np.uint64)
    opt = None if options is None else np.array(options, np.int32)
    _chk(lib().hg_lasso_node_verify(preprocessing.h, num_vars, transcript.h, None if opt is None else _p(opt), _p(pt), _p(val)))
    return pt, val


def shard_merge(field: int, acc, part):
    """acc += part element-wise in the field (message buffers of LassoNode.prove_shard); in place, returns acc."""
    acc = np.ascontiguousarray(acc, np.uint64)
    part = np.ascontiguousarray(part, np.uint64)
    if acc.size != part.size:
        raise HgError("shard_merge: buffers of different length")
    _chk(lib().hg_shard_merge(field, _p(acc), _p(part), acc.size))
    return acc


def shard_merge_device(ctx: "Context", d_parts_ptr: int, world: int, n_words: int, d_acc_ptr: int):
    """acc = element-wise field sum of the `world` gathered message buffers ([world][n_words] at d_parts_ptr), on the context's stream."""
    _chk(lib().hg_shard_merge_device(ctx.h, C.c_void_p(d_parts_ptr), world, n_words, C.c_void_p(d_acc_ptr)))


class ShardExchange:
    """Device-side exchange of one sharded proof (hg_b200.h): per-rank partial buffer -> NCCL all-gather over NVLink (enqueued
    behind the library's stream) -> one merge kernel -> rank 0 serialises. Buffers are torch tensors owned by this object."""

    def __init__(self, ctx: "Context", cap_words: int, group=None):
        import torch
        import torch.distributed as dist
        self.ctx, self.group, self.cap = ctx, group, cap_words
        self.dist = dist if dist.is_available() and dist.is_initialized() else None
        self.rank = self.dist.get_rank(group) if self.dist else 0
        self.world = self.dist.get_world_size(group) if self.dist else 1
        dev = torch.device("cuda", ctx.device)
        self.torch = torch
        self.part = torch.zeros(cap_words, dtype=torch.int64, device=dev)
        self.gathered = torch.zeros(self.world * cap_words, dtype=torch.int64, device=dev)
        self.merged = torch.zeros(cap_words, dtype=torch.int64, device=dev)
        self.stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        self.PART_CAP = max(1 << 14, ((768 * 1024) // max(1, self.world) + 255) & ~255)

    PART_CAP = 1 << 18   # bytes one rank's part of the proof may take in the byte exchange (set per instance: ~768 KB / world; the whole proof is 119 KB for Goldilocks, 238 KB for BN254)

    def run(self, prove_shard_dev, emit_shard_dev, emit_part=None, transcript=None):
        """prove_shard_dev(rank, world, d_out_ptr, cap) -> n_words;  emit_shard_dev(d_merged_ptr, n_words) -> result (rank 0 only).
        With emit_part(d_merged_ptr, n_words, part, nparts) -> bytes and rank 0's transcript, the serialisation is split over the
        ranks as well: every rank serialises one range of the proof, the ranges are all-gathered (fixed-size byte buffers with a
        length header) and rank 0 appends them in order."""
        import time
        timing = os.environ.get("HG_SHARD_TIMING") == "1"   # phase timing costs two extra synchronisations per proof
        t0 = time.perf_counter()
        n = prove_shard_dev(self.rank, self.world, self.part.data_ptr(), self.cap)
        t1 = time.perf_counter()
        # the collective is issued once this device has finished its part: enqueueing it behind ~100 pending launches of three
        # streams cost 2.4 ms per proof on 2 B200s (measured), this wait costs nothing the exchange would not wait for anyway
        self.ctx.synchronize()
        t2 = time.perf_counter()
        if self.world == 1:
            return emit_shard_dev(self.part.data_ptr(), n)
        with self.torch.cuda.stream(self.stream):     # the collective waits for everything the library enqueued
            g = self.gathered[: self.world * n]
            self.dist.all_gather_into_tensor(g, self.part[:n], group=self.group)
        shard_merge_device(self.ctx, g.data_ptr(), self.world, n, self.merged.data_ptr())
        if timing:
            self.ctx.synchronize()
        t3 = time.perf_counter()
        res = None
        if emit_part is not None and self.world > 1:
            part = emit_part(self.merged.data_ptr(), n, self.rank, self.world)   # waits for the merge, serialises this rank's range
            if len(part) + 8 > self.PART_CAP:
                raise HgError("ShardExchange: a part of the proof exceeds the byte-exchange buffer")
            if not hasattr(self, "bytes_host"):
                self.bytes_host = self.torch.zeros(self.PART_CAP, dtype=self.torch.uint8).pin_memory()
                self.bytes_dev = self.torch.zeros(self.PART_CAP, dtype=self.torch.uint8, device=self.part.device)
                self.bytes_all = self.torch.zeros(self.world * self.PART_CAP, dtype=self.torch.uint8, device=self.part.device)
                self.bytes_all_host = self.torch.zeros(self.world * self.PART_CAP, dtype=self.torch.uint8).pin_memory()
            hb = self.bytes_host.numpy()
            hb[:8] = np.frombuffer(np.uint64(len(part)).tobytes(), np.uint8)
            hb[8:8 + len(part)] = np.frombuffer(part, np.uint8)
            used = (8 + len(part) + 255) & ~255
            with self.torch.cuda.stream(self.stream):
                self.bytes_dev[:used].copy_(self.bytes_host[:used], non_blocking=True)
                self.dist.all_gather_into_tensor(self.bytes_all, self.bytes_dev, group=self.group)
                if self.rank == 0:
                    self.bytes_all_host.copy_(self.bytes_all, non_blocking=True)
            self.ctx.synchronize()
            if self.rank == 0:
                ab = self.bytes_all_host.numpy()
                for r in range(self.world):
                    ln = int(np.frombuffer(ab[r * self.PART_CAP: r * self.PART_CAP + 8].tobytes(), np.uint64)[0])
                    transcript.append_bytes(ab[r * self.PART_CAP + 8: r * self.PART_CAP + 8 + ln].tobytes())
                res = True
        elif self.rank != 0:
            self.ctx.synchronize()
        else:
            res = emit_shard_dev(self.merged.data_ptr(), n)
        if timing:
            self.phases = {"enqueue_ms": 1e3 * (t1 - t0), "device_wait_ms": 1e3 * (t2 - t1), "gather_merge_ms": 1e3 * (t3 - t2), "emit_ms": 1e3 * (time.perf_counter() - t3)}
        return res

    exchange_bytes_per_rank = property(lambda self: 8 * self.cap)


def gather_and_merge(field: int, part, group=None):
    """Gathers the per-rank message buffers on rank 0 (NCCL when the group has it, else gloo) and sums them in the field.
    Returns the merged buffer on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if world == 1:
        return part
    backend = dist.get_backend(group)
    t = torch.from_numpy(part.view(np.int64))
    if backend == "nccl":
        t = t.cuda()
    bufs = [torch.empty_like(t) for _ in range(world)] if rank == 0 else None
    dist.gather(t, bufs, dst=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    if rank != 0:
        return None
    acc = part.copy()
    for r in range(1, world):
        shard_merge(field, acc, bufs[r].cpu().numpy().view(np.uint64))
    return acc


def sumcheck_prove(ctx: Context, arity, coeffs_ext, d_tables: DeviceBuffer, num_vars, claim_ext, transcript, mode=MODE_PREFETCH):
    """gkr::sum_check::prove_sum_check for g = poly(0) * sum_i coeffs[i] * prod_{k<arity} poly(arity*i+k)."""
    el = LIMBS[ctx.field] * DEGREE[ctx.field]
    coeffs_ext = np.ascontiguousarray(coeffs_ext, np.uint64)
    nterms = coeffs_ext.size // el
    pt = np.zeros((num_vars, el), np.uint64)
    ev = np.zeros((nterms * arity, el), np.uint64)
    _chk(lib().hg_sumcheck_prove(ctx.h, arity, nterms, num_vars, _p(coeffs_ext), d_tables.ptr, _p(np.ascontiguousarray(claim_ext, np.uint64)),
                                 transcript.h, mode, _p(pt), _p(ev)))
    return pt, ev


def mle_eval_batch(ctx: Context, d_tables: DeviceBuffer, n_tables, num_vars, point_ext, stride=None):
    el = LIMBS[ctx.field] * DEGREE[ctx.field]
    out = np.zeros((n_tables, el), np.uint64)
    stride = (1 << num_vars) if stride is None else stride
    _chk(lib().hg_mle_eval_batch(ctx.h, d_tables.ptr, n_tables, stride, num_vars, _p(np.ascontiguousarray(point_ext, np.uint64)), _p(out)))
    return out


def mle_eval_multi(ctx: Context, tables, points):
    """MLE of each base table at its own point on the device (hg_mle_eval_multi). tables: DeviceBuffer / DeviceView (library
    representation) or host numpy arrays of canonical limbs, all of one kind; points: one [num_vars, el] array per table."""
    el = LIMBS[ctx.field] * DEGREE[ctx.field]
    on_dev = len(tables) > 0 and not isinstance(tables[0], np.ndarray)
    keep = [t if on_dev else np.ascontiguousarray(t, np.uint64).reshape(-1) for t in tables]
    if len(points) != len(keep) or (not on_dev and any(t.size != (LIMBS[ctx.field] << len(p)) for t, p in zip(keep, points))):
        raise HgError("mle_eval_multi: every table must have 2^num_vars elements, one point per table")
    ptrs = (C.c_void_p * max(len(keep), 1))(*[(t.ptr if on_dev else t.ctypes.data) for t in keep])
    nvs = np.array([len(p) for p in points], np.uint64)
    pts = np.ascontiguousarray(np.concatenate([np.asarray(p, np.uint64).reshape(-1) for p in points] + [np.zeros(0, np.uint64)]))
    out = np.zeros((len(keep), el), np.uint64)
    _chk(lib().hg_mle_eval_multi(ctx.h, len(keep), ptrs, _p(nvs), _p(pts), 1 if on_dev else 0, _p(out)))
    return out


def field_selftest(ctx: Context, op, a_ext, b_ext):
    a = np.ascontiguousarray(a_ext, np.uint64)
    b = np.ascontiguousarray(b_ext, np.uint64)
    el = LIMBS[ctx.field] * DEGREE[ctx.field]
    out = np.zeros_like(a)
    _chk(lib().hg_field_selftest(ctx.h, op, _p(a), _p(b), a.size // el, _p(out)))
    return out


def ntt(ctx: Context, d_data: DeviceBuffer, log_n, inverse=False, batch=1):
    """FftNode::forward / ::inverse evaluation, in place on the device (sk_encryption_circuit.rs:224,249,251)."""
    _chk(lib().hg_ntt(ctx.h, d_data.ptr, log_n, 1 if inverse else 0, batch))


class BfvEncrypt:
    """Driver-level mirror of `BfvEncrypt` (sk_encryption_circuit.rs:300-523) for forward evaluation only: circuit.evaluate (:442)
    on the device, returning the two layers the tests look at."""

    def __init__(self, ctx: Context, params):
        self.prover = BfvSkEncryptProver(ctx, params)
        self.ctx, self.P, self.pp, self.node = ctx, params, self.prover.pp, self.prover.lasso

    def upload_inputs(self, ins):
        return self.prover.upload_inputs(ins)

    def evaluate(self, dev_ins):
        """circuit.evaluate: returns (`lasso_inputs_batched` layer, `sum` layer) as device views (library-owned memory)."""
        c = self.prover.circuit
        c.evaluate(dev_ins)
        out = []
        for name in ("lasso_in", "sum"):
            ptr, n = c.node_value(self.prover.ids[name])
            out.append(NodeValueView(self.ctx, ptr, n))
        return tuple(out)


class NodeValueView:
    """Value of a circuit node: device memory owned by the circuit (valid until the next evaluate)."""

    def __init__(self, ctx, ptr, n):
        self.ctx, self.ptr, self.n = ctx, ptr, n

    def download(self, dtype, count):
        out = np.zeros(count, dtype)
        _chk(lib().hg_device_download(self.ctx.h, C.c_void_p(self.ptr), _p(out), out.nbytes))
        return out


class VanillaGate:
    """VanillaGate::new(Option<F>, Vec<(Option<F>, (input, wire))>, Vec<(Option<F>, (input, wire), (input, wire))>) as plain data."""

    def __init__(self, const=None, adds=(), muls=()):
        self.const, self.adds, self.muls = const, list(adds), list(muls)


def mle_eval_host(field: int, table_limbs, num_vars: int, point_ext):
    """MultilinearPoly::evaluate on the HOST (no GPU): table of 2^num_vars base elements as canonical limbs."""
    t = np.ascontiguousarray(table_limbs, np.uint64)
    out = np.zeros(LIMBS[field] * DEGREE[field], np.uint64)
    _chk(lib().hg_mle_eval_host(field, _p(t), t.size // LIMBS[field], num_vars, _p(np.ascontiguousarray(point_ext, np.uint64)), _p(out)))
    return out


class Circuit:
    """gkr::circuit::Circuit on the device (sk_encryption_circuit.rs:434-437): insert / connect / evaluate / prove_gkr."""

    def __init__(self, ctx: Context = None, field=None):
        """ctx given: a circuit on that device. ctx None: a host-only DESCRIPTION of `field` (hg_circuit_new_host), for verify_gkr."""
        self.ctx = ctx
        self.field = ctx.field if ctx is not None else (GOLDILOCKS if field is None else field)
        self.h = C.c_void_p()
        if ctx is not None:
            _chk(lib().hg_circuit_new(ctx.h, C.byref(self.h)))
        else:
            _chk(lib().hg_circuit_new_host(self.field, C.byref(self.h)))
        self._keep = []

    def insert_input(self, log2_size, num_reps=1):
        i = C.c_int(-1)
        _chk(lib().hg_circuit_insert_input(self.h, log2_size, num_reps, C.byref(i)))
        return i.value

    def insert_fft(self, log2_size, inverse=False):
        i = C.c_int(-1)
        _chk(lib().hg_circuit_insert_fft(self.h, log2_size, 1 if inverse else 0, C.byref(i)))
        return i.value

    def insert_lasso(self, node: "LassoNode"):
        i = C.c_int(-1)
        _chk(lib().hg_circuit_insert_lasso(self.h, node.h, C.byref(i)))
        self._keep.append(node)
        return i.value

    def insert_lasso_host(self, preprocessing: "LassoPreprocessing", num_vars: int):
        """the Lasso node of a host-only circuit: described by its preprocessing and num_vars"""
        i = C.c_int(-1)
        _chk(lib().hg_circuit_insert_lasso_host(self.h, preprocessing.h, num_vars, C.byref(i)))
        self._keep.append(preprocessing)
        return i.value

    def verify_gkr(self, output_claims, transcript: "Keccak256Transcript", options=None):
        """gkr::verify_gkr (sk_encryption_circuit.rs:509-510) on the host. Returns per input node a list of (point, value); raises
        HgError where the reference returns Err / panics."""
        lens, pts, vals = self._claims_args(output_claims)
        opt = None if options is None else np.array(options, np.int32)
        _chk(lib().hg_gkr_verify(self.h, len(output_claims), _p(lens), _p(pts), _p(vals), transcript.h, _p(opt)))
        return self._read_input_claims()

    def insert_vanilla_arrays(self, arity, log2_sub, num_reps, has_const, consts, add_ptr, add_coef, add_in, add_wire,
                              mul_ptr=None, mul_coef=None, mul_in0=None, mul_w0=None, mul_in1=None, mul_w1=None):
        """VanillaNode::new with the gates already in CSR arrays (numpy); see include/hg_b200.h."""
        ng = len(has_const)
        z64, z32 = np.zeros(0, np.uint64), np.zeros(0, np.uint32)
        a = lambda v, t: np.ascontiguousarray(v if v is not None else (z64 if t == np.uint64 else z32), t)
        hc = np.ascontiguousarray(has_const, np.uint8)
        mp = a(mul_ptr if mul_ptr is not None else np.zeros(ng + 1, np.uint64), np.uint64)
        limbs = LIMBS[self.field]

        def felts(v):
            """field elements cross the ABI as `limbs` little-endian u64 words each: widen small (u64) coefficients"""
            v = a(v, np.uint64)
            if limbs == 1 or (v.ndim == 2 and v.shape[1] == limbs):
                return np.ascontiguousarray(v.reshape(-1))
            out = np.zeros((v.size, limbs), np.uint64)
            out[:, 0] = v.reshape(-1)
            return out.reshape(-1)

        arrs = [hc, felts(consts), a(add_ptr, np.uint64), felts(add_coef), a(add_in, np.uint32), a(add_wire, np.uint64), mp,
                felts(mul_coef), a(mul_in0, np.uint32), a(mul_w0, np.uint64), a(mul_in1, np.uint32), a(mul_w1, np.uint64)]
        i = C.c_int(-1)
        _chk(lib().hg_circuit_insert_vanilla(self.h, arity, log2_sub, num_reps, ng, *[_p(x) for x in arrs], C.byref(i)))
        return i.value

    def insert_vanilla(self, arity, log2_sub, gates, num_reps=1):
        """VanillaNode::new(input_arity, log2_sub_input_size, gates, num_reps) from a list of VanillaGate. A coefficient or constant is
        a Python int (reduced modulo the field's prime); a coefficient None is one, as Option<F> is in the reference."""
        limbs = LIMBS[self.field]
        p = GL_P if self.field == GOLDILOCKS else BN_R

        def felts(vals):
            out = np.zeros((len(vals), limbs), np.uint64)
            for i, v in enumerate(vals):
                v = (1 if v is None else int(v)) % p
                for j in range(limbs):
                    out[i, j] = (v >> (64 * j)) & 0xFFFFFFFFFFFFFFFF
            return out
        ng = len(gates)
        add_ptr, mul_ptr = np.zeros(ng + 1, np.uint64), np.zeros(ng + 1, np.uint64)
        adds = [a for g in gates for a in g.adds]
        muls = [m for g in gates for m in g.muls]
        add_ptr[1:] = np.cumsum([len(g.adds) for g in gates])
        mul_ptr[1:] = np.cumsum([len(g.muls) for g in gates])
        return self.insert_vanilla_arrays(
            arity, log2_sub, num_reps, [g.const is not None for g in gates], felts([0 if g.const is None else g.const for g in gates]),
            add_ptr, felts([c for c, _ in adds]), [w[0] for _, w in adds], [w[1] for _, w in adds],
            mul_ptr, felts([c for c, _, _ in muls]), [a[0] for _, a, _ in muls], [a[1] for _, a, _ in muls],
            [b[0] for _, _, b in muls], [b[1] for _, _, b in muls])

    def connect(self, frm, to):
        _chk(lib().hg_circuit_connect(self.h, frm, to))

    def evaluate(self, dev_inputs):
        ptrs = (C.c_void_p * len(dev_inputs))(*[b.ptr for b in dev_inputs])
        _chk(lib().hg_circuit_evaluate(self.h, ptrs, len(dev_inputs)))

    def evaluate_host(self, host_inputs):
        """Circuit::evaluate from host vectors (numpy uint64 arrays of canonical limbs; pinned memory makes the copies
        asynchronous). The arrays must stay alive until the next synchronising call (prove_gkr, mle_eval_batch)."""
        arrs = [np.ascontiguousarray(a, np.uint64) for a in host_inputs]
        limbs = LIMBS[self.field]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        lens = (C.c_size_t * len(arrs))(*[a.size // limbs for a in arrs])
        self._host_keepalive = arrs
        _chk(lib().hg_circuit_evaluate_host(self.h, ptrs, lens, len(arrs)))

    def node_value(self, node_id):
        p, n = C.c_void_p(), C.c_size_t(0)
        _chk(lib().hg_circuit_node_value(self.h, node_id, C.byref(p), C.byref(n)))
        return p.value, n.value

    def prove_gkr(self, output_claims, transcript: Keccak256Transcript, mode=MODE_PREFETCH):
        """output_claims: [(point [nv, el] uint64, value [el] uint64), ...]. Returns per input node a list of (point, value)."""
        lens, pts, vals = self._claims_args(output_claims)
        _chk(lib().hg_gkr_prove(self.h, len(output_claims), _p(lens), _p(pts), _p(vals), transcript.h, mode))
        return self._read_input_claims()

    def _read_input_claims(self):
        el = LIMBS[self.field] * DEGREE[self.field]
        out = []
        for i in range(lib().hg_gkr_num_inputs(self.h)):
            cl = []
            for k in range(lib().hg_gkr_num_input_claims(self.h, i)):
                nv = lib().hg_gkr_input_claim_num_vars(self.h, i, k)
                pt, v = np.zeros((nv, el), np.uint64), np.zeros(el, np.uint64)
                _chk(lib().hg_gkr_input_claim(self.h, i, k, _p(pt), _p(v)))
                cl.append((pt, v))
            out.append(cl)
        return out

    def timing(self):
        out = np.zeros(6, np.float64)
        lib().hg_gkr_timing(self.h, _p(out))
        d = dict(zip(("witness_enqueue_us", "challenges_us", "protocol_walk_us", "layer_enqueue_us", "gpu_wait_us", "serialise_us"), (float(x) for x in out)))
        d["ext_challenges"] = int(lib().hg_gkr_num_challenges(self.h))
        return d

    @property
    def shard_words(self):
        return int(lib().hg_gkr_shard_words(self.h))

    def _claims_args(self, output_claims):
        lens = np.array([len(p) for p, _ in output_claims], dtype=np.uint64)
        pts = np.concatenate([np.asarray(p, np.uint64).reshape(-1) for p, _ in output_claims] + [np.zeros(0, np.uint64)])
        vals = np.concatenate([np.asarray(v, np.uint64).reshape(-1) for _, v in output_claims] + [np.zeros(0, np.uint64)])
        return lens, np.ascontiguousarray(pts), np.ascontiguousarray(vals)

    def prove_gkr_shard_dev(self, output_claims, transcript: "Keccak256Transcript", rank: int, world: int, d_out_ptr: int, cap_words: int):
        """This rank's part of ONE gkr::prove_gkr split over `world` GPUs (hg_gkr_prove_shard_dev): its partial message buffer is
        copied to device memory at d_out_ptr. Returns the number of words."""
        lens, pts, vals = self._claims_args(output_claims)
        nw = C.c_size_t(0)
        _chk(lib().hg_gkr_prove_shard_dev(self.h, len(output_claims), _p(lens), _p(pts), _p(vals), transcript.h, rank, world, C.c_void_p(d_out_ptr), cap_words, C.byref(nw)))
        return int(nw.value)

    def emit_shard_dev(self, d_merged_ptr: int, n_words: int):
        """Rank 0: serialise the merged buffer into the transcript given to prove_gkr_shard_dev; returns the input claims."""
        _chk(lib().hg_gkr_emit_shard_dev(self.h, C.c_void_p(d_merged_ptr), n_words))
        return self._read_input_claims()

    def emit_shard_part_dev(self, d_merged_ptr: int, n_words: int, part: int, nparts: int) -> bytes:
        """Every rank: the bytes of range `part` of `nparts` of the proof (hg_gkr_emit_shard_part_dev). Concatenated in order they are the
        proof bytes that emit_shard_dev would have written; append them to rank 0's transcript (Keccak256Transcript.append_bytes)."""
        cap = 1 << 19
        buf = (C.c_uint8 * cap)()
        n = C.c_size_t(0)
        _chk(lib().hg_gkr_emit_shard_part_dev(self.h, C.c_void_p(d_merged_ptr), n_words, part, nparts, buf, cap, C.byref(n)))
        return bytes(memoryview(buf)[: n.value])

    def free(self):
        if self.h:
            lib().hg_circuit_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def build_bfv_circuit(c: Circuit, P, lasso_node=None, lasso_pp=None, lasso_num_vars=0):
    """BfvEncryptBlock::configure (sk_encryption_circuit.rs:86-293) through hg_bfv_configure: the same node order and connections for a
    device circuit (prover: lasso_node) or a host-only description (verifier: lasso_pp + num_vars). Returns the ids of a few nodes."""
    K = P.K
    u = lambda v: np.ascontiguousarray(np.array(v[:K], dtype=np.uint64))
    ids = np.zeros(6, np.int32)
    _chk(lib().hg_bfv_configure(c.h, P.log2_size, K, _p(u(P.QIS)), _p(u(P.K0IS)), _p(u(P.R1_BOUNDS)), _p(u(P.R2_BOUNDS)), P.S_BOUND, P.E_BOUND, P.K1_BOUND,
                                lasso_node.h if lasso_node is not None else None, lasso_pp.h if lasso_pp is not None else None, lasso_num_vars, _p(ids)))
    c._keep.extend([x for x in (lasso_node, lasso_pp) if x is not None])
    return dict(zip(("s", "e", "k1", "lasso_in", "lasso", "sum"), (int(x) for x in ids)))


class BfvSkEncryptVerifier:
    """BfvEncrypt::{setup, configure, verify} (sk_encryption_circuit.rs:300-363, :462-517) on the HOST: no GPU, no context."""

    def __init__(self, params, field=GOLDILOCKS):
        from . import witness
        self.P, self.field = params, field
        self.pp = LassoPreprocessing.preprocess(witness.lasso_lookup_bounds(params))
        self.circuit = Circuit(None, field)
        nv = witness.lasso_num_vars(params)
        self.ids = build_bfv_circuit(self.circuit, params, lasso_pp=self.pp, lasso_num_vars=nv)
        self.ct0is_log2_size = params.log2_size + (params.K.bit_length() - 1)

    def verify(self, host_inputs, host_ct0is, proof: bytes, options=None):
        """verify (:462-517): inputs in get_inputs order as canonical limbs. Raises HgError if the proof is rejected."""
        tr = Keccak256Transcript.from_proof(proof, self.field)                                   # :476
        L = self.ct0is_log2_size
        point = tr.squeeze_challenges(L)                                                          # :499
        value = mle_eval_host(self.field, host_ct0is, L, point)                                   # :500
        el = point.shape[1]
        claims = self.circuit.verify_gkr([(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)], tr, options)   # :504-510
        if len(claims) != len(host_inputs):
            raise HgError("verify: input count mismatch")
        for vec, cl in zip(host_inputs, claims):                                                  # :512-516
            for pt, v in cl:
                if not (mle_eval_host(self.field, vec, pt.shape[0], pt) == v).all():
                    raise HgError("verify: input claim does not match the input (sk_encryption_circuit.rs:515)")
        try:
            tr.read_felt_ext()
        except HgError:
            return claims
        raise HgError("verify: trailing bytes in proof")

    def verify_batch(self, ctx: Context, inputs_list, ct0is_list, proofs, options=None):
        """verify() for a batch of proofs on the device of `ctx` (hg_gkr_verify_batch), with the same verdicts. inputs_list[p] are
        proof p's inputs in get_inputs order and ct0is_list[p] its ct0is: host numpy arrays of canonical limbs, or DeviceBuffers in
        the library's representation (as hg_bfv_witness_generate writes them). proofs are bytes, or transcripts (from_proof or a
        CallbackTranscript with a read callback) positioned at the start of the proof. Returns [(ok, reason)] per proof."""
        n = len(proofs)
        if n == 0:
            return []
        bv = getattr(self, "_batch", None)
        if bv is None or bv.ctx is not ctx or bv.max_batch < n:
            if bv is not None:
                bv.free()
            bv = self._batch = GkrBatchVerifier(ctx, self.circuit, n)
        trs = [Keccak256Transcript.from_proof(p, self.field) if isinstance(p, (bytes, bytearray)) else p for p in proofs]
        L = self.ct0is_log2_size
        points = [t.squeeze_challenges(L) for t in trs]                                           # :499
        values = mle_eval_multi(ctx, list(ct0is_list), points)                                    # :500
        el = points[0].shape[1]
        oc = [[(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (points[p], values[p])] for p in range(n)]
        res = bv.verify_batch(trs, oc, inputs_list, options)                                      # :504-516
        out = []
        for t, (ok, why) in zip(trs, res):
            if ok:
                try:
                    t.read_felt_ext()
                    ok, why = False, "verify: trailing bytes in proof"
                except HgError:
                    pass
            out.append((ok, why))
        return out


class GkrBatchVerifier:
    """Batched device verifier of one circuit (hg_verifier_new): `desc` is a host-only Circuit description of any node shapes the
    host verifier takes (general Vanilla layers included); the verdicts are those of Circuit.verify_gkr plus the input-claim check."""

    def __init__(self, ctx: Context, desc: "Circuit", max_batch: int):
        self.ctx, self.desc, self.max_batch = ctx, desc, max_batch
        self.h = C.c_void_p()
        _chk(lib().hg_verifier_new(ctx.h, desc.h, max_batch, C.byref(self.h)))
        self.input_lens = [int(lib().hg_verifier_input_len(self.h, i)) for i in range(lib().hg_verifier_num_inputs(self.h))]

    def verify_batch(self, transcripts, output_claims, inputs, options=None):
        """transcripts: one per proof; output_claims: per proof a list of (point, value), the same point lengths for every proof;
        inputs: per proof the input tables in insertion order, all DeviceBuffer / DeviceView or all host numpy arrays.
        Returns [(ok, reason)] per proof."""
        n = len(transcripts)
        if n == 0:
            return []
        lens = np.array([len(p) for p, _ in output_claims[0]], np.uint64)
        if len(output_claims) != n or any([len(p) for p, _ in oc] != list(lens) for oc in output_claims):
            raise HgError("verify_batch: one list of output claims per proof, with the same point lengths for every proof")
        pts = np.ascontiguousarray(np.concatenate([np.asarray(p, np.uint64).reshape(-1) for oc in output_claims for p, _ in oc] + [np.zeros(0, np.uint64)]))
        vals = np.ascontiguousarray(np.concatenate([np.asarray(v, np.uint64).reshape(-1) for oc in output_claims for _, v in oc] + [np.zeros(0, np.uint64)]))
        flat = [t for ins in inputs for t in ins]
        on_dev = len(flat) > 0 and not isinstance(flat[0], np.ndarray)
        keep = [t if on_dev else np.ascontiguousarray(t, np.uint64).reshape(-1) for t in flat]
        if len(inputs) != n or any(len(ins) != len(self.input_lens) for ins in inputs) or \
                (not on_dev and any(t.size != LIMBS[self.ctx.field] * m for ins in inputs for t, m in zip(ins, self.input_lens))):
            raise HgError("verify_batch: one list of inputs per proof, each input of its node's size")
        ptrs = (C.c_void_p * max(len(keep), 1))(*[(t.ptr if on_dev else t.ctypes.data) for t in keep])
        trs = (C.c_void_p * n)(*[t.h.value if isinstance(t.h, C.c_void_p) else t.h for t in transcripts])
        status = np.zeros(n, np.int32)
        opt = None if options is None else np.array(options, np.int32)
        _chk(lib().hg_gkr_verify_batch(self.h, n, trs, len(lens), _p(lens), _p(pts), _p(vals), ptrs, 1 if on_dev else 0, _p(opt), _p(status)))
        return [(bool(status[p]), lib().hg_verifier_reason(self.h, p).decode()) for p in range(n)]

    def timing(self):
        """host microseconds of the last batch: replays of every proof, device stages (enqueue and wait), closing the records"""
        out = np.zeros(3, np.float64)
        lib().hg_verifier_timing(self.h, _p(out))
        return dict(zip(("replay_us", "device_us", "close_us"), (float(x) for x in out)))

    def free(self):
        if self.h:
            lib().hg_verifier_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class BfvSkEncryptProver:
    """BfvEncrypt::{setup, configure, prove} (sk_encryption_circuit.rs:300-460) with every table on the device."""

    def __init__(self, ctx: Context, params):
        from . import witness
        P = self.P = params
        self.ctx = ctx
        self.pp = LassoPreprocessing.preprocess(witness.lasso_lookup_bounds(P))                 # setup(): :327-341
        self.lasso = LassoNode(ctx, self.pp, witness.lasso_num_vars(P), witness.lasso_lookup_segments(P))
        c = self.circuit = Circuit(ctx)                                                         # configure(): :351-363, :86-293
        self.ids = build_bfv_circuit(c, P, lasso_node=self.lasso)                               # hg_bfv_configure
        self.ct0is_log2_size = P.log2_size + (P.K.bit_length() - 1)                             # :519-522

    def upload_inputs(self, ins):
        u = lambda v: DeviceBuffer.from_numpy(self.ctx, np.asarray(v, dtype=np.uint64).reshape(-1))
        return [u(ins["s"]), u(ins["e"]), u(ins["k1"])] + [u(a) for a in ins["ais"]] + [u(a) for a in ins["r1is"]] + [u(ins["r2is"])]

    def prove_host(self, host_inputs, host_ct0is, mode=MODE_PREFETCH):
        """BfvEncrypt::prove (:417-460) from HOST vectors (get_inputs order: s, e, k1, ais.., r1is.., r2is; ct0is concatenated):
        uploads, circuit.evaluate, output claim, prove_gkr. Returns (proof bytes, input claims)."""
        ct = np.ascontiguousarray(host_ct0is, np.uint64).reshape(-1)
        if getattr(self, "_d_ct", None) is None or self._d_ct.nbytes != ct.nbytes:
            self._d_ct = DeviceBuffer(self.ctx, ct.nbytes)
        tr = Keccak256Transcript(self.ctx.field)                                                 # :431
        self.circuit.evaluate_host(host_inputs)                                                  # :438-442
        self._d_ct.upload_async(ct)
        if self.ctx.field == BN254:
            _chk(lib().hg_field_encode(self.ctx.h, self._d_ct.ptr, ct.size // LIMBS[BN254]))
        point = tr.squeeze_challenges(self.ct0is_log2_size)                                      # :445
        value = mle_eval_batch(self.ctx, self._d_ct, 1, self.ct0is_log2_size, point)[0]          # :446
        el = point.shape[1]
        claims = self.circuit.prove_gkr([(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)], tr, mode)   # :450-457
        return tr.into_proof(), claims                                                           # :459

    def prove(self, dev_inputs, d_ct0is: DeviceBuffer, mode=MODE_PREFETCH):
        """BfvEncrypt::prove (:417-460). Returns (proof bytes, input claims)."""
        tr = Keccak256Transcript(self.ctx.field)                                                 # :431
        self.circuit.evaluate(dev_inputs)                                                        # :442
        point = tr.squeeze_challenges(self.ct0is_log2_size)                                      # :445
        value = mle_eval_batch(self.ctx, d_ct0is, 1, self.ct0is_log2_size, point)[0]             # :446
        el = point.shape[1]
        claims = self.circuit.prove_gkr([(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point, value)], tr, mode)   # :450-457
        return tr.into_proof(), claims                                                           # :459


# ------------------------------------------------------------------------------------------------ BFV public-key encryption
def build_bfv_pk_circuit(c: Circuit, P, lasso_node=None, lasso_pp=None, lasso_num_vars=0):
    """The circuit of the BFV public-key-encryption relation (params.BfvPkEncryptConstants) through hg_bfv_pk_configure, for a device
    circuit (prover: lasso_node) or a host-only description (verifier: lasso_pp + num_vars). Returns the ids of a few nodes."""
    K = P.K
    u = lambda v: np.ascontiguousarray(np.array(v[:K], dtype=np.uint64))
    ids = np.zeros(8, np.int32)
    _chk(lib().hg_bfv_pk_configure(c.h, P.log2_size, K, _p(u(P.QIS)), _p(u(P.K0IS)), _p(u(P.R1_BOUNDS)), _p(u(P.R2_BOUNDS)), _p(u(P.P1_BOUNDS)),
                                   _p(u(P.P2_BOUNDS)), P.U_BOUND, P.E_BOUND, P.K1_BOUND, lasso_node.h if lasso_node is not None else None,
                                   lasso_pp.h if lasso_pp is not None else None, lasso_num_vars, _p(ids)))
    c._keep.extend([x for x in (lasso_node, lasso_pp) if x is not None])
    return dict(zip(("u", "e0", "e1", "k1", "lasso_in", "lasso", "sum0", "sum1"), (int(x) for x in ids)))


def _pk_output_claims(point0, v0, point1, v1):
    """the Lasso node's empty claim, then sum0 = ct0is at point0 and sum1 = ct1is at point1"""
    el = point0.shape[1]
    return [(np.zeros((0, el), np.uint64), np.zeros(el, np.uint64)), (point0, v0), (point1, v1)]


class BfvPkEncryptProver:
    """Proves the BFV public-key-encryption relation with every table on the device. A proof: a fresh transcript, circuit.evaluate,
    point0 (L + log2 K challenges) and v0 = MLE(ct0is)(point0), point1 and v1 = MLE(ct1is)(point1) the same way, prove_gkr with the
    output claims [(), 0], [point0, v0], [point1, v1] (the Lasso node, sum0, sum1)."""

    def __init__(self, ctx: Context, params):
        from . import witness
        P = self.P = params
        self.ctx = ctx
        self.pp = LassoPreprocessing.preprocess(witness.pk_lasso_lookup_bounds(P))
        self.lasso = LassoNode(ctx, self.pp, witness.pk_lasso_num_vars(P), witness.pk_lasso_lookup_segments(P))
        c = self.circuit = Circuit(ctx)
        self.ids = build_bfv_pk_circuit(c, P, lasso_node=self.lasso)
        self.ct_log2_size = P.log2_size + (P.K.bit_length() - 1)

    def upload_inputs(self, ins):
        """pk_get_inputs' dict -> device buffers in input-node order"""
        from . import witness
        return [DeviceBuffer.from_numpy(self.ctx, np.asarray(v, dtype=np.uint64).reshape(-1)) for v in witness.pk_input_list(ins)]

    def _prove(self, d_ct0is, d_ct1is, mode, transcript):
        tr = Keccak256Transcript(self.ctx.field) if transcript is None else transcript
        L = self.ct_log2_size
        point0 = tr.squeeze_challenges(L)
        v0 = mle_eval_batch(self.ctx, d_ct0is, 1, L, point0)[0]
        point1 = tr.squeeze_challenges(L)
        v1 = mle_eval_batch(self.ctx, d_ct1is, 1, L, point1)[0]
        claims = self.circuit.prove_gkr(_pk_output_claims(point0, v0, point1, v1), tr, mode)
        return tr.into_proof(), claims

    def prove(self, dev_inputs, d_ct0is, d_ct1is, mode=MODE_PREFETCH, transcript=None):
        """dev_inputs in input-node order, d_ct0is / d_ct1is device buffers in the library's representation (as
        hg_bfv_pk_witness_generate writes them). transcript: a fresh one by default, or a caller-owned CallbackTranscript.
        Returns (proof bytes, input claims)."""
        self.circuit.evaluate(dev_inputs)
        return self._prove(d_ct0is, d_ct1is, mode, transcript)

    def prove_host(self, host_inputs, host_ct0is, host_ct1is, mode=MODE_PREFETCH, transcript=None):
        """prove() from HOST vectors of canonical limbs (input-node order; ct0is and ct1is concatenated over the moduli)."""
        cts = [np.ascontiguousarray(c, np.uint64).reshape(-1) for c in (host_ct0is, host_ct1is)]
        if getattr(self, "_d_ct", None) is None or self._d_ct[0].nbytes != cts[0].nbytes:
            self._d_ct = [DeviceBuffer(self.ctx, cts[0].nbytes) for _ in range(2)]
        self.circuit.evaluate_host(host_inputs)
        for d, c in zip(self._d_ct, cts):
            d.upload(c)
            if self.ctx.field == BN254:
                _chk(lib().hg_field_encode(self.ctx.h, d.ptr, c.size // LIMBS[BN254]))
        return self._prove(self._d_ct[0], self._d_ct[1], mode, transcript)


class BfvPkEncryptVerifier:
    """Verifies proofs of BfvPkEncryptProver on the HOST (verify: no GPU, no context) or in batches on a device (verify_batch)."""

    def __init__(self, params, field=GOLDILOCKS):
        from . import witness
        self.P, self.field = params, field
        self.pp = LassoPreprocessing.preprocess(witness.pk_lasso_lookup_bounds(params))
        self.circuit = Circuit(None, field)
        self.ids = build_bfv_pk_circuit(self.circuit, params, lasso_pp=self.pp, lasso_num_vars=witness.pk_lasso_num_vars(params))
        self.ct_log2_size = params.log2_size + (params.K.bit_length() - 1)
        self._el_bytes = 8 * LIMBS[field] * DEGREE[field]   # a proof is whole extension elements: a shorter tail is trailing bytes

    def verify(self, host_inputs, host_ct0is, host_ct1is, proof: bytes, options=None):
        """host_inputs in input-node order as canonical limbs. Raises HgError if the proof is rejected; returns the input claims."""
        if len(proof) % self._el_bytes:
            raise HgError("verify: trailing bytes in proof")
        tr = Keccak256Transcript.from_proof(proof, self.field)
        L = self.ct_log2_size
        point0 = tr.squeeze_challenges(L)
        v0 = mle_eval_host(self.field, host_ct0is, L, point0)
        point1 = tr.squeeze_challenges(L)
        v1 = mle_eval_host(self.field, host_ct1is, L, point1)
        claims = self.circuit.verify_gkr(_pk_output_claims(point0, v0, point1, v1), tr, options)
        if len(claims) != len(host_inputs):
            raise HgError("verify: input count mismatch")
        for vec, cl in zip(host_inputs, claims):
            for pt, v in cl:
                if not (mle_eval_host(self.field, vec, pt.shape[0], pt) == v).all():
                    raise HgError("verify: input claim does not match the input")
        try:
            tr.read_felt_ext()
        except HgError:
            return claims
        raise HgError("verify: trailing bytes in proof")

    def verify_batch(self, ctx: Context, inputs_list, ct0is_list, ct1is_list, proofs, options=None):
        """verify() for a batch of proofs on the device of `ctx` (GkrBatchVerifier), with the same verdicts. inputs_list[p], ct0is_list[p]
        and ct1is_list[p] belong to proof p: host numpy arrays of canonical limbs, or device buffers in the library's representation.
        proofs are bytes, or transcripts positioned at the start of the proof. Returns [(ok, reason)] per proof."""
        n = len(proofs)
        if n == 0:
            return []
        bv = getattr(self, "_batch", None)
        if bv is None or bv.ctx is not ctx or bv.max_batch < n:
            if bv is not None:
                bv.free()
            bv = self._batch = GkrBatchVerifier(ctx, self.circuit, n)
        trs = [Keccak256Transcript.from_proof(p, self.field) if isinstance(p, (bytes, bytearray)) else p for p in proofs]
        L = self.ct_log2_size
        points = []
        for t in trs:
            points += [t.squeeze_challenges(L), t.squeeze_challenges(L)]
        tables = [c for pair in zip(ct0is_list, ct1is_list) for c in pair]
        values = mle_eval_multi(ctx, tables, points)
        oc = [_pk_output_claims(points[2 * p], values[2 * p], points[2 * p + 1], values[2 * p + 1]) for p in range(n)]
        res = bv.verify_batch(trs, oc, inputs_list, options)
        out = []
        for t, pr, (ok, why) in zip(trs, proofs, res):
            if ok:
                try:
                    t.read_felt_ext()
                    ok, why = False, "verify: trailing bytes in proof"
                except HgError:
                    if isinstance(pr, (bytes, bytearray)) and len(pr) % self._el_bytes:
                        ok, why = False, "verify: trailing bytes in proof"
            out.append((ok, why))
        return out
