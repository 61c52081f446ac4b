"""Host-side mirror of the reference's verifier interfaces over the C ABI.

  RiscZeroVerifier  <- IRiscZeroVerifier, /root/reference/contracts/src/risc0/verifier.rs:18-42
  Sp1Verifier       <- ISp1Verifier,      /root/reference/contracts/src/sp1/verifier.rs:16-29
  Groth16Verifier   <- Groth16Verifier::verify_proof_with_key, contracts/src/common/groth16.rs:23-49
  RiscZeroVerifierRouter, Sp1VerifierGateway <- the routers that forward a seal / proof to the verifier version its first 4 bytes select
  VerificationKey   <- contracts/src/common/types.rs:17-23

Same method names, argument meaning and error behaviour: the single-proof calls return on success and
raise the reference's custom error (errors.py; `.payload` is the exact revert byte string) otherwise;
`verify` never returns False (risc0/verifier.rs:191-195).  The `*_batch` variants take N proofs and
return N status bytes (numpy uint8; 0 = accept).  All verification work runs in the sm_100a kernels.
"""
import ctypes as C

import numpy as np

from . import _native as N
from . import errors as E


def _offsets(blobs):
    off = np.zeros(len(blobs) + 1, dtype=np.uint64)
    if len(blobs):
        off[1:] = np.cumsum(np.fromiter((len(b) for b in blobs), dtype=np.uint64, count=len(blobs)))
    return off


def _dev_array(devices):
    if not devices:
        return None, 0
    arr = (C.c_int * len(devices))(*devices)
    return arr, len(devices)


def _tune(handle_vk, option, value):
    """zkv_vk_tune on a key handle: returns the previous value; value=None only reads the setting (include/zkv.h lists the options)."""
    r = N.lib().zkv_vk_tune(handle_vk, N.TUNE[option], N.ZKV_TUNE_QUERY if value is None else int(value))
    if r < 0:
        N.check(r)
    return r


def _need32(**kw):
    """the reference takes typed B256 / FixedBytes<32> values (risc0/verifier.rs:78-104, sp1/verifier.rs:39-46): anything else is a caller bug"""
    for name, v in kw.items():
        if len(v) != 32:
            raise ValueError("%s must be exactly 32 bytes, got %d" % (name, len(v)))


def _need32_each(n, **kw):
    for name, seq in kw.items():
        if len(seq) != n:
            raise ValueError("%s: expected %d entries, got %d" % (name, n, len(seq)))
        for v in seq:
            if len(v) != 32:
                raise ValueError("every element of %s must be exactly 32 bytes" % name)


class VerificationKey:
    """common/types.rs:17-23.  Points as EVM words: alpha 64 B, beta/gamma/delta 128 B each in wire order
    x[0],x[1],y[0],y[1]; ic = list of 64-byte points."""

    def __init__(self, vm_type, alpha, beta, gamma, delta, ic, devices=None):
        self.vm_type, self.n_ic = vm_type, len(ic)
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_vk_load(vm_type, alpha, beta, gamma, delta, b"".join(ic), len(ic), arr, nd, C.byref(self._h)))

    @classmethod
    def risc0(cls, devices=None):
        self = cls.__new__(cls); self.vm_type, self.n_ic, self._h = N.ZKV_VM_RISC0, 6, C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_vk_load_risc0(arr, nd, C.byref(self._h)))
        return self

    @classmethod
    def sp1(cls, devices=None):
        self = cls.__new__(cls); self.vm_type, self.n_ic, self._h = N.ZKV_VM_SP1, 3, C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_vk_load_sp1(arr, nd, C.byref(self._h)))
        return self

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_vk_free(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stage_ms(self, device=0):
        out = (C.c_float * 5)()
        n = N.lib().zkv_last_stage_ms(self._h, device, out, 5)
        return dict(zip(("decode_hash", "vk_x", "g2_check", "miller", "final_exp"), list(out)[:max(n, 0)]))

    def tune(self, option, value=None):
        """Per-key tuning (overlap, miller_segments, final_exp_stages); returns the previous value.  normalised_lines and layout are
        fixed at 1: they read 1, and setting 0 raises ZkvError (the round-1 kernels and the unscaled verification lines were removed)."""
        return _tune(self._h, option, value)


class VerificationKeySet:
    """1..256 loaded VerificationKeys for Groth16Verifier.verify_batch_keys (zkv_vkset_create).  Every key must be loaded on every
    device of the set; the set keeps references to its keys so that they outlive it."""

    def __init__(self, keys, devices=None):
        self.keys = list(keys)
        self._h = C.c_void_p()
        handles = (C.c_void_p * max(len(self.keys), 1))(*[k._h for k in self.keys])
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_vkset_create(handles, len(self.keys), arr, nd, C.byref(self._h)))

    def __len__(self):
        return len(self.keys)

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_vkset_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def raw_key_bytes(alpha, beta, gamma, delta, ic):
    """One key in the byte form of RawKeyVerifier / zkv_groth16_verify_batch_rawkeys: alpha (64 B), beta, gamma, delta (128 B each, wire order),
    then the IC points (64 B each)."""
    return bytes(alpha) + bytes(beta) + bytes(gamma) + bytes(delta) + b"".join(bytes(p) for p in ic)


class RawKeyVerifier:
    """Groth16 verification under keys passed as bytes with each call (zkv_rawkey_create): nothing is loaded, so every proof may bring its own
    key.  The handle owns a workspace and streams per device (devices=None -> device 0)."""

    def __init__(self, devices=None):
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_rawkey_create(arr, nd, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_rawkey_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _pack_keys(keys):
        """keys: (vm_type, alpha, beta, gamma, delta, ic) tuples -> key blob, key offsets (uint64), vm bytes (uint8)"""
        blobs = [raw_key_bytes(*k[1:]) for k in keys]
        return b"".join(blobs), _offsets(blobs), np.array([k[0] for k in keys], dtype=np.uint8)

    @staticmethod
    def _pack_signals(signals):
        off = _offsets([b"\0" * 32 * len(s) for s in signals]) // 32
        return b"".join(int(v).to_bytes(32, "big") for s in signals for v in s), off

    def verify_batch(self, keys, key_idx, proofs, signals):
        """Proof i (256 B; one n x 256-byte blob or a list of 256-byte proofs) under keys[key_idx[i]] with the integers signals[i] -> n status
        bytes (ZKV_OK or ZKV_VERIFICATION_FAILED): what verify_proof_with_key returns for each."""
        n = len(key_idx)
        if len(signals) != n:
            raise ValueError("signals: expected %d entries, got %d" % (n, len(signals)))
        kb, ko, kv = self._pack_keys(keys)
        sb, so = self._pack_signals(signals)
        pr = proofs if isinstance(proofs, (bytes, bytearray, np.ndarray)) else b"".join(proofs)
        return self.verify_batch_packed(kb, ko, kv, key_idx, pr, sb, so)

    def verify_batch_packed(self, key_blob, key_off, key_vm, key_idx, proofs, sig_blob, sig_off, status_out=None):
        """Zero-copy form: key_blob with n_keys + 1 uint64 byte offsets key_off and n_keys vm bytes; key_idx (uint32), proofs n x 256 B,
        sig_blob = the signals as 32-byte words with n + 1 uint64 word offsets sig_off."""
        key_off = np.ascontiguousarray(key_off, dtype=np.uint64)
        key_vm = np.ascontiguousarray(key_vm, dtype=np.uint8)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        sig_off = np.ascontiguousarray(sig_off, dtype=np.uint64)
        n, nk = len(key_idx), len(key_vm)
        if len(key_off) != nk + 1:
            raise ValueError("key_off: expected %d offsets, got %d" % (nk + 1, len(key_off)))
        if (proofs.nbytes if isinstance(proofs, np.ndarray) else len(proofs)) != 256 * n:
            raise ValueError("proofs: expected %d bytes" % (256 * n))
        if len(sig_off) != n + 1:
            raise ValueError("sig_off: expected %d offsets, got %d" % (n + 1, len(sig_off)))
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        nkb = key_blob.nbytes if isinstance(key_blob, np.ndarray) else len(key_blob)
        nsb = sig_blob.nbytes if isinstance(sig_blob, np.ndarray) else len(sig_blob)
        N.check(N.lib().zkv_groth16_verify_batch_rawkeys(self._h, N.buf(key_blob) if nkb else None, key_off.ctypes.data, key_vm.ctypes.data if nk else None, nk,
                                                         key_idx.ctypes.data, N.buf(proofs) if n else None, N.buf(sig_blob) if nsb else None,
                                                         sig_off.ctypes.data, n, st.ctypes.data))
        return st

    def verify_batch_device(self, device, d_keys, d_key_off, d_key_vm, n_keys, d_key_idx, d_proofs, d_signals, d_sig_off, n, d_status, stream=None):
        """Inputs already in HBM (raw device pointers as ints; the offsets index d_keys and d_signals directly); asynchronous on `stream`.
        A malformed key, a bad key index or a decreasing offset fails that proof."""
        N.check(N.lib().zkv_groth16_verify_batch_rawkeys_device(self._h, device, d_keys, d_key_off, d_key_vm, n_keys, d_key_idx, d_proofs, d_signals,
                                                                d_sig_off, n, d_status, stream))

    def vk_x_batch(self, keys, key_idx, signals):
        """vk_x of proof i under keys[key_idx[i]] (keys as for verify_batch; the vm byte is not used) -> (n x 64-byte points, n failed flags)"""
        n = len(key_idx)
        kb, ko, _ = self._pack_keys(keys)
        sb, so = self._pack_signals(signals)
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        out = C.create_string_buffer(64 * max(n, 1))
        failed = np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_vk_x_rawkeys_batch(self._h, N.buf(kb) if kb else None, ko.ctypes.data, len(keys), key_idx.ctypes.data,
                                               N.buf(sb) if sb else None, so.ctypes.data, n, out, failed.ctypes.data))
        return [out.raw[64 * i:64 * i + 64] for i in range(n)], failed


_raw_default = None


class Groth16Verifier:
    """common/groth16.rs:16-49."""

    @staticmethod
    def verify_proof_with_raw_key(vm_type, alpha, beta, gamma, delta, ic, a, b, c, signals):
        """verify_proof_with_key(vm, &vk, a, b, c, &signals) with the key as bytes (alpha 64 B, beta / gamma / delta 128 B in wire order, ic a
        list of 64-byte points), nothing loaded; a, b, c, signals as for verify_proof_with_key.  Returns bool.  Runs on device 0."""
        global _raw_default
        if _raw_default is None:
            _raw_default = RawKeyVerifier()
        w = lambda v: int(v).to_bytes(32, "big")
        proof = w(a[0]) + w(a[1]) + w(b[0][0]) + w(b[0][1]) + w(b[1][0]) + w(b[1][1]) + w(c[0]) + w(c[1])
        st = _raw_default.verify_batch([(vm_type, alpha, beta, gamma, delta, ic)], [0], proof, [list(signals)])
        return bool(st[0] == N.ZKV_OK)

    @staticmethod
    def verify_proof_with_key(vk, a, b, c, signals):
        """a = [x, y], b = [[x0, x1], [y0, y1]], c = [x, y], signals: integers (U256).  Returns bool."""
        w = lambda v: int(v).to_bytes(32, "big")
        proof = w(a[0]) + w(a[1]) + w(b[0][0]) + w(b[0][1]) + w(b[1][0]) + w(b[1][1]) + w(c[0]) + w(c[1])
        st = Groth16Verifier.verify_batch(vk, proof, b"".join(w(s) for s in signals), len(signals), 1)
        return bool(st[0] == N.ZKV_OK)

    @staticmethod
    def verify_batch(vk, proofs, signals, k, n):
        """proofs: n x 256 B, signals: n x k x 32 B -> n status bytes."""
        st = np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_groth16_verify_batch(vk._h, N.buf(proofs), N.buf(signals) if k else None, k, n, st.ctypes.data))
        return st

    @staticmethod
    def verify_batch_keys(keyset, key_idx, proofs, signals):
        """N verify_proof_with_key calls in one batch: proof i (256 B; `proofs` is one n x 256-byte blob or a list of 256-byte proofs) under
        keyset.keys[key_idx[i]] with the integers signals[i] -> n status bytes.  A signal count other than that key's n_ic - 1 fails that proof."""
        n = len(key_idx)
        if len(signals) != n:
            raise ValueError("signals: expected %d entries, got %d" % (n, len(signals)))
        off = np.zeros(n + 1, dtype=np.uint64)
        if n:
            off[1:] = np.cumsum(np.fromiter((len(s) for s in signals), dtype=np.uint64, count=n))
        blob = b"".join(int(v).to_bytes(32, "big") for s in signals for v in s)
        return Groth16Verifier.verify_batch_keys_packed(keyset, key_idx, proofs if isinstance(proofs, (bytes, bytearray, np.ndarray)) else b"".join(proofs), blob, off)

    @staticmethod
    def verify_batch_keys_packed(keyset, key_idx, proofs, sig_blob, sig_off, status_out=None):
        """Zero-copy form: key_idx (uint32), proofs n x 256 B, sig_blob = the signals as 32-byte words, sig_off = n + 1 uint64 word offsets."""
        key_idx = np.ascontiguousarray(key_idx, dtype=np.uint32)
        n = len(key_idx)
        sig_off = np.ascontiguousarray(sig_off, dtype=np.uint64)
        if (proofs.nbytes if isinstance(proofs, np.ndarray) else len(proofs)) != 256 * n:
            raise ValueError("proofs: expected %d bytes" % (256 * n))
        if len(sig_off) != n + 1:
            raise ValueError("sig_off: expected %d offsets, got %d" % (n + 1, len(sig_off)))
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_groth16_verify_batch_keys(keyset._h, key_idx.ctypes.data, N.buf(proofs) if n else None,
                                                      N.buf(sig_blob) if len(sig_blob) else None, sig_off.ctypes.data, n, st.ctypes.data))
        return st

    @staticmethod
    def verify_batch_keys_device(keyset, device, d_key_idx, d_proofs, d_signals, d_sig_off, n, d_status, stream=None):
        """Inputs already in HBM (raw device pointers as ints: n uint32 key indices, n x 256-byte proofs, signal words, n + 1 uint64 offsets
        into them); asynchronous on `stream`."""
        N.check(N.lib().zkv_groth16_verify_batch_keys_device(keyset._h, device, d_key_idx, d_proofs, d_signals, d_sig_off, n, d_status, stream))


class RiscZeroVerifier:
    """risc0/verifier.rs:44-124 (storage + IRiscZeroVerifier)."""

    def __init__(self, vk=None, devices=None):
        self._vk = vk
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_risc0_create(vk._h if vk is not None else None, arr, nd, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_risc0_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- IRiscZeroVerifier
    def tune(self, option, value=None):
        return _tune(N.lib().zkv_risc0_vk(self._h), option, value)

    def initialize(self, control_root, bn254_control_id):
        _need32(control_root=control_root, bn254_control_id=bn254_control_id)
        rc = N.lib().zkv_risc0_initialize(self._h, control_root, bn254_control_id)
        if rc == N.ZKV_ERR_STATE:
            raise E.AlreadyInitialized()
        N.check(rc)

    def verify(self, seal, image_id, journal_digest):
        _need32(image_id=image_id, journal_digest=journal_digest)
        st = C.c_uint8(0)
        N.check(N.lib().zkv_risc0_verify(self._h, seal, len(seal), image_id, journal_digest, C.byref(st)))
        return self._result(st.value, seal)

    def verify_integrity(self, receipt_seal, claim_digest):
        _need32(claim_digest=claim_digest)
        st = C.c_uint8(0)
        N.check(N.lib().zkv_risc0_verify_integrity(self._h, receipt_seal, len(receipt_seal), claim_digest, C.byref(st)))
        return self._result(st.value, receipt_seal)

    def get_selector(self):
        out = C.create_string_buffer(4); N.check(N.lib().zkv_risc0_get_selector(self._h, out)); return out.raw

    def get_control_root(self):
        a, b = C.create_string_buffer(16), C.create_string_buffer(16)
        N.check(N.lib().zkv_risc0_get_control_root(self._h, a, b)); return a.raw, b.raw

    def get_bn254_control_id(self):
        out = C.create_string_buffer(32); N.check(N.lib().zkv_risc0_get_bn254_control_id(self._h, out)); return out.raw

    def get_verifier_key_digest(self):
        out = C.create_string_buffer(32); N.check(N.lib().zkv_risc0_get_verifier_key_digest(self._h, out)); return out.raw

    def is_initialized(self):
        return bool(N.lib().zkv_risc0_is_initialized(self._h))

    # -- batch variants
    def verify_batch(self, seals, image_ids, journal_digests):
        n = len(seals)
        _need32_each(n, image_ids=image_ids, journal_digests=journal_digests)
        st = np.zeros(n, dtype=np.uint8)
        off = _offsets(seals)
        N.check(N.lib().zkv_risc0_verify_batch(self._h, b"".join(seals) or b"\0", off.ctypes.data, b"".join(image_ids) or b"\0",
                                               b"".join(journal_digests) or b"\0", n, st.ctypes.data))
        return st

    def verify_integrity_batch(self, seals, claim_digests):
        n = len(seals)
        _need32_each(n, claim_digests=claim_digests)
        st = np.zeros(n, dtype=np.uint8)
        off = _offsets(seals)
        N.check(N.lib().zkv_risc0_verify_integrity_batch(self._h, b"".join(seals) or b"\0", off.ctypes.data, b"".join(claim_digests) or b"\0", n, st.ctypes.data))
        return st

    def verify_batch_packed(self, seal_blob, seal_off, image_ids, journal_digests, n, status_out=None):
        """Zero-copy form: contiguous buffers (bytes or numpy uint8) + numpy uint64 offsets."""
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_risc0_verify_batch(self._h, N.buf(seal_blob), seal_off.ctypes.data, N.buf(image_ids), N.buf(journal_digests), n, st.ctypes.data))
        return st

    def verify_batch_device(self, device, d_seals260, d_image_ids, d_journal_digests, n, d_status, stream=None):
        """Inputs already in HBM (raw device pointers as ints); asynchronous on `stream`."""
        N.check(N.lib().zkv_risc0_verify_batch_device(self._h, device, d_seals260, d_image_ids, d_journal_digests, n, d_status, stream))

    def stage_ms(self, device=0):
        out = (C.c_float * 5)()
        n = N.lib().zkv_last_stage_ms(N.lib().zkv_risc0_vk(self._h), device, out, 5)
        return dict(zip(("decode_hash", "vk_x", "g2_check", "miller", "final_exp"), list(out)[:max(n, 0)]))

    def _result(self, status, seal):
        if status == N.ZKV_OK:
            return True
        if status == N.ZKV_INVALID_INITIALIZATION:
            raise E.InvalidInitialization()
        if status == N.ZKV_INVALID_PROOF_DATA:
            raise E.InvalidProofData()
        if status == N.ZKV_SELECTOR_MISMATCH:
            raise E.SelectorMismatch(seal[:4], self.get_selector())
        raise E.VerificationFailed()


class Sp1Verifier:
    """sp1/verifier.rs:31-54 (ISp1Verifier).  verifier_hash / version: another verifier version's 32-byte hash (its first 4 bytes are
    the selector) and version string, with that version's key as `vk` (None: the embedded v5 key); by default the embedded v5 ones."""

    def __init__(self, vk=None, devices=None, verifier_hash=None, version=None):
        self._vk = vk
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        if verifier_hash is None:
            if version is not None:
                raise ValueError("version needs the verifier_hash of that version")
            N.check(N.lib().zkv_sp1_create(vk._h if vk is not None else None, arr, nd, C.byref(self._h)))
        else:
            _need32(verifier_hash=verifier_hash)
            N.check(N.lib().zkv_sp1_create_version(vk._h if vk is not None else None, bytes(verifier_hash), (version or "").encode(), arr, nd, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_sp1_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def tune(self, option, value=None):
        return _tune(N.lib().zkv_sp1_vk(self._h), option, value)

    def verify_proof(self, program_vkey, public_values, proof_bytes):
        _need32(program_vkey=program_vkey)
        st = C.c_uint8(0)
        N.check(N.lib().zkv_sp1_verify_proof(self._h, program_vkey, public_values or b"\0", len(public_values), proof_bytes or b"\0", len(proof_bytes), C.byref(st)))
        if st.value == N.ZKV_OK:
            return None
        if st.value == N.ZKV_INVALID_PROOF_DATA:
            raise E.InvalidProofData()
        if st.value == N.ZKV_SELECTOR_MISMATCH:
            raise E.WrongVerifierSelector(proof_bytes[:4], self.verifier_hash()[:4])
        raise E.VerificationFailed()

    def verifier_hash(self):
        out = C.create_string_buffer(32); N.check(N.lib().zkv_sp1_verifier_hash(self._h, out)); return out.raw

    def version(self):
        return N.lib().zkv_sp1_version(self._h).decode()

    def verify_batch(self, program_vkeys, public_values, proofs):
        n = len(proofs)
        _need32_each(n, program_vkeys=program_vkeys)
        if len(public_values) != n:
            raise ValueError("public_values: expected %d entries, got %d" % (n, len(public_values)))
        st = np.zeros(n, dtype=np.uint8)
        po, vo = _offsets(proofs), _offsets(public_values)
        N.check(N.lib().zkv_sp1_verify_batch(self._h, b"".join(program_vkeys) or b"\0", b"".join(public_values) or b"\0", vo.ctypes.data,
                                             b"".join(proofs) or b"\0", po.ctypes.data, n, st.ctypes.data))
        return st

    def verify_batch_packed(self, vkeys, pv_blob, pv_off, proof_blob, proof_off, n, status_out=None):
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_sp1_verify_batch(self._h, N.buf(vkeys), N.buf(pv_blob), pv_off.ctypes.data, N.buf(proof_blob), proof_off.ctypes.data, n, st.ctypes.data))
        return st

    def verify_batch_device(self, device, d_vkeys, d_public_values, pv_stride, d_proofs260, n, d_status, stream=None):
        N.check(N.lib().zkv_sp1_verify_batch_device(self._h, device, d_vkeys, d_public_values, pv_stride, d_proofs260, n, d_status, stream))

    def stage_ms(self, device=0):
        out = (C.c_float * 5)()
        n = N.lib().zkv_last_stage_ms(N.lib().zkv_sp1_vk(self._h), device, out, 5)
        return dict(zip(("decode_hash", "vk_x", "g2_check", "miller", "final_exp"), list(out)[:max(n, 0)]))


def _route_error(status):
    """the error a route handle raises for a status other than OK / SELECTOR_MISMATCH"""
    if status == N.ZKV_INVALID_PROOF_DATA:
        return E.InvalidProofData()
    return E.VerificationFailed()


def _handles(verifiers):
    return (C.c_void_p * max(len(verifiers), 1))(*[v._h for v in verifiers])


class RiscZeroVerifierRouter:
    """RiscZeroVerifierRouter: 1..256 initialised RiscZeroVerifier handles (zkv_risc0_router_create), each registered under its selector.
    A seal goes to the verifier whose selector is bytes4(seal[0:4]); a selector no verifier has raises SelectorUnknown.  The router keeps
    references to its verifiers, which must outlive it."""

    def __init__(self, verifiers, devices=None):
        self.verifiers = list(verifiers)
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_risc0_router_create(_handles(self.verifiers), len(self.verifiers), arr, nd, C.byref(self._h)))
        self._by_selector = {v.get_selector(): v for v in self.verifiers}

    def __len__(self):
        return len(self.verifiers)

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_risc0_router_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def get_verifier(self, selector):
        v = self._by_selector.get(bytes(selector))
        if v is None:
            raise E.SelectorUnknown(selector)
        return v

    def _result(self, status, seal):
        if status == N.ZKV_OK:
            return True
        if status == N.ZKV_SELECTOR_MISMATCH:
            raise E.SelectorUnknown(seal[:4])
        raise _route_error(status)

    def verify(self, seal, image_id, journal_digest):
        return self._result(int(self.verify_batch([seal], [image_id], [journal_digest])[0]), seal)

    def verify_integrity(self, receipt_seal, claim_digest):
        return self._result(int(self.verify_integrity_batch([receipt_seal], [claim_digest])[0]), receipt_seal)

    def verify_batch(self, seals, image_ids, journal_digests):
        n = len(seals)
        _need32_each(n, image_ids=image_ids, journal_digests=journal_digests)
        return self.verify_batch_packed(b"".join(seals) or b"\0", _offsets(seals), b"".join(image_ids) or b"\0", b"".join(journal_digests) or b"\0", n)

    def verify_integrity_batch(self, seals, claim_digests):
        n = len(seals)
        _need32_each(n, claim_digests=claim_digests)
        st = np.zeros(n, dtype=np.uint8)
        off = _offsets(seals)
        N.check(N.lib().zkv_risc0_router_verify_integrity_batch(self._h, N.buf(b"".join(seals) or b"\0"), off.ctypes.data, N.buf(b"".join(claim_digests) or b"\0"), n, st.ctypes.data))
        return st

    def verify_batch_packed(self, seal_blob, seal_off, image_ids, journal_digests, n, status_out=None):
        """Zero-copy form: contiguous buffers (bytes or numpy uint8) + numpy uint64 offsets."""
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_risc0_router_verify_batch(self._h, N.buf(seal_blob), seal_off.ctypes.data, N.buf(image_ids), N.buf(journal_digests), n, st.ctypes.data))
        return st

    def verify_batch_device(self, device, d_seals260, d_image_ids, d_journal_digests, n, d_status, stream=None):
        """Inputs already in HBM (raw device pointers as ints, n x 260-byte seals); asynchronous on `stream`."""
        N.check(N.lib().zkv_risc0_router_verify_batch_device(self._h, device, d_seals260, d_image_ids, d_journal_digests, n, d_status, stream))


class Sp1VerifierGateway:
    """SP1VerifierGateway: 1..256 Sp1Verifier handles of different verifier versions (zkv_sp1_gateway_create).  A proof goes to the verifier
    whose verifier hash starts with proof[:4]; a selector no verifier has raises RouteNotFound.  The gateway keeps references to its
    verifiers, which must outlive it."""

    def __init__(self, verifiers, devices=None):
        self.verifiers = list(verifiers)
        self._h = C.c_void_p()
        arr, nd = _dev_array(devices)
        N.check(N.lib().zkv_sp1_gateway_create(_handles(self.verifiers), len(self.verifiers), arr, nd, C.byref(self._h)))

    def __len__(self):
        return len(self.verifiers)

    def close(self):
        if getattr(self, "_h", None):
            N.lib().zkv_sp1_gateway_destroy(self._h); self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def verify_proof(self, program_vkey, public_values, proof_bytes):
        _need32(program_vkey=program_vkey)
        st = int(self.verify_batch([program_vkey], [public_values], [proof_bytes])[0])
        if st == N.ZKV_OK:
            return None
        if st == N.ZKV_SELECTOR_MISMATCH:
            raise E.RouteNotFound(proof_bytes[:4])
        raise _route_error(st)

    def verify_batch(self, program_vkeys, public_values, proofs):
        n = len(proofs)
        _need32_each(n, program_vkeys=program_vkeys)
        if len(public_values) != n:
            raise ValueError("public_values: expected %d entries, got %d" % (n, len(public_values)))
        return self.verify_batch_packed(b"".join(program_vkeys) or b"\0", b"".join(public_values) or b"\0", _offsets(public_values),
                                        b"".join(proofs) or b"\0", _offsets(proofs), n)

    def verify_batch_packed(self, vkeys, pv_blob, pv_off, proof_blob, proof_off, n, status_out=None):
        st = status_out if status_out is not None else np.zeros(n, dtype=np.uint8)
        N.check(N.lib().zkv_sp1_gateway_verify_batch(self._h, N.buf(vkeys), N.buf(pv_blob), pv_off.ctypes.data, N.buf(proof_blob), proof_off.ctypes.data, n, st.ctypes.data))
        return st

    def verify_batch_device(self, device, d_vkeys, d_public_values, pv_stride, d_proofs260, n, d_status, stream=None):
        """Inputs already in HBM (raw device pointers as ints, n x 260-byte proofs, n x pv_stride public values); asynchronous on `stream`."""
        N.check(N.lib().zkv_sp1_gateway_verify_batch_device(self._h, device, d_vkeys, d_public_values, pv_stride, d_proofs260, n, d_status, stream))


# ------------------------------------------------------------------ precompile-shaped services and hooks
def ec_add_batch(data, n, device=0):
    out = np.zeros(n * 64, dtype=np.uint8); rev = np.zeros(n, dtype=np.uint8)
    N.check(N.lib().zkv_ec_add_batch(N.buf(data), n, out.ctypes.data, rev.ctypes.data, device))
    return out, rev


def ec_mul_batch(data, n, device=0):
    out = np.zeros(n * 64, dtype=np.uint8); rev = np.zeros(n, dtype=np.uint8)
    N.check(N.lib().zkv_ec_mul_batch(N.buf(data), n, out.ctypes.data, rev.ctypes.data, device))
    return out, rev


def g2_mul_batch(points, scalars, n, broadcast=False, device=0):
    out = np.zeros(n * 128, dtype=np.uint8); rev = np.zeros(n, dtype=np.uint8)
    N.check(N.lib().zkv_g2_mul_batch(N.buf(points), 1 if broadcast else 0, N.buf(scalars), n, out.ctypes.data, rev.ctypes.data, device))
    return out, rev


def pairing4_batch(vk, g1s, g2s, n, want_gt=False, want_miller=False):
    ok = np.zeros(n, dtype=np.uint8)
    gt = np.zeros(n * 384, dtype=np.uint8) if want_gt else None
    ml = np.zeros(n * 384, dtype=np.uint8) if want_miller else None
    N.check(N.lib().zkv_pairing4_batch(vk._h, N.buf(g1s), N.buf(g2s), n, ok.ctypes.data, gt.ctypes.data if want_gt else None, ml.ctypes.data if want_miller else None))
    return ok, gt, ml


def vk_x_batch(vk, signals, k, n):
    out = np.zeros(n * 64, dtype=np.uint8)
    N.check(N.lib().zkv_vk_x_batch(vk._h, N.buf(signals), k, n, out.ctypes.data))
    return out


def ec_pairing_batch(data, k, n, want_miller=False, device=0):
    """Precompile 0x08 on n instances of k pairs (every G2 variable): returns (words n x 32 uint8, reverted n uint8[, miller n x 384])."""
    out = np.zeros(n * 32, dtype=np.uint8); rev = np.zeros(n, dtype=np.uint8)
    ml = np.zeros(n * 384, dtype=np.uint8) if want_miller else None
    N.check(N.lib().zkv_ec_pairing_batch(N.buf(data) if (k and n) else None, k, n, out.ctypes.data, rev.ctypes.data, ml.ctypes.data if want_miller else None, device))
    return (out, rev, ml) if want_miller else (out, rev)


def ec_pairing(data, device=0):
    """One precompile 0x08 call on raw bytes: the 32-byte return word, or None if the call fails (what the reference sees as a revert)."""
    out = C.create_string_buffer(32); rev = C.c_uint8(0)
    N.check(N.lib().zkv_ec_pairing(data or None, len(data), out, C.byref(rev), device))
    return None if rev.value else out.raw


def fp_mul_batch(a, b, n, device=0):
    out = np.zeros(n * 32, dtype=np.uint8)
    N.check(N.lib().zkv_fp_mul_batch(N.buf(a), N.buf(b), n, out.ctypes.data, device))
    return out


def fp12_op_batch(op, a, b, n, device=0):
    """Fp12 tower operation `op` (see zkv.h) on n operands of 384 bytes; b may be None for unary operations.  Ops 0-9 run the round-1
    tower (bn254.cuh); op 16 + k runs operation k on the shared-memory, lazily reduced tower of the verification kernels (lazy.cuh), plus
    op 25 (the normalised-line product) and op 26 (the verification Miller loop on the single pair of op 9)."""
    out = C.create_string_buffer(384 * n)
    N.check(N.lib().zkv_fp12_op_batch(op, N.buf(a), N.buf(b) if b is not None else None, n, out, device))
    return out.raw


def g2_check_batch(g2s, n, device=0):
    out = np.zeros(n, dtype=np.uint8)
    N.check(N.lib().zkv_g2_check_batch(N.buf(g2s), n, out.ctypes.data, device))
    return out


class _PinnedBlock:
    """owner of one zkv_host_alloc block (freed with the last numpy view of it)"""

    def __init__(self, nbytes):
        self.ptr = N.lib().zkv_host_alloc(nbytes)
        if not self.ptr:
            raise N.ZkvError(N.ZKV_ERR_CUDA, (N.lib().zkv_last_error() or b"").decode())

    def __del__(self):
        try:
            N.lib().zkv_host_free(self.ptr)
        except Exception:
            pass


def pinned_copy(a):
    """Copy of a bytes object / numpy array in page-locked memory (zkv_host_alloc).  Batch calls whose inputs are all page-locked upload them
    in place instead of gathering them into the library's staging buffer first (include/zkv.h)."""
    src = np.frombuffer(a, dtype=np.uint8) if isinstance(a, (bytes, bytearray)) else np.ascontiguousarray(a)
    blk = _PinnedBlock(max(src.nbytes, 1))
    buf = (C.c_uint8 * max(src.nbytes, 1)).from_address(blk.ptr)
    buf._zkv_owner = blk                                   # the ctypes array keeps the block alive, numpy keeps the ctypes array alive
    out = np.frombuffer(buf, dtype=np.uint8, count=src.nbytes).view(src.dtype).reshape(src.shape)
    out[...] = src
    return out


def device_count():
    """number of CUDA devices the library sees (0 without a driver)"""
    return int(N.lib().zkv_device_count())


def wave_proofs(device, kernel):
    """Proofs in one full wave of the verification Miller-loop kernel (kernel 0) or the final exponentiation (kernel 1) on `device`."""
    w = int(N.lib().zkv_wave_proofs(int(device), int(kernel)))
    if w <= 0:
        N.check(w if w < 0 else N.ZKV_ERR_CUDA)
    return w


def launch_count():
    """Kernels launched by the verification chains since the library was loaded."""
    return int(N.lib().zkv_launch_count())


def imad_peak(device=0):
    w, f = C.c_double(0), C.c_double(0)
    N.check(N.lib().zkv_imad_peak(device, C.byref(w), C.byref(f)))
    return w.value, f.value


class GpuBackend:
    """synth.py backend: multiples of the group generators through the library's own batched ecMul / G2 hook."""

    def __init__(self, device=0):
        self.device = device

    def g1_mul(self, scalars):
        from .synth import G1_GEN
        n = len(scalars)
        if n == 0:
            return []
        data = b"".join(G1_GEN + int(s).to_bytes(32, "big") for s in scalars)
        out, rev = ec_mul_batch(data, n, self.device)
        assert not rev.any()
        raw = out.tobytes()
        return [raw[64 * i:64 * i + 64] for i in range(n)]

    def g2_mul(self, scalars):
        from .synth import G2_GEN
        n = len(scalars)
        if n == 0:
            return []
        out, rev = g2_mul_batch(G2_GEN, b"".join(int(s).to_bytes(32, "big") for s in scalars), n, broadcast=True, device=self.device)
        assert not rev.any()
        raw = out.tobytes()
        return [raw[128 * i:128 * i + 128] for i in range(n)]
