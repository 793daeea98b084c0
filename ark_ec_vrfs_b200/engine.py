"""Batch engine: a thin, typed wrapper over the C ABI (include/vrfs_b200.h).  Array conventions are the
ABI's: scalars (n,32) uint8 little-endian, points (n,64) uint8 affine x||y little-endian."""
import ctypes as C
import os

import numpy as np

from . import _lib

BANDERSNATCH, ED25519, P256, BANDERSNATCH_SW, JUBJUB, BABYJUBJUB = 0, 1, 2, 3, 4, 5
SUITE_NAMES = {0: "Bandersnatch_SHA-512_ELL2", 1: "Ed25519_SHA-512_TAI", 2: "secp256r1 (RFC 9381 suite 0x01)",
               3: "Bandersnatch_SW_SHA-512_TAI", 4: "JubJub_SHA-512_TAI", 5: "BabyJubJub_SHA-512_TAI"}


def _u8(a, shape):
    a = np.frombuffer(a, dtype=np.uint8) if isinstance(a, (bytes, bytearray, memoryview)) else np.asarray(a, dtype=np.uint8)
    return np.ascontiguousarray(a).reshape(shape)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


ITEM_OK, ITEM_VERIFICATION_FAILURE, ITEM_INVALID_DATA = 0, 1, 2      # vrfs_item_status: Ok(()) / Error::VerificationFailure / Error::InvalidData


def pack_var(items, n=None):
    """list of bytes -> (uint8 data, uint64 offsets[n+1]); `items` may already be such a pair, or None.
    n: the batch size the C side will read offsets for - a shorter list would make it read past the arrays, so it is an error here."""
    if items is None:
        return None, None
    if isinstance(items, tuple):
        data, off = items
        off = np.ascontiguousarray(off, dtype=np.uint64)
        data = np.ascontiguousarray(data if data is not None else np.zeros(16, np.uint8), dtype=np.uint8).reshape(-1)
    else:
        off = np.zeros(len(items) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(b) for b in items], dtype=np.uint64)
        data = np.frombuffer(b"".join(items), dtype=np.uint8).copy() if off[-1] else np.zeros(16, dtype=np.uint8)
    if n is not None and len(off) - 1 != n:
        raise ValueError(f"{len(off) - 1} variable-length items for a batch of {n}")
    if len(off) and int(off[-1]) > data.size:
        raise ValueError("offsets run past the data buffer")
    return data, off


class PreparedBases:
    def __init__(self, engine, handle, n):
        self.engine, self.handle, self.n = engine, handle, n

    def msm(self, scalars, n_columns=1):
        scalars = _u8(scalars, (n_columns * self.n, 32)); out = np.zeros((n_columns, 96), np.uint8)
        self.engine._call("vrfs_msm_g1_prepared", self.handle, _p(scalars), int(n_columns), _p(out))
        return out

    def msm_partial(self, scalars, n_columns=1):
        """projective partial sums (n_columns, 144) over this handle's bases - one rank's share of a multi-GPU MSM"""
        scalars = _u8(scalars, (n_columns * self.n, 32)); out = np.zeros((n_columns, 144), np.uint8)
        self.engine._call("vrfs_msm_g1_prepared_partial", self.handle, _p(scalars), int(n_columns), _p(out))
        return out

    def kzg_open(self, coeffs, zs):
        """KZG openings over this handle as a monomial SRS [tau^j] G1: coeffs (k, len, 32) low to high, zs (k, 32) ->
        (values (k, 32) = p_i(z_i), proofs (k, 96) = [(p_i - v_i) / (X - z_i)](tau) G1) (vrfs_kzg_open_batch)"""
        coeffs = np.asarray(coeffs, np.uint8)
        if coeffs.ndim != 3 or coeffs.shape[2] != 32:
            raise ValueError(f"coeffs must have shape (k, len, 32), not {coeffs.shape}")
        k, n_coeffs = coeffs.shape[0], coeffs.shape[1]
        coeffs = _u8(coeffs, (k, n_coeffs, 32)); zs = _u8(zs, (k, 32))
        values = np.zeros((k, 32), np.uint8); proofs = np.zeros((k, 96), np.uint8)
        self.engine._call("vrfs_kzg_open_batch", self.handle, C.c_size_t(k), C.c_size_t(n_coeffs), _p(coeffs), _p(zs), _p(values), _p(proofs))
        return values, proofs

    def kzg_open_aggregated(self, polys, group_sizes, zs, nus):
        """Aggregated KZG openings over this handle as a monomial SRS: polys a list of (len_i, 32) coefficient arrays, low to high,
        in group order; group g is the next group_sizes[g] of them, opened at zs[g]; nus (n_polys, 32) one coefficient per
        polynomial -> (values (n_polys, 32) = p_i(z_g), agg_values (n_groups, 32) = P_g(z_g), proofs (n_groups, 96) =
        [(P_g - P_g(z_g)) / (X - z_g)](tau) G1) with P_g = sum_{i in g} nu_i p_i (vrfs_kzg_open_aggregated_batch)"""
        polys = [_u8(p, (-1, 32)) for p in polys]
        sizes = np.asarray(group_sizes, np.int64).reshape(-1)
        if (sizes < 0).any() or int(sizes.sum()) != len(polys):
            raise ValueError(f"group sizes {sizes.tolist()} do not partition {len(polys)} polynomials")
        n_groups, n_polys = len(sizes), len(polys)
        group_off = np.zeros(n_groups + 1, np.uint64); group_off[1:] = np.cumsum(sizes)
        coeff_off = np.zeros(n_polys + 1, np.uint64); coeff_off[1:] = np.cumsum([p.shape[0] for p in polys])
        coeffs = np.ascontiguousarray(np.concatenate(polys) if int(coeff_off[-1]) else np.zeros((1, 32), np.uint8))
        zs = _u8(zs, (n_groups, 32)); nus = _u8(nus, (n_polys, 32))
        values = np.zeros((n_polys, 32), np.uint8); agg = np.zeros((n_groups, 32), np.uint8); proofs = np.zeros((n_groups, 96), np.uint8)
        self.engine._call("vrfs_kzg_open_aggregated_batch", self.handle, C.c_size_t(n_groups), C.c_size_t(n_polys), _p(group_off), _p(coeff_off),
                          _p(coeffs), _p(zs), _p(nus), _p(values), _p(agg), _p(proofs))
        return values, agg, proofs

    def ring_commit(self, keys, keyset_part_size, padding, tail, lagrange=True):
        """(cx, cy, selector) commitments (3, 96) of the ring's fixed columns over this SRS (vrfs_ring_commit)"""
        keys = _u8(keys, (-1, 64)); tail = _u8(tail, (-1, 64)); padding = _u8(padding, (64,)); out = np.zeros((3, 96), np.uint8)
        self.engine._call("vrfs_ring_commit", self.handle, int(bool(lagrange)), C.c_size_t(keyset_part_size), C.c_size_t(len(keys)), _p(keys),
                          _p(padding), C.c_size_t(len(tail)), _p(tail), _p(out))
        return out

    def ring_commit_rows_partial(self, row_lo, keyset_part_size, n_keys, keys_rows, padding, tail):
        """this handle = the prepared Lagrange bases of rows [row_lo, row_lo + n): projective partial commitments (3, 144) of those rows"""
        keys_rows = _u8(keys_rows, (-1, 64)); tail = _u8(tail, (-1, 64)); padding = _u8(padding, (64,)); out = np.zeros((3, 144), np.uint8)
        self.engine._call("vrfs_ring_commit_rows_partial", self.handle, C.c_size_t(row_lo), C.c_size_t(keyset_part_size), C.c_size_t(n_keys), _p(keys_rows),
                          _p(padding), C.c_size_t(len(tail)), _p(tail), _p(out))
        return out

    def msm_allgather(self, scalars, n_columns=1):
        """COLLECTIVE over the engine's peer group: this rank's scalars over its slice of the SRS -> the full commitments
        (n_columns, 96) on every rank; the partials travel GPU to GPU inside the MSM's last kernel (vrfs_msm_g1_prepared_allgather)"""
        scalars = _u8(scalars, (n_columns * self.n, 32)); out = np.zeros((n_columns, 96), np.uint8)
        self.engine._call("vrfs_msm_g1_prepared_allgather", self.handle, _p(scalars), int(n_columns), _p(out))
        return out

    def ring_commit_rows_allgather(self, row_lo, keyset_part_size, n_keys, keys_rows, padding, tail):
        """COLLECTIVE: the ring commitment (3, 96) with the domain's rows split over the ranks (vrfs_ring_commit_rows_allgather)"""
        keys_rows = _u8(keys_rows, (-1, 64)); tail = _u8(tail, (-1, 64)); padding = _u8(padding, (64,)); out = np.zeros((3, 96), np.uint8)
        self.engine._call("vrfs_ring_commit_rows_allgather", self.handle, C.c_size_t(row_lo), C.c_size_t(keyset_part_size), C.c_size_t(n_keys), _p(keys_rows),
                          _p(padding), C.c_size_t(len(tail)), _p(tail), _p(out))
        return out

    def ring_commit_delta(self, keys, padding):
        """[sum (x_i - pad_x) L_i, sum (y_i - pad_y) L_i] over a Lagrange-basis SRS: (2, 96) (vrfs_ring_commit_delta)"""
        keys = _u8(keys, (-1, 64)); padding = _u8(padding, (64,)); out = np.zeros((2, 96), np.uint8)
        self.engine._call("vrfs_ring_commit_delta", self.handle, C.c_size_t(len(keys)), _p(keys), _p(padding), _p(out))
        return out

    def release(self):
        if self.handle:
            self.engine._lib.vrfs_msm_g1_release(self.handle)
            self.handle = None
            if self in self.engine._prepared:
                self.engine._prepared.remove(self)


def _dev_ptr(x):
    """a device pointer: an int, or a torch CUDA tensor (its data_ptr())"""
    if x is None:
        return None
    return C.c_void_p(x.data_ptr() if hasattr(x, "data_ptr") else int(x) or None)


class PreparedPublics:
    """Public keys prepared once for many verifies (vrfs_public_keys_prepare): one fixed-base table per key on the engine's GPU.
    key_ok[k] = 1 where keys[k] is a key ietf_verify accepts.  Usable as a context manager; release() frees the tables.
    from_encodings: made by Engine.public_keys_prepare_encoded, which verify_wire requires."""

    def __init__(self, engine, handle, suite, key_ok, from_encodings=False):
        self.engine, self.handle, self.suite, self.key_ok, self.from_encodings = engine, handle, suite, key_ok, from_encodings

    @property
    def n_keys(self):
        return len(self.key_ok)

    def verify(self, key_index, inp, outp, c, s, ad=None, status=False):
        """ietf_verify with pk[i] = keys[key_index[i]] (an index >= n_keys: ITEM_INVALID_DATA) -> ok flags [, status]"""
        key_index = np.ascontiguousarray(key_index, dtype=np.uint32).reshape(-1); n = len(key_index)
        inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64)); c = _u8(c, (n, 32)); s = _u8(s, (n, 32))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self.engine._call("vrfs_ietf_verify_prepared_batch", self.handle, C.c_size_t(n), _p(key_index), _p(inp), _p(outp), _p(c), _p(s),
                          _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    def verify_dev(self, n, d_key_index, d_inp, d_outp, d_c, d_s, d_ok, d_ad=None, d_off=None, d_status=None):
        """device buffers (ints or torch CUDA tensors; key_index uint32, 16-byte aligned); enqueued on the context stream
        (Engine.stream) - the caller orders its producers before and its readers after it (e.g. Engine.sync())"""
        self.engine._call("vrfs_ietf_verify_prepared_batch_dev", self.handle, C.c_size_t(n), _dev_ptr(d_key_index), _dev_ptr(d_inp), _dev_ptr(d_outp),
                          _dev_ptr(d_c), _dev_ptr(d_s), _dev_ptr(d_ad), _dev_ptr(d_off), _dev_ptr(d_ok), _dev_ptr(d_status))

    def verify_wire(self, key_index, datas, sig, ad=None, want_hash=True, status=False, out_ok=None, out_hash=None):
        """Engine.ietf_verify_wire with pk_enc[i] = the encoding of key key_index[i] (vrfs_ietf_verify_prepared_wire_batch; keys from
        Engine.public_keys_prepare_encoded) -> (ok, beta[, status]) like that call; a key with key_ok = 0 or an index >= n_keys:
        ITEM_INVALID_DATA"""
        e = self.engine
        key_index = np.ascontiguousarray(key_index, dtype=np.uint32).reshape(-1); n = len(key_index)
        sig = _u8(sig, (n, e.ietf_signature_len(self.suite))); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        hl = e.hash_len(self.suite)
        ok = _u8(out_ok, (n,)) if out_ok is not None else np.zeros(n, np.uint8)
        h = (_u8(out_hash, (n, hl)) if out_hash is not None else np.zeros((n, hl), np.uint8)) if want_hash else None
        st = np.zeros(n, np.uint8) if status else None
        e._call("vrfs_ietf_verify_prepared_wire_batch", self.handle, C.c_size_t(n), _p(key_index), _p(data), _p(doff), _p(sig), _p(adb), _p(off),
                _p(ok), _p(h), _p(st))
        res = (ok, h) if want_hash else (ok,)
        res = res + (st,) if status else res
        return res if len(res) > 1 else res[0]

    def verify_io(self, inputs, key_index, input_index, outp, c, s, ad=None, status=False):
        """verify with inp[i] = inputs.points[input_index[i]] (vrfs_ietf_verify_prepared_io_batch; `inputs` from
        Engine.inputs_prepare) -> ok flags [, status]; an input index >= n_inputs or an input with input_ok = 0: ITEM_INVALID_DATA"""
        key_index = np.ascontiguousarray(key_index, dtype=np.uint32).reshape(-1); n = len(key_index)
        input_index = np.ascontiguousarray(input_index, dtype=np.uint32).reshape(n)
        outp = _u8(outp, (n, 64)); c = _u8(c, (n, 32)); s = _u8(s, (n, 32))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self.engine._call("vrfs_ietf_verify_prepared_io_batch", self.handle, inputs.handle, C.c_size_t(n), _p(key_index), _p(input_index), _p(outp),
                          _p(c), _p(s), _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    def verify_io_dev(self, inputs, n, d_key_index, d_input_index, d_outp, d_c, d_s, d_ok, d_ad=None, d_off=None, d_status=None):
        """verify_io on device buffers (ints or torch CUDA tensors; indices uint32, 16-byte aligned); enqueued on the context stream"""
        self.engine._call("vrfs_ietf_verify_prepared_io_batch_dev", self.handle, inputs.handle, C.c_size_t(n), _dev_ptr(d_key_index),
                          _dev_ptr(d_input_index), _dev_ptr(d_outp), _dev_ptr(d_c), _dev_ptr(d_s), _dev_ptr(d_ad), _dev_ptr(d_off), _dev_ptr(d_ok),
                          _dev_ptr(d_status))

    def verify_io_wire(self, inputs, key_index, input_index, sig, ad=None, want_hash=True, status=False):
        """verify_wire with datas[i] = the data of input input_index[i] (vrfs_ietf_verify_prepared_io_wire_batch; keys from
        Engine.public_keys_prepare_encoded) -> (ok, beta[, status]); an input index >= n_inputs or an input with input_ok = 0:
        ITEM_INVALID_DATA with a zero hash"""
        e = self.engine
        key_index = np.ascontiguousarray(key_index, dtype=np.uint32).reshape(-1); n = len(key_index)
        input_index = np.ascontiguousarray(input_index, dtype=np.uint32).reshape(n)
        sig = _u8(sig, (n, e.ietf_signature_len(self.suite))); adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8)
        h = np.zeros((n, e.hash_len(self.suite)), np.uint8) if want_hash else None
        st = np.zeros(n, np.uint8) if status else None
        e._call("vrfs_ietf_verify_prepared_io_wire_batch", self.handle, inputs.handle, C.c_size_t(n), _p(key_index), _p(input_index), _p(sig),
                _p(adb), _p(off), _p(ok), _p(h), _p(st))
        res = (ok, h) if want_hash else (ok,)
        res = res + (st,) if status else res
        return res if len(res) > 1 else res[0]

    def release(self):
        if self.handle:
            self.engine._lib.vrfs_public_keys_release(self.handle)
            self.handle = None
            if self in self.engine._prepared:
                self.engine._prepared.remove(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.release()


class PreparedInputs:
    """VRF inputs prepared once for many verifies (vrfs_inputs_prepare): Input::new of each data item, and one fixed-base table per
    input point on the engine's GPU.  input_ok[j] / points[j] are what Engine.data_to_point gives for datas[j].  Usable as a
    context manager; release() frees the tables."""

    def __init__(self, engine, handle, suite, input_ok, points):
        self.engine, self.handle, self.suite, self.input_ok, self.points = engine, handle, suite, input_ok, points

    @property
    def n_inputs(self):
        return len(self.input_ok)

    def release(self):
        if self.handle:
            self.engine._lib.vrfs_inputs_release(self.handle)
            self.handle = None
            if self in self.engine._prepared:
                self.engine._prepared.remove(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.release()


def host_buffer(shape):
    """A zeroed uint8 array in page-locked host memory (vrfs_host_alloc): batch calls on such buffers copy beside their kernels.
    The allocation is freed when the array (and every view of it) is gone."""
    import weakref
    lib = _lib.load()
    shape = (int(shape),) if np.isscalar(shape) else tuple(int(x) for x in shape)
    nbytes = int(np.prod(shape)) if shape else 1
    p = C.c_void_p()
    st = lib.vrfs_host_alloc(C.c_size_t(max(nbytes, 1)), C.byref(p))
    if st != _lib.OK or not p.value:
        raise _lib.VrfsError(st, "page-locked host allocation of %d bytes failed" % nbytes)
    raw = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    weakref.finalize(raw, lib.vrfs_host_free, C.c_void_p(p.value))
    a = np.frombuffer(raw, dtype=np.uint8, count=nbytes).reshape(shape)
    a[...] = 0
    return a


def host_copy(a):
    """the same bytes in page-locked host memory"""
    a = np.ascontiguousarray(a)
    out = host_buffer(a.nbytes)
    out[:] = a.view(np.uint8).reshape(-1)
    return out.reshape(a.shape) if a.dtype == np.uint8 else out.view(a.dtype).reshape(a.shape)


class Engine:
    """One context on one GPU (`device` = CUDA ordinal).  Not thread-safe; one per process per GPU."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        self._prepared = []
        self._ctx = C.c_void_p()
        st = self._lib.vrfs_ctx_create(int(device), C.byref(self._ctx))
        if st != _lib.OK:
            msg = self._lib.vrfs_last_error(self._ctx).decode() if self._ctx else "context allocation failed"
            if self._ctx:
                self._lib.vrfs_ctx_destroy(self._ctx)
                self._ctx = None
            raise _lib.VrfsError(st, msg)
        self.device = device

    def close(self):
        if getattr(self, "_ctx", None):
            for p in list(self._prepared):          # outstanding prepared bases go with their context
                p.release()
            self._lib.vrfs_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, st):
        if st != _lib.OK:
            raise _lib.VrfsError(st, self._lib.vrfs_last_error(self._ctx).decode())

    def sync(self):
        self._check(self._lib.vrfs_ctx_sync(self._ctx))

    @property
    def launch_count(self):
        return int(self._lib.vrfs_ctx_launch_count(self._ctx))

    @property
    def stream(self):
        return self._lib.vrfs_ctx_stream(self._ctx)

    # ---- peer group (one process per GPU): device-side exchange of MSM partials over NVLink
    def peer_export(self, rank, world):
        """allocate this rank's mailbox; returns its 64-byte CUDA IPC handle (to be all-gathered by the caller)"""
        h = np.zeros(64, np.uint8)
        self._call("vrfs_ctx_peer_export", int(rank), int(world), _p(h))
        return h

    def peer_connect(self, handles):
        handles = _u8(handles, (-1, 64))
        self._call("vrfs_ctx_peer_connect", _p(handles))

    def peer_set_timeout_ms(self, ms):
        self._call("vrfs_ctx_peer_set_timeout_ms", C.c_uint(int(ms)))

    @property
    def peer_world(self):
        return int(self._lib.vrfs_ctx_peer_world(self._ctx))

    # ---- ietf
    def ietf_verify(self, suite, pk, inp, outp, c, s, ad=None, status=False):
        """ietf::Verifier::verify -> ok flags; status=True: (ok, vrfs_item_status per item)"""
        pk = _u8(pk, (-1, 64)); n = len(pk)
        inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64)); c = _u8(c, (n, 32)); s = _u8(s, (n, 32))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self._check(self._lib.vrfs_ietf_verify_batch(self._ctx, suite, C.c_size_t(n), _p(pk), _p(inp), _p(outp), _p(c), _p(s), _p(adb), _p(off), _p(ok), _p(st)))
        return (ok, st) if status else ok

    def ietf_verify_dev(self, suite, n, d_pk, d_inp, d_outp, d_c, d_s, d_ok, d_ad=None, d_off=None, d_status=None):
        """device pointers (ints); enqueues on the context stream, returns immediately"""
        v = lambda x: C.c_void_p(x) if x else None
        self._check(self._lib.vrfs_ietf_verify_batch_dev(self._ctx, suite, C.c_size_t(n), v(d_pk), v(d_inp), v(d_outp), v(d_c), v(d_s), v(d_ad), v(d_off), v(d_ok), v(d_status)))

    def public_keys_prepare(self, suite, pks):
        """(n_keys, 64) affine keys of one suite -> PreparedPublics: per-key fixed-base tables (~400 KB per key) on this GPU, so that
        proofs of known signers are verified by key index (vrfs_public_keys_prepare)"""
        pks = _u8(pks, (-1, 64)); key_ok = np.zeros(len(pks), np.uint8)
        h = C.c_void_p()
        self._call("vrfs_public_keys_prepare", suite, C.c_size_t(len(pks)), _p(pks), _p(key_ok), C.byref(h))
        p = PreparedPublics(self, h, suite, key_ok)
        self._prepared.append(p)
        return p

    def public_keys_prepare_encoded(self, suite, pk_enc):
        """(n_keys, point_enc_len) encoded keys -> PreparedPublics (from_encodings=True): each key decoded with the subgroup check
        once, then prepared like public_keys_prepare; key_ok = 0 where the encoding or the decoded key is rejected
        (vrfs_public_keys_prepare_encoded).  Its verify_wire verifies serialised signatures by key index."""
        pk_enc = _u8(pk_enc, (-1, self.point_enc_len(suite))); key_ok = np.zeros(len(pk_enc), np.uint8)
        h = C.c_void_p()
        self._call("vrfs_public_keys_prepare_encoded", suite, C.c_size_t(len(pk_enc)), _p(pk_enc), _p(key_ok), C.byref(h))
        p = PreparedPublics(self, h, suite, key_ok, from_encodings=True)
        self._prepared.append(p)
        return p

    def inputs_prepare(self, suite, datas):
        """VRF input data of one suite -> PreparedInputs: hashed to the curve once, one fixed-base table per input point (~400 KB)
        on this GPU, so that proofs over a few distinct inputs are verified by input index (vrfs_inputs_prepare)"""
        data, off = pack_var(datas); n = len(off) - 1
        input_ok = np.zeros(n, np.uint8); pts = np.zeros((n, 64), np.uint8)
        h = C.c_void_p()
        self._call("vrfs_inputs_prepare", suite, C.c_size_t(n), _p(data), _p(off), _p(input_ok), _p(pts), C.byref(h))
        p = PreparedInputs(self, h, suite, input_ok, pts)
        self._prepared.append(p)
        return p

    def ietf_verify_host_ptrs(self, suite, n, pk, inp, outp, c, s, ok, ad=None, off=None, status=None):
        """raw host pointers (ints), e.g. of pinned torch tensors; synchronous"""
        v = lambda x: C.c_void_p(x) if x else None
        self._check(self._lib.vrfs_ietf_verify_batch(self._ctx, suite, C.c_size_t(n), v(pk), v(inp), v(outp), v(c), v(s), v(ad), v(off), v(ok), v(status)))

    def debug_read_staging(self, slot, nbytes, offset=0):
        """test hook (vrfs_ctx_debug_read_staging): bytes of an internal staging buffer after a call returned"""
        out = np.zeros(nbytes, np.uint8)
        self._call("vrfs_ctx_debug_read_staging", int(slot), C.c_size_t(offset), _p(out), C.c_size_t(nbytes))
        return out

    # ---- keys, inputs, outputs (Secret / Public / Input / Output of the reference API)
    def _call(self, fn, *args):
        self._check(getattr(self._lib, fn)(self._ctx, *args))

    def hash_len(self, suite):
        return self._lib.vrfs_suite_hash_len(suite)

    def point_enc_len(self, suite):
        return self._lib.vrfs_suite_point_enc_len(suite)

    def challenge_len(self, suite):
        return self._lib.vrfs_suite_challenge_len(suite)

    def secret_from_seed(self, suite, seeds, want_pk=True):
        data, off = pack_var(seeds); n = len(off) - 1
        if data is None:
            raise ValueError("seeds are required")
        sk = np.zeros((n, 32), np.uint8); pk = np.zeros((n, 64), np.uint8) if want_pk else None
        self._call("vrfs_secret_from_seed_batch", suite, C.c_size_t(n), _p(data), _p(off), _p(sk), _p(pk))
        return (sk, pk) if want_pk else sk

    def data_to_point(self, suite, datas):
        data, off = pack_var(datas); n = len(off) - 1
        pts = np.zeros((n, 64), np.uint8); ok = np.zeros(n, np.uint8)
        self._call("vrfs_data_to_point_batch", suite, C.c_size_t(n), _p(data), _p(off), _p(pts), _p(ok))
        return pts, ok

    def output(self, suite, sk, inp):
        sk = _u8(sk, (-1, 32)); n = len(sk); inp = _u8(inp, (n, 64)); out = np.zeros((n, 64), np.uint8)
        self._call("vrfs_output_batch", suite, C.c_size_t(n), _p(sk), _p(inp), _p(out))
        return out

    def point_to_hash(self, suite, pts):
        pts = _u8(pts, (-1, 64)); n = len(pts); out = np.zeros((n, self.hash_len(suite)), np.uint8)
        self._call("vrfs_point_to_hash_batch", suite, C.c_size_t(n), _p(pts), _p(out))
        return out

    def point_encode(self, suite, pts):
        pts = _u8(pts, (-1, 64)); n = len(pts); out = np.zeros((n, self.point_enc_len(suite)), np.uint8)
        self._call("vrfs_point_encode_batch", suite, C.c_size_t(n), _p(pts), _p(out))
        return out

    def point_decode(self, suite, enc):
        enc = _u8(enc, (-1, self.point_enc_len(suite))); n = len(enc)
        pts = np.zeros((n, 64), np.uint8); ok = np.zeros(n, np.uint8)
        self._call("vrfs_point_decode_batch", suite, C.c_size_t(n), _p(enc), _p(pts), _p(ok))
        return pts, ok

    def nonce(self, suite, sk, inp):
        sk = _u8(sk, (-1, 32)); n = len(sk); inp = _u8(inp, (n, 64)); out = np.zeros((n, 32), np.uint8)
        self._call("vrfs_nonce_batch", suite, C.c_size_t(n), _p(sk), _p(inp), _p(out))
        return out

    def ietf_prove(self, suite, sk, inp, outp, ad=None, out=None):
        """ietf::Prover::prove -> (c, s); out = (c, s) arrays to fill (e.g. views of pinned memory) instead of fresh ones"""
        sk = _u8(sk, (-1, 32)); n = len(sk); inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64))
        adb, off = pack_var(ad, n)
        c, s = out if out is not None else (np.zeros((n, 32), np.uint8), np.zeros((n, 32), np.uint8))
        assert c.shape == (n, 32) and s.shape == (n, 32) and c.dtype == np.uint8 and s.dtype == np.uint8 and c.flags.c_contiguous and s.flags.c_contiguous
        self._call("vrfs_ietf_prove_batch", suite, C.c_size_t(n), _p(sk), _p(inp), _p(outp), _p(adb), _p(off), _p(c), _p(s))
        return c, s

    # ---- wire formats (CanonicalSerialize / CanonicalDeserialize of Public, Output, ietf::Proof)
    def ietf_signature_len(self, suite):
        return int(self._lib.vrfs_suite_ietf_signature_len(suite))

    def point_decode_checked(self, suite, enc):
        """`Public` / `Output` deserialisation: codec decode + on-curve + prime-order-subgroup check."""
        enc = _u8(enc, (-1, self.point_enc_len(suite))); n = len(enc)
        pts = np.zeros((n, 64), np.uint8); ok = np.zeros(n, np.uint8)
        self._call("vrfs_point_decode_checked_batch", suite, C.c_size_t(n), _p(enc), _p(pts), _p(ok))
        return pts, ok

    def subgroup_check(self, suite, pts):
        pts = _u8(pts, (-1, 64)); n = len(pts); ok = np.zeros(n, np.uint8)
        self._call("vrfs_subgroup_check_batch", suite, C.c_size_t(n), _p(pts), _p(ok))
        return ok

    def ietf_sign_wire(self, suite, sk, datas, ad=None):
        """signature_i = point_encode(Output) || c || s for Input::new(datas[i]); returns (sig (n, sig_len), ok)."""
        sk = _u8(sk, (-1, 32)); n = len(sk); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        sig = np.zeros((n, self.ietf_signature_len(suite)), np.uint8); ok = np.zeros(n, np.uint8)
        self._call("vrfs_ietf_sign_wire_batch", suite, C.c_size_t(n), _p(sk), _p(data), _p(doff), _p(adb), _p(off), _p(sig), _p(ok))
        return sig, ok

    def ietf_verify_wire(self, suite, pk_enc, datas, sig, ad=None, want_hash=True, status=False, out_ok=None, out_hash=None):
        """serialised public keys + VRF input data + signatures -> (ok, beta) with beta = Output::hash of accepted items
        (status=True appends the per-item vrfs_item_status).  out_ok / out_hash: caller-owned result arrays (page-locked ones
        make the device -> host copies asynchronous and full speed)."""
        pk_enc = _u8(pk_enc, (-1, self.point_enc_len(suite))); n = len(pk_enc)
        sig = _u8(sig, (n, self.ietf_signature_len(suite))); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        ok = _u8(out_ok, (n,)) if out_ok is not None else np.zeros(n, np.uint8)
        h = (_u8(out_hash, (n, self.hash_len(suite))) if out_hash is not None else np.zeros((n, self.hash_len(suite)), np.uint8)) if want_hash else None
        st = np.zeros(n, np.uint8) if status else None
        self._call("vrfs_ietf_verify_wire_batch", suite, C.c_size_t(n), _p(pk_enc), _p(data), _p(doff), _p(sig), _p(adb), _p(off), _p(ok), _p(h), _p(st))
        res = (ok, h) if want_hash else (ok,)
        res = res + (st,) if status else res
        return res if len(res) > 1 else res[0]

    def pedersen_signature_len(self, suite):
        return int(self._lib.vrfs_suite_pedersen_signature_len(suite))

    def pedersen_sign_wire(self, suite, sk, datas, ad=None):
        """Output || pedersen::Proof serialised (4 encoded points + 2 scalars); returns (sig, blinding, ok)"""
        sk = _u8(sk, (-1, 32)); n = len(sk); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        sig = np.zeros((n, self.pedersen_signature_len(suite)), np.uint8); bl = np.zeros((n, 32), np.uint8); ok = np.zeros(n, np.uint8)
        self._call("vrfs_pedersen_sign_wire_batch", suite, C.c_size_t(n), _p(sk), _p(data), _p(doff), _p(adb), _p(off), _p(sig), _p(bl), _p(ok))
        return sig, bl, ok

    def pedersen_verify_wire(self, suite, datas, sig, ad=None, status=False):
        sig = _u8(sig, (-1, self.pedersen_signature_len(suite))); n = len(sig); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self._call("vrfs_pedersen_verify_wire_batch", suite, C.c_size_t(n), _p(data), _p(doff), _p(sig), _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    # ---- pedersen
    def pedersen_prove(self, suite, sk, inp, outp, ad=None, out=None):
        sk = _u8(sk, (-1, 32)); n = len(sk); inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64))
        adb, off = pack_var(ad, n)
        proof, bl = out if out is not None else (np.zeros((n, 256), np.uint8), np.zeros((n, 32), np.uint8))
        assert proof.shape == (n, 256) and bl.shape == (n, 32) and proof.dtype == np.uint8 and bl.dtype == np.uint8 and proof.flags.c_contiguous and bl.flags.c_contiguous
        self._call("vrfs_pedersen_prove_batch", suite, C.c_size_t(n), _p(sk), _p(inp), _p(outp), _p(adb), _p(off), _p(proof), _p(bl))
        return proof, bl

    def pedersen_verify(self, suite, inp, outp, proof, ad=None, status=False):
        inp = _u8(inp, (-1, 64)); n = len(inp); outp = _u8(outp, (n, 64)); proof = _u8(proof, (n, 256))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self._call("vrfs_pedersen_verify_batch", suite, C.c_size_t(n), _p(inp), _p(outp), _p(proof), _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    def _batch_verify(self, fn, n, args, seed, per_item, status):
        seed = _u8(os.urandom(32) if seed is None else seed, (32,))
        all_ok = np.zeros(1, np.uint8)
        ok = np.zeros(n, np.uint8) if per_item else None
        st = np.zeros(n, np.uint8) if status else None
        self._call(fn, *args, _p(seed), _p(all_ok), _p(ok), _p(st))
        res = (bool(all_ok[0]),) + ((ok,) if per_item else ()) + ((st,) if status else ())
        return res if len(res) > 1 else res[0]

    def pedersen_batch_verify(self, suite, inp, outp, proof, ad=None, seed=None, per_item=False, status=False):
        """Bandersnatch Pedersen proofs checked together by one random linear combination (vrfs_pedersen_batch_verify) -> all_ok.
        seed: 32 secret bytes (default: os.urandom(32)).  per_item / status=True append the per-item ok flags / vrfs_item_status,
        which are computed by the per-item verifier only when the batch is rejected."""
        inp = _u8(inp, (-1, 64)); n = len(inp); outp = _u8(outp, (n, 64)); proof = _u8(proof, (n, 256))
        adb, off = pack_var(ad, n)
        return self._batch_verify("vrfs_pedersen_batch_verify", n, (suite, C.c_size_t(n), _p(inp), _p(outp), _p(proof), _p(adb), _p(off)), seed, per_item, status)

    def pedersen_batch_verify_wire(self, suite, datas, sig, ad=None, seed=None, per_item=False, status=False):
        """pedersen_batch_verify from serialised signatures (the layout of pedersen_verify_wire)"""
        sig = _u8(sig, (-1, self.pedersen_signature_len(suite))); n = len(sig); data, doff = pack_var(datas, n); adb, off = pack_var(ad, n)
        return self._batch_verify("vrfs_pedersen_batch_verify_wire", n, (suite, C.c_size_t(n), _p(data), _p(doff), _p(sig), _p(adb), _p(off)), seed, per_item, status)

    def pedersen_proof_len(self, suite):
        return int(self._lib.vrfs_suite_pedersen_proof_len(suite))

    def pedersen_prove_compressed(self, suite, sk, inp, outp, ad=None):
        """pedersen::Prover::prove with the proof in its serialised form (3 encoded points + s + sb; 160 B for Bandersnatch)"""
        sk = _u8(sk, (-1, 32)); n = len(sk); inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64))
        adb, off = pack_var(ad, n)
        proof = np.zeros((n, self.pedersen_proof_len(suite)), np.uint8); bl = np.zeros((n, 32), np.uint8)
        self._call("vrfs_pedersen_prove_compressed_batch", suite, C.c_size_t(n), _p(sk), _p(inp), _p(outp), _p(adb), _p(off), _p(proof), _p(bl))
        return proof, bl

    def pedersen_verify_compressed(self, suite, inp, outp, proof, ad=None, status=False):
        inp = _u8(inp, (-1, 64)); n = len(inp); outp = _u8(outp, (n, 64)); proof = _u8(proof, (n, self.pedersen_proof_len(suite)))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self._call("vrfs_pedersen_verify_compressed_batch", suite, C.c_size_t(n), _p(inp), _p(outp), _p(proof), _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    # ---- ring commitment MSM (BLS12-381 G1)
    def msm_g1(self, bases, scalars, n_columns=1, window_bits=0):
        bases = _u8(bases, (-1, 96)); n = len(bases); scalars = _u8(scalars, (n_columns * n, 32))
        out = np.zeros((n_columns, 96), np.uint8)
        if window_bits: self._call("vrfs_msm_g1_bls12_381_ex", C.c_size_t(n), _p(bases), _p(scalars), int(n_columns), int(window_bits), _p(out))
        else: self._call("vrfs_msm_g1_bls12_381", C.c_size_t(n), _p(bases), _p(scalars), int(n_columns), _p(out))
        return out

    def msm_g1_prepare(self, bases, window_bits=0, threads_per_bucket=0):
        """RingContext analogue: returns a handle holding 2^(c w) * P_i on the device (window_bits / threads_per_bucket 0 = the
        plan's own choice; anything else is a tuning hint, vrfs_msm_g1_prepare_ex)"""
        bases = _u8(bases, (-1, 96)); n = len(bases)
        h = C.c_void_p()
        self._call("vrfs_msm_g1_prepare_ex", C.c_size_t(n), _p(bases), int(window_bits), int(threads_per_bucket), C.byref(h))
        p = PreparedBases(self, h, n)
        self._prepared.append(p)
        return p

    def msm_g1_partial(self, bases, scalars, n_columns=1):
        bases = _u8(bases, (-1, 96)); n = len(bases); scalars = _u8(scalars, (n_columns * n, 32))
        out = np.zeros((n_columns, 144), np.uint8)
        self._call("vrfs_msm_g1_partial", C.c_size_t(n), _p(bases), _p(scalars), int(n_columns), _p(out))
        return out

    def g1_sum_partials(self, partials, n_columns=1):
        partials = _u8(partials, (-1, n_columns, 144)); out = np.zeros((n_columns, 96), np.uint8)
        self._call("vrfs_g1_sum_partials", int(len(partials)), int(n_columns), _p(partials), _p(out))
        return out

    # ---- ring fixed columns (SURVEY 8f-2)
    def ring_fixed_columns(self, domain_size, keyset_part_size, keys, padding, tail):
        """xs | ys | selector of the ring's fixed columns: (3, domain_size, 32) canonical LE values of BLS12-381 Fr"""
        keys = _u8(keys, (-1, 64)); tail = _u8(tail, (-1, 64)); padding = _u8(padding, (64,))
        out = np.zeros((3, domain_size, 32), np.uint8)
        self._call("vrfs_ring_fixed_columns", C.c_size_t(domain_size), C.c_size_t(keyset_part_size), C.c_size_t(len(keys)), _p(keys), _p(padding),
                   C.c_size_t(len(tail)), _p(tail), _p(out))
        return out

    def fr_fft(self, values, n_columns=1, inverse=False):
        """Radix2EvaluationDomain::fft / ifft over BLS12-381 Fr on n_columns vectors of 2^k canonical LE values"""
        values = _u8(values, (-1, 32)); n = len(values) // n_columns
        assert n * n_columns == len(values) and n and not (n & (n - 1)), "column length must be a power of two"
        out = np.zeros_like(values)
        self._call("vrfs_fr_fft_batch", int(n.bit_length() - 1), int(n_columns), int(bool(inverse)), _p(values), _p(out))
        return out

    def g1_fft(self, points, inverse=False):
        """the same transform over BLS12-381 G1 (vrfs_g1_fft_batch): (n, 96) affine LE points in G1, n a power of two, -> (n, 96)
        out_i = sum_j [w^ij] P_j, or [1/n] sum_j [w^-ij] P_j for the inverse; the inverse of [tau^j] G1 is the Lagrange basis [L_i(tau)] G1"""
        points = _u8(points, (-1, 96)); n = len(points)
        if n == 0 or n & (n - 1):
            raise ValueError(f"the vector length must be a power of two, not {n}")
        out = np.zeros_like(points)
        self._call("vrfs_g1_fft_batch", int(n.bit_length() - 1), int(bool(inverse)), _p(points), _p(out))
        return out

    def g1_compress(self, points):
        """(n, 96) affine LE G1 points (zeros = identity) -> (n, 48) ark-bls12-381 / zcash compressed encodings"""
        points = _u8(points, (-1, 96)); out = np.zeros((len(points), 48), np.uint8)
        self._call("vrfs_g1_compress_batch", C.c_size_t(len(points)), _p(points), _p(out))
        return out

    def g1_decompress(self, enc, check_subgroup=True):
        """(n, 48) compressed encodings -> ((n, 96) affine LE points, ok flags); validated like CanonicalDeserialize"""
        enc = _u8(enc, (-1, 48)); out = np.zeros((len(enc), 96), np.uint8); ok = np.zeros(len(enc), np.uint8)
        self._call("vrfs_g1_decompress_batch", C.c_size_t(len(enc)), _p(enc), int(bool(check_subgroup)), _p(out), _p(ok))
        return out, ok

    def fq381_inv(self, values):
        """self-test helper: inverses in BLS12-381 Fq of (n, 48) canonical LE values -> (inverses, fast-path flags)"""
        values = _u8(values, (-1, 48)); out = np.zeros_like(values); ok = np.zeros(len(values), np.uint8)
        self._call("vrfs_fq381_inv_batch", C.c_size_t(len(values)), _p(values), _p(out), _p(ok))
        return out, ok

    # ---- BLS12-381 pairing / batched KZG opening check (SURVEY 8f-3)
    def pairing_products(self, g1, g2, n_pairs=1, negate_masks=None, want_gt=False):
        """n products of n_pairs pairings each: verdicts (1 = product is one, 0 = not, 2 = malformed point) [and GT values (n, 576)]"""
        g1 = _u8(g1, (-1, n_pairs * 96)); n = len(g1); g2 = _u8(g2, (n, n_pairs * 192))
        neg = None if negate_masks is None else np.ascontiguousarray(negate_masks, dtype=np.uint32).reshape(n)
        ok = np.zeros(n, np.uint8); gt = np.zeros((n, 576), np.uint8) if want_gt else None
        self._call("vrfs_pairing_product_batch", C.c_size_t(n), int(n_pairs), _p(g1), _p(g2), _p(neg), _p(ok), _p(gt))
        return (ok, gt) if want_gt else ok

    def kzg_batch_verify(self, commitments, zs, vs, proofs, rs, g2, tau_g2, check_points=1):
        """1 accepted / 0 rejected / 2 malformed point for k openings aggregated with the coefficients rs (vrfs_kzg_batch_verify)"""
        commitments = _u8(commitments, (-1, 96)); k = len(commitments)
        proofs = _u8(proofs, (k, 96)); zs = _u8(zs, (k, 32)); vs = _u8(vs, (k, 32)); rs = _u8(rs, (k, 32))
        g2 = _u8(g2, (192,)); tau_g2 = _u8(tau_g2, (192,))
        ok = np.zeros(1, np.uint8)
        self._call("vrfs_kzg_batch_verify", C.c_size_t(k), _p(commitments), _p(zs), _p(vs), _p(proofs), _p(rs), _p(g2), _p(tau_g2), int(check_points), _p(ok))
        return int(ok[0])

    # ---- measurement
    def enable_kernel_timing(self, on=True):
        self._check(self._lib.vrfs_ctx_enable_kernel_timing(self._ctx, int(bool(on))))

    def kernel_timings(self):
        """[(kernel name, device ms)] of the most recent batch call (syncs the stream)"""
        names = (C.c_char_p * 64)(); ms = (C.c_float * 64)()
        n = self._lib.vrfs_ctx_kernel_timings(self._ctx, names, ms, 64)
        return [(names[i].decode(), float(ms[i])) for i in range(n)]

    def measure_mac32_peak(self, variant=0):
        macs = C.c_double(); mhz = C.c_double()
        self._check(self._lib.vrfs_measure_mac32_peak(self._ctx, int(variant), C.byref(macs), C.byref(mhz)))
        return macs.value, mhz.value


class MultiPreparedBases:
    def __init__(self, mengine, handle, n):
        self.mengine, self.handle, self.n = mengine, handle, n

    def msm(self, scalars, n_columns=1):
        scalars = _u8(scalars, (n_columns * self.n, 32)); out = np.zeros((n_columns, 96), np.uint8)
        self.mengine._call("vrfs_multi_msm_g1_prepared", self.handle, _p(scalars), int(n_columns), _p(out))
        return out

    def ring_commit(self, keys, keyset_part_size, padding, tail):
        keys = _u8(keys, (-1, 64)); tail = _u8(tail, (-1, 64)); padding = _u8(padding, (64,)); out = np.zeros((3, 96), np.uint8)
        self.mengine._call("vrfs_multi_ring_commit", self.handle, C.c_size_t(keyset_part_size), C.c_size_t(len(keys)), _p(keys), _p(padding),
                           C.c_size_t(len(tail)), _p(tail), _p(out))
        return out

    def release(self):
        if self.handle:
            self.mengine._lib.vrfs_multi_msm_g1_release(self.handle)
            self.handle = None


class MultiEngine:
    """One caller, several GPUs of one node (vrfs_ctx_create_multi): verify batches are sharded by index range, the commitment
    MSM by point range with the partials exchanged device to device."""

    def __init__(self, devices):
        self._lib = _lib.load()
        self._m = C.c_void_p()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        st = self._lib.vrfs_ctx_create_multi(devs, len(devices), C.byref(self._m))
        if st != _lib.OK:
            msg = self._lib.vrfs_mctx_last_error(self._m).decode() if self._m else "context allocation failed"
            if self._m:
                self._lib.vrfs_mctx_destroy(self._m)
                self._m = None
            raise _lib.VrfsError(st, msg)
        self.devices = list(devices)
        self._prepared = []

    def _call(self, fn, *args):
        st = getattr(self._lib, fn)(self._m, *args)
        if st != _lib.OK:
            raise _lib.VrfsError(st, self._lib.vrfs_mctx_last_error(self._m).decode())

    @property
    def launch_count(self):
        return int(self._lib.vrfs_mctx_launch_count(self._m))

    def ietf_verify(self, suite, pk, inp, outp, c, s, ad=None, status=False):
        pk = _u8(pk, (-1, 64)); n = len(pk)
        inp = _u8(inp, (n, 64)); outp = _u8(outp, (n, 64)); c = _u8(c, (n, 32)); s = _u8(s, (n, 32))
        adb, off = pack_var(ad, n)
        ok = np.zeros(n, np.uint8); st = np.zeros(n, np.uint8) if status else None
        self._call("vrfs_multi_ietf_verify_batch", suite, C.c_size_t(n), _p(pk), _p(inp), _p(outp), _p(c), _p(s), _p(adb), _p(off), _p(ok), _p(st))
        return (ok, st) if status else ok

    def ietf_verify_host_ptrs(self, suite, n, pk, inp, outp, c, s, ok, ad=None, off=None, status=None):
        v = lambda x: C.c_void_p(x) if x else None
        self._call("vrfs_multi_ietf_verify_batch", suite, C.c_size_t(n), v(pk), v(inp), v(outp), v(c), v(s), v(ad), v(off), v(ok), v(status))

    def msm_g1_prepare(self, bases):
        bases = _u8(bases, (-1, 96)); h = C.c_void_p()
        self._call("vrfs_multi_msm_g1_prepare", C.c_size_t(len(bases)), _p(bases), C.byref(h))
        p = MultiPreparedBases(self, h, len(bases))
        self._prepared.append(p)
        return p

    def close(self):
        if getattr(self, "_m", None):
            for p in self._prepared:
                p.release()
            self._lib.vrfs_mctx_destroy(self._m)
            self._m = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
