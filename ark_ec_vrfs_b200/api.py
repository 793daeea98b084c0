"""Host-side mirror of the reference's public API for the hot path, in batch form.

The reference (ark-ec-vrfs = ark-vrf 0.1.0; names re-exported at /root/reference/src/lib.rs:13-17) exposes,
per item:  Secret::from_seed / Secret::public / Secret::output,  Input::new,  Output::hash,
ietf::Prover::prove / ietf::Verifier::verify,  pedersen::Prover::prove / pedersen::Verifier::verify,
and the ring commitment built by RingContext::verifier_key.  Here every type holds a BATCH of n values
(numpy uint8 arrays in the C ABI's layout) and every method is one call into libvrfs_b200.so; same names,
same argument meaning, and the reference's error behaviour mapped onto arrays:
   Result<(), Error>  ->  uint8[n], 1 = Ok(()), 0 = Err(_); with status=True also the variant per item
                          (ITEM_OK / ITEM_VERIFICATION_FAILURE / ITEM_INVALID_DATA = Ok / Error::VerificationFailure / Error::InvalidData)
   Option<Input>      ->  (Input, uint8[n] ok)
There is no CPU implementation behind these classes: constructing a Suite needs a CUDA device."""
from dataclasses import dataclass

import numpy as np

from .engine import Engine, BANDERSNATCH, ED25519, P256


# prime subgroup orders (SURVEY Appendix C), used only to judge whether a serialised scalar is canonical
_ORDER = {BANDERSNATCH: 0x1cfb69d4ca675f520cce760202687600ff8f87007419047174fd06b52876e7e1,
          ED25519: 2**252 + 27742317777372353535851937790883648493,
          P256: 0xffffffff00000000ffffffffffffffffbce6faada7179e84f3b9cac2fc632551}


class Error(Exception):
    """mirror of ark_vrf::Error for whole-call failures; per-item failures come back as flags"""


@dataclass
class Suite:
    """ark_vrf::Suite: one ciphersuite bound to one GPU context"""
    suite_id: int
    engine: Engine

    @classmethod
    def bandersnatch(cls, device=0):
        return cls(BANDERSNATCH, Engine(device))

    @classmethod
    def ed25519(cls, device=0):
        return cls(ED25519, Engine(device))

    @classmethod
    def secp256r1(cls, device=0):
        return cls(P256, Engine(device))

    @property
    def CHALLENGE_LEN(self):
        return self.engine.challenge_len(self.suite_id)

    # Suite::data_to_point / nonce / challenge / point_to_hash live on the typed values below
    def data_to_point(self, datas):
        pts, ok = self.engine.data_to_point(self.suite_id, datas)
        return pts, ok


@dataclass
class Public:
    suite: Suite
    points: np.ndarray          # (n, 64)

    def verify(self, input, output, ad, proof, status=False):
        """ietf::Verifier::verify -> uint8[n] (status=True: (ok, Error variant per item))"""
        return self.suite.engine.ietf_verify(self.suite.suite_id, self.points, input.points, output.points, proof.c, proof.s, ad, status=status)

    def encode(self):
        return self.suite.engine.point_encode(self.suite.suite_id, self.points)

    serialize_compressed = encode

    def prepare(self):
        """these keys prepared once for many verifies (per-key fixed-base tables on the suite's GPU) -> PreparedPublic"""
        return PreparedPublic(self.suite, self.suite.engine.public_keys_prepare(self.suite.suite_id, self.points))

    @staticmethod
    def prepare_compressed(suite, enc):
        """serialised keys (e.g. a published validator set) deserialised with validation and prepared once -> PreparedPublic whose
        verify_signatures takes serialised signatures by key index; key_ok = 0 where deserialize_compressed rejects the key"""
        return PreparedPublic(suite, suite.engine.public_keys_prepare_encoded(suite.suite_id, enc))

    @classmethod
    def deserialize_compressed(cls, suite, enc):
        """CanonicalDeserialize with validation (canonical, on curve, prime-order subgroup) -> (Public, ok flags)"""
        pts, ok = suite.engine.point_decode_checked(suite.suite_id, enc)
        return cls(suite, pts), ok

    @staticmethod
    def verify_signatures(suite, pk_enc, datas, signatures, ad=None, status=False):
        """serialised keys + VRF input data + serialised signatures (Output || ietf::Proof) -> (ok flags, Output::hash[, status]);
        one call: deserialise, Input::new, verify, hash"""
        return suite.engine.ietf_verify_wire(suite.suite_id, pk_enc, datas, signatures, ad, status=status)


@dataclass
class PreparedPublic:
    """a Public that is reused (Public.prepare): verify takes, per proof, the index of its key among the prepared ones"""
    suite: Suite
    keys: object                # engine.PreparedPublics

    @property
    def key_ok(self):
        """1 where the key is one Public.verify accepts"""
        return self.keys.key_ok

    def verify(self, key_index, input, output, ad, proof, status=False):
        """ietf::Verifier::verify with pk[i] = keys[key_index[i]] -> uint8[n] (status=True: (ok, Error variant per item));
        an index out of range is ITEM_INVALID_DATA for its item"""
        return self.keys.verify(key_index, input.points, output.points, proof.c, proof.s, ad, status=status)

    def verify_signatures(self, key_index, datas, signatures, ad=None, status=False):
        """Public.verify_signatures with pk_enc[i] = the encoding of key key_index[i] -> (ok flags, Output::hash[, status]);
        only for keys from Public.prepare_compressed"""
        return self.keys.verify_wire(key_index, datas, signatures, ad, status=status)

    def verify_prepared_input(self, key_index, inputs, input_index, output, ad, proof, status=False):
        """verify with input[i] = the point of prepared input input_index[i] (`inputs` from Input.prepare) -> uint8[n]
        (status=True: (ok, Error variant per item)); an input index out of range is ITEM_INVALID_DATA for its item"""
        return self.keys.verify_io(inputs.inputs, key_index, input_index, output.points, proof.c, proof.s, ad, status=status)

    def verify_signatures_prepared_input(self, key_index, inputs, input_index, signatures, ad=None, status=False):
        """verify_signatures with datas[i] = the data of prepared input input_index[i] -> (ok flags, Output::hash[, status]);
        only for keys from Public.prepare_compressed; no hash-to-curve per signature"""
        return self.keys.verify_io_wire(inputs.inputs, key_index, input_index, signatures, ad, status=status)

    def release(self):
        self.keys.release()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.release()


@dataclass
class Input:
    suite: Suite
    points: np.ndarray

    @classmethod
    def new(cls, suite, datas):
        """Input::new(data) = Suite::data_to_point; returns (Input, ok flags) for Option<Input>"""
        pts, ok = suite.engine.data_to_point(suite.suite_id, datas)
        return cls(suite, pts), ok

    @staticmethod
    def prepare(suite, datas):
        """Input::new of a few inputs that many proofs share (a lottery or beacon round), done once, with a fixed-base table per input
        point on the suite's GPU -> PreparedInput, whose proofs PreparedPublic verifies by input index"""
        return PreparedInput(suite, suite.engine.inputs_prepare(suite.suite_id, datas))


@dataclass
class PreparedInput:
    """Inputs that are reused (Input.prepare)"""
    suite: Suite
    inputs: object              # engine.PreparedInputs

    @property
    def input_ok(self):
        """Input::new's Option as flags: 0 where no point was found"""
        return self.inputs.input_ok

    @property
    def points(self):
        return self.inputs.points

    def release(self):
        self.inputs.release()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.release()


@dataclass
class Output:
    suite: Suite
    points: np.ndarray

    def hash(self):
        """Output::hash = Suite::point_to_hash"""
        return self.suite.engine.point_to_hash(self.suite.suite_id, self.points)

    def serialize_compressed(self):
        return self.suite.engine.point_encode(self.suite.suite_id, self.points)

    @classmethod
    def deserialize_compressed(cls, suite, enc):
        pts, ok = suite.engine.point_decode_checked(suite.suite_id, enc)
        return cls(suite, pts), ok


@dataclass
class IetfProof:
    c: np.ndarray               # (n, 32) little-endian scalars
    s: np.ndarray

    def to_bytes(self, suite):
        """codec layout c (cLen bytes) || s (32 bytes), in the suite's scalar encoding"""
        cl = suite.CHALLENGE_LEN
        if suite.suite_id == P256:
            return np.concatenate([self.c[:, :cl][:, ::-1], self.s[:, ::-1]], axis=1)
        return np.concatenate([self.c[:, :cl], self.s], axis=1)

    @classmethod
    def from_bytes(cls, suite, raw):
        """inverse of to_bytes; returns (proof, ok) - ok = 0 where s is not a canonical scalar (the engine reduces c mod r)"""
        cl = suite.CHALLENGE_LEN
        raw = np.asarray(raw, np.uint8).reshape(-1, cl + 32)
        be = suite.suite_id == P256
        c = np.zeros((len(raw), 32), np.uint8)
        c[:, :cl] = raw[:, :cl][:, ::-1] if be else raw[:, :cl]
        s = np.ascontiguousarray(raw[:, cl:][:, ::-1] if be else raw[:, cl:])
        r = _ORDER[suite.suite_id]
        ok = np.array([int.from_bytes(x.tobytes(), "little") < r for x in s], np.uint8)
        return cls(c, s), ok


@dataclass
class PedersenProof:
    raw: np.ndarray             # (n, 256): pk_com || r || ok || s || sb

    pk_com = property(lambda self: self.raw[:, 0:64])
    r = property(lambda self: self.raw[:, 64:128])
    ok = property(lambda self: self.raw[:, 128:192])
    s = property(lambda self: self.raw[:, 192:224])
    sb = property(lambda self: self.raw[:, 224:256])

    def to_bytes(self, suite):
        """CanonicalSerialize: point_encode(pk_com) || point_encode(r) || point_encode(ok) || s || sb (160 B for the 32-byte codecs)"""
        e = suite.engine; sid = suite.suite_id
        sc = (lambda a: a[:, ::-1]) if sid == P256 else (lambda a: a)
        return np.concatenate([e.point_encode(sid, self.pk_com), e.point_encode(sid, self.r), e.point_encode(sid, self.ok), sc(self.s), sc(self.sb)], axis=1)

    @classmethod
    def from_bytes(cls, suite, raw):
        """CanonicalDeserialize with validation of the three points -> (proof, ok flags)"""
        e = suite.engine; sid = suite.suite_id; L = e.point_enc_len(sid)
        raw = np.asarray(raw, np.uint8).reshape(-1, 3 * L + 64)
        pts, oks = zip(*(e.point_decode_checked(sid, np.ascontiguousarray(raw[:, k * L:(k + 1) * L])) for k in range(3)))
        sc = (lambda a: a[:, ::-1]) if sid == P256 else (lambda a: a)
        s, sb = sc(raw[:, 3 * L:3 * L + 32]), sc(raw[:, 3 * L + 32:])
        r = _ORDER[sid]
        canon = np.array([int.from_bytes(a.tobytes(), "little") < r and int.from_bytes(b.tobytes(), "little") < r for a, b in zip(s, sb)], np.uint8)
        return cls(np.ascontiguousarray(np.concatenate(list(pts) + [s, sb], axis=1))), oks[0] & oks[1] & oks[2] & canon


@dataclass
class Secret:
    suite: Suite
    scalars: np.ndarray         # (n, 32)
    public_points: np.ndarray   # (n, 64)

    @classmethod
    def from_seed(cls, suite, seeds):
        sk, pk = suite.engine.secret_from_seed(suite.suite_id, seeds)
        return cls(suite, sk, pk)

    def public(self):
        return Public(self.suite, self.public_points)

    def output(self, input):
        return Output(self.suite, self.suite.engine.output(self.suite.suite_id, self.scalars, input.points))

    def prove(self, input, output, ad=None):
        """ietf::Prover::prove"""
        c, s = self.suite.engine.ietf_prove(self.suite.suite_id, self.scalars, input.points, output.points, ad)
        return IetfProof(c, s)

    def sign(self, datas, ad=None):
        """Input::new(data) -> output -> ietf prove -> serialised signatures point_encode(Output) || c || s; returns (sig, ok)"""
        return self.suite.engine.ietf_sign_wire(self.suite.suite_id, self.scalars, datas, ad)

    def pedersen_sign(self, datas, ad=None):
        """Input::new(data) -> output -> pedersen prove -> serialised Output || pedersen::Proof; returns (sig, blinding, ok)"""
        return self.suite.engine.pedersen_sign_wire(self.suite.suite_id, self.scalars, datas, ad)

    def pedersen_prove(self, input, output, ad=None, serialized=False):
        """pedersen::Prover::prove -> (Proof, blinding); serialized=True returns the proofs' CanonicalSerialize bytes instead
        (3 encoded points + s + sb, 160 B each for Bandersnatch)"""
        if serialized:
            return self.suite.engine.pedersen_prove_compressed(self.suite.suite_id, self.scalars, input.points, output.points, ad)
        pr, bl = self.suite.engine.pedersen_prove(self.suite.suite_id, self.scalars, input.points, output.points, ad)
        return PedersenProof(pr), bl


def pedersen_verify(suite, input, output, ad, proof, status=False):
    """pedersen::Verifier::verify (needs no public key) -> uint8[n].  `proof`: a PedersenProof, or the serialised proofs
    ((n, proof_len) bytes, 160 B each for Bandersnatch) which are deserialised with validation on the GPU first"""
    if isinstance(proof, PedersenProof):
        return suite.engine.pedersen_verify(suite.suite_id, input.points, output.points, proof.raw, ad, status=status)
    return suite.engine.pedersen_verify_compressed(suite.suite_id, input.points, output.points, proof, ad, status=status)


def pedersen_verify_signatures(suite, datas, signatures, ad=None, status=False):
    """serialised Output || pedersen::Proof + VRF input data -> ok flags (deserialise with validation, Input::new, verify)"""
    return suite.engine.pedersen_verify_wire(suite.suite_id, datas, signatures, ad, status=status)


def pedersen_batch_verify(suite, input, output, ad, proof, seed=None, per_item=False, status=False):
    """all of a batch of Pedersen proofs (a PedersenProof) verified together by one random linear combination -> bool
    (Bandersnatch only).  seed: 32 secret bytes, fresh per call (default os.urandom(32)).  per_item / status=True append the
    per-item verdicts, which the per-item verifier computes only when the batch is rejected."""
    return suite.engine.pedersen_batch_verify(suite.suite_id, input.points, output.points, proof.raw, ad, seed=seed, per_item=per_item, status=status)


def pedersen_batch_verify_signatures(suite, datas, signatures, ad=None, seed=None, per_item=False, status=False):
    """pedersen_batch_verify from serialised Output || pedersen::Proof signatures and VRF input data"""
    return suite.engine.pedersen_batch_verify_wire(suite.suite_id, datas, signatures, ad, seed=seed, per_item=per_item, status=status)


def ring_commitment_msm(suite_or_engine, bases, scalar_columns):
    """the three KZG commitments behind RingContext::verifier_key: one MSM per column over the SRS bases"""
    eng = suite_or_engine.engine if isinstance(suite_or_engine, Suite) else suite_or_engine
    cols = np.concatenate([np.asarray(c, np.uint8).reshape(-1, 32) for c in scalar_columns])
    return eng.msm_g1(bases, cols, len(scalar_columns))


# ---- ring (SURVEY.md 8f-2): the verifier-key part of `ring::RingContext` ------------------------------------------------------
# [RECALL, unpinned] ring-proof's PiopParams: the domain keeps ZK_ROWS = 3 rows for blinding (capacity = N - 3), the fixed
# columns hold `keyset_part_size = capacity - scalar_bitlen - 1` key slots (unused ones filled with the suite's padding point)
# followed by the scalar_bitlen powers 2^j * H of the Pedersen blinding base; the selector is 1 on the key slots.  These numbers
# are DEFAULTS of this mirror, passed to the engine as parameters; the engine itself hard-codes none of them.
RING_ZK_ROWS = 3


def g1_compress(points):
    """host-side twin of Engine.g1_compress (kept as an independent cross-check for the tests):
    ark-bls12-381's G1 `serialize_compressed` (the zcash format): 48 bytes big-endian x; bit 7 of byte 0 = compressed,
    bit 6 = infinity, bit 5 = y is the lexicographically larger root.  points: (n, 96) affine LE, zeros = identity."""
    P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
    pts = np.asarray(points, np.uint8).reshape(-1, 96); out = np.zeros((len(pts), 48), np.uint8)
    for i, p in enumerate(pts):
        if not p.any():
            out[i, 0] = 0xC0
            continue
        x = int.from_bytes(p[:48].tobytes(), "little"); y = int.from_bytes(p[48:].tobytes(), "little")
        b = bytearray(x.to_bytes(48, "big")); b[0] |= 0x80 | (0x20 if y > P - y else 0)
        out[i] = np.frombuffer(bytes(b), np.uint8)
    return out


class RingContext:
    """Holds the prepared SRS of one domain size and commits to rings of public keys: `RingContext::verifier_key(pks)` up to the
    commitment (`RingCommitment` = cx, cy, selector).  srs_g1: (N, 96) affine G1 points, either the Lagrange basis [L_i(tau)]G1
    over the radix-2 domain (lagrange=True, ring-proof's updatable `Ring`) or the monomial powers [tau^i]G1 (lagrange=False)."""

    def __init__(self, suite, srs_g1, lagrange, padding, blinding_base_powers, keyset_part_size=None):
        self.suite, self.engine, self.lagrange = suite, suite.engine, bool(lagrange)
        srs_g1 = np.asarray(srs_g1, np.uint8).reshape(-1, 96)
        self.domain_size = len(srs_g1)
        assert self.domain_size & (self.domain_size - 1) == 0, "the SRS must cover a power-of-two domain"
        self.tail = np.asarray(blinding_base_powers, np.uint8).reshape(-1, 64)
        self.padding = np.asarray(padding, np.uint8).reshape(64)
        self.keyset_part_size = (self.domain_size - RING_ZK_ROWS - len(self.tail) - 1) if keyset_part_size is None else int(keyset_part_size)
        self.srs = self.engine.msm_g1_prepare(srs_g1)
        self._empty = None                                            # commitment of the ring of padding only (Lagrange SRS)

    @classmethod
    def from_compressed_srs(cls, suite, srs_bytes, lagrange, padding, blinding_base_powers, keyset_part_size=None, check_subgroup=True):
        """the SRS as it is stored (48-byte compressed G1 points, ark-bls12-381 / zcash format): validated on the GPU
        (canonical, on curve, prime-order subgroup) like `deserialize_compressed`; raises ValueError on the first bad point"""
        pts, ok = suite.engine.g1_decompress(np.asarray(srs_bytes, np.uint8).reshape(-1, 48), check_subgroup)
        if not ok.all():
            raise ValueError("SRS point %d is not a valid compressed G1 point" % int(np.argmin(ok)))
        return cls(suite, pts, lagrange, padding, blinding_base_powers, keyset_part_size)

    @classmethod
    def from_powers(cls, suite, powers_g1, domain_size, padding, blinding_base_powers, keyset_part_size=None):
        """ring-proof's `RingBuilderKey::from_srs`: the published monomial powers [tau^j]G1 ((m, 96) affine points in G1, m >= domain_size;
        an SRS is longer, only the first domain_size are used) -> their Lagrange basis over the radix-2 domain (one inverse G1 FFT on the
        GPU) -> a Lagrange-basis context, whose verifier_key_commitment takes the incremental path"""
        powers = np.asarray(powers_g1, np.uint8).reshape(-1, 96)
        n = int(domain_size)
        if n < 1 or n & (n - 1):
            raise ValueError(f"domain_size must be a power of two, not {n}")
        if len(powers) < n:
            raise ValueError(f"{len(powers)} powers of tau for a domain of {n}")
        lagrange = suite.engine.g1_fft(powers[:n], inverse=True)
        return cls(suite, lagrange, True, padding, blinding_base_powers, keyset_part_size)

    def max_ring_size(self):
        return self.keyset_part_size

    def fixed_columns(self, public_keys):
        return self.engine.ring_fixed_columns(self.domain_size, self.keyset_part_size, public_keys, self.padding, self.tail)

    def verifier_key_commitment(self, public_keys, incremental=None):
        """(3, 96) affine commitments cx, cy, selector.  With a Lagrange-basis SRS the commitment of the all-padding ring is kept
        and only sum (pk_i - padding) L_i over the real keys is computed per ring (incremental=False forces the full MSM)"""
        keys = np.asarray(public_keys, np.uint8).reshape(-1, 64)
        if incremental is None:
            incremental = self.lagrange
        if not incremental:
            return self.srs.ring_commit(keys, self.keyset_part_size, self.padding, self.tail, self.lagrange)
        assert self.lagrange, "the incremental form needs a Lagrange-basis SRS"
        assert len(keys) <= self.keyset_part_size
        if self._empty is None:
            self._empty = self.srs.ring_commit(np.zeros((0, 64), np.uint8), self.keyset_part_size, self.padding, self.tail, True)
        delta = self.srs.ring_commit_delta(keys, self.padding)
        parts = np.zeros((2, 3, 144), np.uint8)                       # projective X | Y | Z; identity (0 : 1 : 0)
        for k, pts in enumerate((self._empty, np.concatenate([delta, np.zeros((1, 96), np.uint8)]))):
            for c in range(3):
                if pts[c].any():
                    parts[k, c, :96] = pts[c]; parts[k, c, 96] = 1
                else:
                    parts[k, c, 48] = 1
        return self.engine.g1_sum_partials(parts, 3)

    def ring_commitment_bytes(self, public_keys):
        """the 144-byte serialised RingCommitment: three compressed G1 points"""
        return self.engine.g1_compress(self.verifier_key_commitment(public_keys)).reshape(-1)

    def release(self):
        self.srs.release()
