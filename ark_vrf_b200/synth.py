"""Synthetic Thin- and Pedersen-VRF workloads (SURVEY.md section 8d), generated on the GPU.

Signer k has sk_k = Secret::from_seed(LE64(k) || 0^24) (reference src/lib.rs:346-369);
proof j is signed by k = j mod K; inputs I_{j,i} = data_to_point(LE64(j) || LE32(i));
O = sk * I; ad_j = b"ad-{j}" (reference benches/thin.rs:55); proofs by the reference's
deterministic prove (src/thin.rs:111-129; make_pedersen_batch: src/pedersen.rs:136-186).  Only `secret_from_seed` (two SHA-512 calls per
signer) runs on the host; everything else uses the library's feeder kernels.
"""
from __future__ import annotations

import hashlib
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import ops
from .thin import Format, Suite

SUITE_ID = {
    Suite.BANDERSNATCH_SHA512_ELL2: b"Bandersnatch-SHA512-ELL2-v1",
    Suite.ED25519_SHA512_TAI: b"Ed25519-SHA512-TAI-v1",
    Suite.BABYJUBJUB_SHA512_TAI: b"BabyJubJub-SHA512-TAI-v1",
}
ORDER = {
    Suite.BANDERSNATCH_SHA512_ELL2: 13108968793781547619861935127046491459309155893440570251786403306729687672801,
    Suite.ED25519_SHA512_TAI: 2**252 + 27742317777372353535851937790883648493,
    Suite.BABYJUBJUB_SHA512_TAI: 2736030358979909402780800718157159386076813972158567259200215660948447373041,
}
FIELD = {      # base-field moduli (SURVEY.md Appendix A.1)
    Suite.BANDERSNATCH_SHA512_ELL2: 52435875175126190479447740508185965837690552500527637822603658699938581184513,
    Suite.ED25519_SHA512_TAI: 2**255 - 19,
    Suite.BABYJUBJUB_SHA512_TAI: 21888242871839275222246405745257275088548364400416034343698204186575808495617,
}


def identity_point(suite, fmt: Format) -> np.ndarray:
    """The group identity (0, 1) as a 64-byte affine point in `fmt` (an InvalidData trigger, thin.rs:266-271)."""
    one = 1 if Format(fmt) == Format.CANONICAL else (1 << 256) % FIELD[Suite(suite)]
    return np.frombuffer(bytes(32) + one.to_bytes(32, "little"), dtype=np.uint8).copy()


def _stream(data: bytes, n: int) -> bytes:
    """HashTranscript squeeze (src/utils/transcript.rs:230-273)."""
    seed = hashlib.sha512(data).digest()
    out = b""
    i = 0
    while len(out) < n:
        out += hashlib.sha512(seed + i.to_bytes(8, "little")).digest()
        i += 1
    return out[:n]


def secret_from_seed(suite: Suite, seed: bytes) -> int:
    """Secret::from_seed (src/lib.rs:346-369) with utils::nonce (src/utils/common.rs:313-328)."""
    r = ORDER[Suite(suite)]
    sid = SUITE_ID[Suite(suite)]
    sk0 = int.from_bytes(seed, "little") % r
    cnt = 0
    while True:
        t = sid + seed + (bytes([cnt]) if cnt else b"")
        h = _stream(t + b"\x10" + sk0.to_bytes(32, "little"), 64)
        k = int.from_bytes(_stream(t + b"\x11" + h, (r.bit_length() + 128 + 7) // 8), "little") % r
        if k:
            return k
        cnt += 1


@dataclass
class Batch:
    suite: Suite
    fmt: Format
    n: int
    m: int
    pk: np.ndarray          # (n, 64)
    ios: np.ndarray         # (n*m, 128)  input || output
    io_offsets: np.ndarray  # (n+1,) uint32
    ad_blob: np.ndarray     # uint8
    ad_offsets: np.ndarray  # (n+1,) uint32
    r: np.ndarray           # (n, 64)
    s: np.ndarray           # (n, 32)
    sk: Optional[np.ndarray] = None   # (n, 32) canonical, per proof (kept for tests)

    @property
    def h2d_bytes(self) -> int:
        return (self.pk.nbytes + self.ios.nbytes + self.io_offsets.nbytes + self.ad_blob.nbytes +
                self.ad_offsets.nbytes + self.r.nbytes + self.s.nbytes)


def _mont_scalars(suite: Suite, sk_ints) -> np.ndarray:
    r = ORDER[Suite(suite)]
    return np.frombuffer(b"".join(((k << 256) % r).to_bytes(32, "little") for k in sk_ints), dtype=np.uint8).reshape(-1, 32).copy()


def _inputs(suite: Suite, n: int, m: int, signers: int, fmt: Format, first: int):
    """Signer keys, I/O pairs and ad of proofs first .. first+n-1 (shared by the Thin and Pedersen generators)."""
    K = max(1, min(signers, 4096))
    sk_int = [secret_from_seed(suite, k.to_bytes(8, "little") + bytes(24)) for k in range(K)]
    sk_can = np.frombuffer(b"".join(k.to_bytes(32, "little") for k in sk_int), dtype=np.uint8).reshape(K, 32)
    sk_fmt = sk_can if fmt == Format.CANONICAL else _mont_scalars(suite, sk_int)
    pk_k = ops.public_keys(suite, sk_fmt, fmt)
    j = np.arange(first, first + n, dtype=np.uint64)
    signer = (j % K).astype(np.int64)
    sk = np.ascontiguousarray(sk_fmt[signer])
    pk = np.ascontiguousarray(pk_k[signer])
    # messages LE64(j) || LE32(i)
    msgs = np.zeros((n, m, 12), dtype=np.uint8)
    msgs[:, :, :8] = j.view(np.uint8).reshape(n, 8)[:, None, :]
    msgs[:, :, 8:] = np.arange(m, dtype=np.uint32).view(np.uint8).reshape(m, 4)[None, :, :]
    moff = (np.arange(n * m + 1, dtype=np.uint64) * 12).astype(np.uint32)
    blob = np.concatenate([msgs.reshape(-1), np.zeros(16, dtype=np.uint8)])
    if n * m:
        inputs, ok = ops.hash_to_curve(suite, blob, moff, fmt)
        assert ok.all()
        outputs = ops.vrf_output(suite, np.repeat(sk, m, axis=0), inputs, fmt)
        ios = np.ascontiguousarray(np.concatenate([inputs, outputs], axis=1))
    else:
        ios = np.zeros((0, 128), dtype=np.uint8)
    io_offsets = (np.arange(n + 1, dtype=np.uint64) * m).astype(np.uint32)
    ads = [b"ad-%d" % int(x) for x in j]
    ad_offsets = np.zeros(n + 1, dtype=np.uint32)
    ad_offsets[1:] = np.cumsum([len(a) for a in ads], dtype=np.uint64).astype(np.uint32)
    ad_blob = np.frombuffer(b"".join(ads) + bytes(16), dtype=np.uint8).copy()
    return sk, pk, ios, io_offsets, ad_blob, ad_offsets


def make_batch(suite, n: int, m: int = 1, signers: int = 4096, fmt: Format = Format.MONTGOMERY,
               first: int = 0) -> Batch:
    """Proofs first .. first+n-1 of the synthetic set, as host arrays in `fmt`."""
    suite = Suite(suite)
    sk, pk, ios, io_offsets, ad_blob, ad_offsets = _inputs(suite, n, m, signers, fmt, first)
    r, s = ops.thin_prove_many(suite, sk, pk, ios, io_offsets, ad_blob, ad_offsets, fmt)
    return Batch(suite, Format(fmt), n, m, pk, ios, io_offsets, ad_blob, ad_offsets, r, s, sk)


@dataclass
class PedersenBatch:
    suite: Suite
    fmt: Format
    n: int
    m: int
    ios: np.ndarray         # (n*m, 128)  input || output
    io_offsets: np.ndarray  # (n+1,) uint32
    ad_blob: np.ndarray     # uint8
    ad_offsets: np.ndarray  # (n+1,) uint32
    pk_com: np.ndarray      # (n, 64)
    r: np.ndarray           # (n, 64)
    ok: np.ndarray          # (n, 64)
    s: np.ndarray           # (n, 32)
    sb: np.ndarray          # (n, 32)
    blinding: np.ndarray    # (n, 32) the blinding factor of each proof
    sk: np.ndarray          # (n, 32) per proof, in `fmt`
    pk: np.ndarray          # (n, 64) sk * G


def make_pedersen_batch(suite, n: int, m: int = 1, signers: int = 4096, fmt: Format = Format.MONTGOMERY,
                        first: int = 0) -> PedersenBatch:
    """The Pedersen twin of `make_batch`: the same signers, messages and ad, proofs by the GPU's
    pedersen::Prover::prove (src/pedersen.rs:136-186)."""
    suite = Suite(suite)
    sk, pk, ios, io_offsets, ad_blob, ad_offsets = _inputs(suite, n, m, signers, fmt, first)
    pk_com, r, ok, s, sb, blinding = ops.pedersen_prove_many(suite, sk, pk, ios, io_offsets, ad_blob, ad_offsets, fmt)
    return PedersenBatch(suite, Format(fmt), n, m, ios, io_offsets, ad_blob, ad_offsets, pk_com, r, ok, s, sb, blinding,
                         sk, pk)


def splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
    z = x
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
    return z ^ (z >> 31)
