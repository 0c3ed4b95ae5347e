"""Synthetic signed-packet workloads for tests and bench.py (SURVEY §8d configs 2/3/5).

Not on the hot path: this only MAKES inputs (RSA signing on the host with OpenSSL via
`cryptography`, packet bytes per packet/packet.go:35-60) — verification is never done here."""
import hashlib
import json
import os
import struct
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
KEYS_JSON = os.path.join(_HERE, "..", "tests", "golden", "rsa_keys_bf7c0001.json")
SHA256_PREFIX = bytes.fromhex("3031300d060960864801650304020105000420")


def load_keys(k: int):
    """First k deterministic RSA-2048 test keys: list of dicts with p, q, n, d, e (ints)."""
    data = json.load(open(KEYS_JSON))
    out = []
    for kd in data["keys"][:k]:
        p, q = int(kd["p"], 16), int(kd["q"], 16)
        n, e = p * q, data["e"]
        d = pow(e, -1, (p - 1) * (q - 1))
        out.append({"p": p, "q": q, "n": n, "d": d, "e": e})
    assert len(out) == k, "not enough fixture keys"
    return out


def _private_key(k):
    from cryptography.hazmat.primitives.asymmetric.rsa import RSAPrivateNumbers, RSAPublicNumbers
    p, q, d = k["p"], k["q"], k["d"]
    return RSAPrivateNumbers(p, q, d, d % (p - 1), d % (q - 1), pow(q, -1, p),
                             RSAPublicNumbers(k["e"], k["n"])).private_key()


def tbs_packet(x: bytes, v: bytes, t: int) -> bytes:
    """packet.Serialize(x, v, t) == the TBS bytes (packet/packet.go:35-60,156-168)."""
    return struct.pack(">Q", len(x)) + x + struct.pack(">Q", len(v)) + v + struct.pack(">Q", t)


def make_verify_batch(n_items: int, n_keys: int = 16, seed: int = 0xBF7C0002, corrupt_rate: float = 0.01,
                      unknown_rate: float = 0.001, corrupt_seed: int = 0xBF7C0003, threads: int = 0):
    """Config 2: N tuples over K keys.  message_i = packet.Serialize(x_i(16 B), v_i(32 B), t=i);
    digest_i = SHA-256(message_i) (the raw PKCS#1 case; the OpenPGP v4 digest adds a suffix, see
    pgp host layer); signatures by OpenSSL; a seeded fraction corrupted / given an unknown key.
    Returns dict(keys, key_idx u32[N], sig u8[N,256], digest u8[N,32], expect u8[N])."""
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import padding
    from cryptography.hazmat.primitives.asymmetric.utils import Prehashed
    keys = load_keys(n_keys)
    privs = [_private_key(k) for k in keys]
    rng = np.random.default_rng(seed)
    key_idx = rng.integers(0, n_keys, n_items).astype(np.uint32)
    xv = rng.integers(0, 256, (n_items, 48), dtype=np.uint8)
    digest = np.empty((n_items, 32), np.uint8)
    sig = np.empty((n_items, 256), np.uint8)
    threads = threads or min(32, os.cpu_count() or 1)

    def work(lo_hi):
        lo, hi = lo_hi
        pad, ph = padding.PKCS1v15(), Prehashed(hashes.SHA256())
        for i in range(lo, hi):
            m = tbs_packet(xv[i, :16].tobytes(), xv[i, 16:].tobytes(), i)
            d = hashlib.sha256(m).digest()
            digest[i] = np.frombuffer(d, np.uint8)
            sig[i] = np.frombuffer(privs[key_idx[i]].sign(d, pad, ph), np.uint8)

    step = max(1, (n_items + threads * 4 - 1) // (threads * 4))
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(work, [(lo, min(n_items, lo + step)) for lo in range(0, n_items, step)]))
    expect = np.zeros(n_items, np.uint8)
    crng = np.random.default_rng(corrupt_seed)
    bad = crng.random(n_items) < corrupt_rate
    for i in np.nonzero(bad)[0]:
        sig[i, crng.integers(0, 256)] ^= np.uint8(1 << crng.integers(0, 8))
        expect[i] = 1
    unk = crng.random(n_items) < unknown_rate
    key_idx[unk] = n_keys + 7
    expect[unk] = 4
    return {"keys": keys, "key_idx": key_idx, "sig": sig, "digest": digest, "expect": expect}


def em_for_digest(digest: bytes) -> int:
    return int.from_bytes(b"\x00\x01" + b"\xff" * 202 + b"\x00" + SHA256_PREFIX + digest, "big")


# Per-operation response mixes for make_read_ops: (share of the operations, p_ok, p_stale, p_bad); the rest of each
# operation's replicas do not answer.  HARD_MIX makes a visible part of the operations end rejected or undecided, and
# some decide on the stale value, so that every arm of Client.Read's decision is exercised at scale.
HARD_MIX = [(0.80, 0.90, 0.05, 0.03), (0.08, 0.35, 0.30, 0.15), (0.07, 0.25, 0.05, 0.45), (0.05, 0.15, 0.60, 0.10)]


def make_read_ops(pool, n_ops: int, n_replicas: int, seed: int = 0xBF7C0004, p_ok=0.90, p_stale=0.05, p_bad=0.03, mix=None,
                  shuffle_arrival=False):
    """Configs 3 / 5: M read ops x R replicas.  Replica r of every op answers with key r.  Each
    response is (valid, current value) w.p. p_ok, (valid, stale t) p_stale, invalid signature p_bad,
    missing otherwise (SURVEY §8d).  Signed tuples are drawn from `pool` (make_verify_batch output
    with n_keys == n_replicas, no corruption): slot (op, r) takes a pool item signed by key r, so
    every signature is genuine; uniqueness across ops is limited by the pool size (stated in
    bench.py's `data`).  mix: per-operation classes [(share, p_ok, p_stale, p_bad), ...] instead of one
    global triple (HARD_MIX).  shuffle_arrival: the responses of an operation arrive in a seeded random
    order instead of replica order (Client.Read's decision depends on it).  Returns op_off, key_idx, sig,
    digest, pre_status, ts, value_id and the expected per-item status."""
    rng = np.random.default_rng(seed)
    R, M = n_replicas, n_ops
    by_key = [np.nonzero(pool["key_idx"] == r)[0] for r in range(R)]
    assert all(len(b) for b in by_key), "pool lacks items for some replica key"
    N = M * R
    key_idx = np.tile(np.arange(R, dtype=np.uint32), M)
    if shuffle_arrival:
        key_idx = rng.permuted(key_idx.reshape(M, R), axis=1).reshape(N).astype(np.uint32)
    pick = np.empty(N, np.int64)
    for r in range(R):
        sel = np.nonzero(key_idx == r)[0]
        pick[sel] = by_key[r][rng.integers(0, len(by_key[r]), len(sel))]
    sig = pool["sig"][pick]
    digest = pool["digest"][pick]
    u = rng.random(N)
    if mix is None:
        pk, ps, pb = p_ok, p_stale, p_bad
    else:
        cls = rng.choice(len(mix), size=M, p=[m[0] for m in mix])
        pk = np.repeat(np.array([m[1] for m in mix])[cls], R)
        ps = np.repeat(np.array([m[2] for m in mix])[cls], R)
        pb = np.repeat(np.array([m[3] for m in mix])[cls], R)
    kind = np.where(u < pk, 0, np.where(u < pk + ps, 1, np.where(u < pk + ps + pb, 2, 3)))
    bad = np.nonzero(kind == 2)[0]
    sig[bad, rng.integers(0, 256, len(bad))] ^= np.uint8(0x10)
    pre = np.where(kind == 3, 6, 0).astype(np.uint8)                  # BFTQ_ST_MISSING
    ts = np.where(kind == 1, 6, 7).astype(np.uint64)                  # stale replicas are one write behind
    value_id = np.where(kind == 1, 1, 0).astype(np.uint32)
    expect = np.where(kind == 2, 1, pre).astype(np.uint8)
    op_off = (np.arange(M + 1, dtype=np.uint64) * R).astype(np.uint32)
    return {"op_off": op_off, "key_idx": key_idx, "sig": sig, "digest": digest, "pre_status": pre, "ts": ts,
            "value_id": value_id, "expect_status": expect}


# ---- OpenPGP-packet form of config 2: what crypto.Signature.Verify actually receives -----------------

def _mpi(x: int) -> bytes:
    return struct.pack(">H", x.bit_length()) + x.to_bytes((x.bit_length() + 7) // 8, "big")


def _old_packet(tag: int, body: bytes) -> bytes:
    """Old-format header with a 2-octet length (what GnuPG writes for keys and signatures)."""
    if tag == 13 and len(body) < 256:
        return bytes([0x80 | (tag << 2) | 0, len(body)]) + body
    return bytes([0x80 | (tag << 2) | 1]) + struct.pack(">H", len(body)) + body


def pgp_key_id(pub_body: bytes) -> int:
    """Low 64 bits of SHA-1(0x99 || len16 || public-key packet body) (RFC 4880 §12.2)."""
    return int.from_bytes(hashlib.sha1(b"\x99" + struct.pack(">H", len(pub_body)) + pub_body).digest()[12:], "big")


def _v4_sig_packet(priv, key_id: int, sig_type: int, hashed_prefix: bytes, ctime: int, extra_hashed: bytes = b"") -> bytes:
    """A v4 RSA/SHA-256 signature packet over `hashed_prefix` (the bytes hashed before the signature's
    own hashed area), RFC 4880 §5.2.3/§5.2.4: hashed = creation time (+ extra), unhashed = issuer."""
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import padding
    from cryptography.hazmat.primitives.asymmetric.utils import Prehashed
    hashed = bytes([5, 2]) + struct.pack(">I", ctime) + extra_hashed
    head = bytes([4, sig_type, 1, 8]) + struct.pack(">H", len(hashed)) + hashed
    digest = hashlib.sha256(hashed_prefix + head + b"\x04\xff" + struct.pack(">I", len(head))).digest()
    s = int.from_bytes(priv.sign(digest, padding.PKCS1v15(), Prehashed(hashes.SHA256())), "big")
    unhashed = bytes([9, 16]) + struct.pack(">Q", key_id)
    return _old_packet(2, head + struct.pack(">H", len(unhashed)) + unhashed + digest[:2] + _mpi(s))


def pgp_public_key_block(k, priv, uid: bytes, ctime: int = 0x5E000000):
    """Transferable public key: public-key packet, user id, positive self-certification with key
    flags certify|sign.  Returns (block bytes, key id)."""
    body = bytes([4]) + struct.pack(">I", ctime) + bytes([1]) + _mpi(k["n"]) + _mpi(k["e"])
    kid = pgp_key_id(body)
    prefix = b"\x99" + struct.pack(">H", len(body)) + body + b"\xb4" + struct.pack(">I", len(uid)) + uid
    selfsig = _v4_sig_packet(priv, kid, 0x13, prefix, ctime, extra_hashed=bytes([2, 27, 0x03]))
    return _old_packet(6, body) + _old_packet(13, uid) + selfsig, kid


def make_pgp_verify_batch(n_items: int, n_keys: int = 16, seed: int = 0xBF7C0002, corrupt_rate: float = 0.01,
                          unknown_rate: float = 0.001, corrupt_seed: int = 0xBF7C0003, threads: int = 0):
    """Config 2 in the form crypto.Signature.Verify sees it (crypto_pgp.go:319-330): tbs_i =
    packet.Serialize(x_i, v_i, t=i) and sig_i = ONE detached OpenPGP v4 RSA-2048/SHA-256 signature
    packet (binary, type 0x00) by key key_idx[i]; a seeded fraction has a flipped bit in the signature
    MPI (-> ErrInvalidSignature) or is issued by a key outside the keyring (-> ErrUnknownIssuer, which
    Verify also reports as ErrInvalidSignature).  Returns dict(keyring=public key blocks of the n_keys
    keys, key_ids, tbs=[bytes], sigs=[bytes], expect_ok bool[N], key_idx)."""
    keys = load_keys(n_keys + 1)                      # the extra key signs the "unknown issuer" items
    privs = [_private_key(k) for k in keys]
    blocks, kids = [], []
    for i, k in enumerate(keys):
        b, kid = pgp_public_key_block(k, privs[i], b"bftq-node-%02d <n%02d@bftq.test>" % (i, i))
        blocks.append(b); kids.append(kid)
    rng = np.random.default_rng(seed)
    key_idx = rng.integers(0, n_keys, n_items).astype(np.uint32)
    xv = rng.integers(0, 256, (n_items, 48), dtype=np.uint8)
    crng = np.random.default_rng(corrupt_seed)
    bad = crng.random(n_items) < corrupt_rate
    bad_byte = crng.integers(0, 200, n_items)
    bad_bit = crng.integers(0, 8, n_items)
    unk = crng.random(n_items) < unknown_rate
    tbs = [None] * n_items
    sigs = [None] * n_items
    threads = threads or min(32, os.cpu_count() or 1)

    def work(lo_hi):
        lo, hi = lo_hi
        for i in range(lo, hi):
            m = tbs_packet(xv[i, :16].tobytes(), xv[i, 16:].tobytes(), i)
            ki = n_keys if unk[i] else int(key_idx[i])
            pkt = bytearray(_v4_sig_packet(privs[ki], kids[ki], 0x00, m, 0x5F000000 + (i & 0xFFFF)))
            if bad[i]:
                pkt[len(pkt) - 1 - int(bad_byte[i])] ^= 1 << int(bad_bit[i])      # inside the 256-byte MPI
            tbs[i], sigs[i] = m, bytes(pkt)

    step = max(1, (n_items + threads * 4 - 1) // (threads * 4))
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(work, [(lo, min(n_items, lo + step)) for lo in range(0, n_items, step)]))
    return {"keyring": b"".join(blocks[:n_keys]), "key_ids": kids[:n_keys], "outsider_block": blocks[n_keys],
            "tbs": tbs, "sigs": sigs, "expect_ok": ~(bad | unk), "key_idx": key_idx}


# ---- hand-built signature packets of the rarer kinds (v3 packets, any digest) for the parity tests ----------------
# DigestInfo prefixes: Go crypto/rsa hashPrefixes == crypto/threshold/rsa/rsa.go:345-354, by OpenPGP hash id.
_DIGESTINFO = {
    1: "3020300c06082a864886f70d020505000410", 2: "3021300906052b0e03021a05000414", 3: "3021300906052b2403020105000414",
    8: "3031300d060960864801650304020105000420", 9: "3041300d060960864801650304020205000430",
    10: "3051300d060960864801650304020305000440", 11: "302d300d06096086480165030402040500041c"}
_HASHLIB = {1: "md5", 2: "sha1", 3: "ripemd160", 8: "sha256", 9: "sha384", 10: "sha512", 11: "sha224"}


def raw_rsa_sign(k, hash_id: int, digest: bytes) -> int:
    """EMSA-PKCS1-v1_5 signature by textbook exponentiation (k carries d): works for digests OpenSSL refuses to sign.
    With the primes in k the exponentiation goes through the CRT (same signature, about four times faster)."""
    t = bytes.fromhex(_DIGESTINFO[hash_id]) + digest
    klen = (k["n"].bit_length() + 7) // 8
    em = int.from_bytes(b"\x00\x01" + b"\xff" * (klen - len(t) - 3) + b"\x00" + t, "big")
    if "p" not in k:
        return pow(em, k["d"], k["n"])
    p, q = k["p"], k["q"]
    sp, sq = pow(em, k["d"] % (p - 1), p), pow(em, k["d"] % (q - 1), q)
    return sq + q * ((sp - sq) * pow(q, -1, p) % p)


def canonical_text(data: bytes) -> bytes:
    """Text-mode canonicalisation as x/crypto's canonicalTextHash does it: bare LF -> CRLF, CRLF kept."""
    out, i = bytearray(), 0
    while i < len(data):
        if data[i] == 0x0D and i + 1 < len(data) and data[i + 1] == 0x0A:
            out += b"\r\n"; i += 2
        elif data[i] == 0x0A:
            out += b"\r\n"; i += 1
        else:
            out.append(data[i]); i += 1
    return bytes(out)


def sig_packet_v3(k, key_id: int, hash_id: int, data: bytes, ctime: int, sig_type: int = 0) -> bytes:
    """A version-3 RSA signature packet (RFC 4880 §5.2.2): digest = H(data || sig type || creation time).
    `data` is signed as given for sig_type 0 and after text canonicalisation for sig_type 1."""
    signed = canonical_text(data) if sig_type == 1 else data
    suffix = bytes([sig_type]) + struct.pack(">I", ctime)
    d = hashlib.new(_HASHLIB[hash_id], signed + suffix).digest()
    body = bytes([3, 5]) + suffix + struct.pack(">Q", key_id) + bytes([1, hash_id]) + d[:2] + _mpi(raw_rsa_sign(k, hash_id, d))
    return _old_packet(2, body)


def sig_packet_v4(k, key_id: int, hash_id: int, data: bytes, ctime: int, sig_type: int = 0, plus_n: bool = False) -> bytes:
    """A version-4 RSA signature packet with any digest (hashed: creation time; unhashed: issuer).
    plus_n: store s + n instead of s (same residue; Go 1.13 accepts it, Go >= 1.20 rejects s >= n) — None if s + n needs 2049 bits."""
    signed = canonical_text(data) if sig_type == 1 else data
    hashed = bytes([5, 2]) + struct.pack(">I", ctime)
    head = bytes([4, sig_type, 1, hash_id]) + struct.pack(">H", len(hashed)) + hashed
    d = hashlib.new(_HASHLIB[hash_id], signed + head + b"\x04\xff" + struct.pack(">I", len(head))).digest()
    unhashed = bytes([9, 16]) + struct.pack(">Q", key_id)
    sv = raw_rsa_sign(k, hash_id, d)
    if plus_n:
        sv += k["n"]
        if sv.bit_length() > 2048:
            return None
    return _old_packet(2, head + struct.pack(">H", len(unhashed)) + unhashed + d[:2] + _mpi(sv))


# ---- transport messages: what openpgp.Encrypt(signer) puts inside the SymmetricallyEncrypted packet --------------------
# crypto_pgp.go:418-451 (Message.Encrypt / EncryptStream): one-pass signature, literal data (binary, FileName =
# base64(nonce), time 0), signature — each written by x/crypto's serializers: new-format headers, and the literal data
# through packet.serializeStreamHeader's partialLengthWriter, which turns EVERY Write into power-of-two partial chunks.

def _new_packet(tag: int, body: bytes) -> bytes:
    n = len(body)
    if n < 192:
        ln = bytes([n])
    elif n < 8384:
        ln = bytes([((n - 192) >> 8) + 192, (n - 192) & 0xFF])
    else:
        ln = b"\xff" + struct.pack(">I", n)
    return bytes([0xC0 | tag]) + ln + body


def go_partial_write(data: bytes) -> bytes:
    """packet.partialLengthWriter.Write (x/crypto @53104e6ec876): the largest power of two that fits, repeatedly."""
    out, p = bytearray(), 0
    while p < len(data):
        for power in range(14, -1, -1):
            l = 1 << power
            if len(data) - p >= l:
                out.append(224 + power)
                out += data[p:p + l]
                p += l
                break
    return bytes(out)


def go_literal_packet(plain: bytes, file_name: bytes, binary: bool = True, time: int = 0) -> bytes:
    """packet.SerializeLiteral + Write(plain) + Close: four Writes (format+len, name, time, body), then a zero length."""
    body = go_partial_write(bytes([ord("b") if binary else ord("t"), len(file_name)])) + go_partial_write(file_name) + \
        go_partial_write(struct.pack(">I", time)) + go_partial_write(plain)
    return bytes([0xC0 | 11]) + body + b"\x00"


def one_pass_packet(sig_type: int, hash_id: int, pk_algo: int, key_id: int, is_last: int = 1) -> bytes:
    return _new_packet(4, bytes([3, sig_type, hash_id, pk_algo]) + struct.pack(">Q", key_id) + bytes([is_last]))


def go_signature_packet(k, key_id: int, hash_id: int, signed: bytes, ctime: int, sig_type: int = 0) -> bytes:
    """packet.Signature.Serialize after Sign: v4, hashed area = creation time + issuer (x/crypto puts both there)."""
    hashed = bytes([5, 2]) + struct.pack(">I", ctime) + bytes([9, 16]) + struct.pack(">Q", key_id)
    head = bytes([4, sig_type, 1, hash_id]) + struct.pack(">H", len(hashed)) + hashed
    d = hashlib.new(_HASHLIB[hash_id], signed + head + b"\x04\xff" + struct.pack(">I", len(head))).digest()
    return _new_packet(2, head + struct.pack(">H", 0) + d[:2] + _mpi(raw_rsa_sign(k, hash_id, d)))


def make_transport_message(k, key_id: int, plain: bytes, nonce: bytes, ctime: int = 0x5F000000, hash_id: int = 8) -> bytes:
    """The decrypted content of one bftkv transport message (Message.Encrypt, crypto_pgp.go:418-438)."""
    import base64
    return one_pass_packet(0, hash_id, 1, key_id) + go_literal_packet(plain, base64.b64encode(nonce)) + \
        go_signature_packet(k, key_id, hash_id, plain, ctime)


def make_read_answers(n_ops: int, n_replicas: int, seed: int = 0xBF7C0007, ss_signers: int = 11, p_ok=0.90, p_stale=0.05, p_bad=0.03,
                      mix=None, shuffle_arrival=True):
    """Configs 3 / 5 in the form Client.Read receives them: for every (operation, replica) the decrypted transport
    answer — one-pass signature, literal data (FileName = base64(nonce)), signature, as Message.Encrypt writes them —
    whose plain text is the replica's stored packet packet.Serialize(x, v, t, sig, ss): x 16 B, v 32 B, the writer's
    signature (one OpenPGP packet) and a collective signature of `ss_signers` packets (suff = 11 for n = 16), about
    4 kB per answer.  The transport signature covers the literal BODY only, so one signed template per (replica, current /
    stale) serves every operation and only the nonce in the FileName differs per answer; a corrupted answer has one bit
    of its signature MPI flipped; a missing one is flagged in pre_status.
    Returns dict(keyring, ids, op_off, peer_ids, msgs (list of bytes), nonces (N, 8), pre_status, expect_status, ts, value_len)."""
    import base64
    from oracle import packet_oracle as pk          # only MAKES inputs (byte layout of packet.Serialize), never verifies
    rng = np.random.default_rng(seed)
    R, M = n_replicas, n_ops
    keys = load_keys(R)
    blocks, kids = [], []
    for i, k in enumerate(keys):
        b, kid = pgp_public_key_block(k, _private_key(k), b"a%02d (http://localhost:57%02d) <a%02d@bftq.test>" % (i, i, i))
        blocks.append(b); kids.append(kid)
    x = bytes(range(16))
    vals = {0: (bytes(rng.integers(0, 256, 32, dtype=np.uint8)), 7), 1: (bytes(rng.integers(0, 256, 32, dtype=np.uint8)), 6)}
    templates = {}
    for kind, (v, t) in vals.items():
        tbs = tbs_packet(x, v, t)
        wsig = sig_packet_v4(keys[0], kids[0], 8, tbs, 0x5F000001)
        ss = b"".join(sig_packet_v4(keys[j % R], kids[j % R], 8, tbs, 0x5F000002) for j in range(ss_signers))
        plain = pk.serialize(x, v, t, pk.SignaturePacket(type=1, version=1, completed=False, data=wsig, cert=b""),
                             pk.SignaturePacket(type=1, version=1, completed=True, data=ss, cert=b""))
        for r in range(R):
            m = make_transport_message(keys[r], kids[r], plain, b"\x00" * 8)
            # the 12 FileName characters: an 8-byte and a 4-byte partial chunk right after the 2-byte literal header chunk
            p0 = 15 + 1 + 1 + 2 + 1                      # one-pass (15) | CB | E1 | 'b' len | E3
            assert m[15] == 0xCB and m[16] == 0xE1 and m[19] == 0xE3 and m[28] == 0xE2
            templates[(kind, r)] = (bytearray(m), p0, p0 + 9)
    N = M * R
    key_idx = np.tile(np.arange(R, dtype=np.uint32), M)
    if shuffle_arrival:
        key_idx = rng.permuted(key_idx.reshape(M, R), axis=1).reshape(N).astype(np.uint32)
    u = rng.random(N)
    if mix is None:
        pk_, ps, pb = p_ok, p_stale, p_bad
    else:
        cls = rng.choice(len(mix), size=M, p=[m[0] for m in mix])
        pk_ = np.repeat(np.array([m[1] for m in mix])[cls], R)
        ps = np.repeat(np.array([m[2] for m in mix])[cls], R)
        pb = np.repeat(np.array([m[3] for m in mix])[cls], R)
    kind = np.where(u < pk_, 0, np.where(u < pk_ + ps, 1, np.where(u < pk_ + ps + pb, 2, 3)))
    nonces = rng.integers(0, 256, (N, 8), dtype=np.uint8)
    flip = rng.integers(8, 200, N)
    msgs = []
    for i in range(N):
        tpl, a, b = templates[(1 if kind[i] == 1 else 0, int(key_idx[i]))]
        m = bytearray(tpl)
        n64 = base64.b64encode(nonces[i].tobytes())
        m[a:a + 8] = n64[:8]
        m[b:b + 4] = n64[8:]
        if kind[i] == 2:
            m[len(m) - int(flip[i])] ^= 0x10                      # inside the signature MPI
        msgs.append(bytes(m) if kind[i] != 3 else b"")
    pre = np.where(kind == 3, 6, 0).astype(np.uint8)
    expect = np.where(kind == 2, 1, pre).astype(np.uint8)
    ts = np.where(kind == 1, 6, 7).astype(np.uint64)
    op_off = (np.arange(M + 1, dtype=np.uint64) * R).astype(np.uint32)
    return {"keyring": b"".join(blocks), "ids": kids, "op_off": op_off, "peer_ids": np.array(kids, np.uint64)[key_idx], "msgs": msgs,
            "nonces": nonces, "pre_status": pre, "expect_status": expect, "ts": ts, "value_id": np.where(kind == 1, 1, 0).astype(np.uint32),
            "key_idx": key_idx}
