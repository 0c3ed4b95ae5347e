"""Every literal-data framing the read path's message parser (K0m, msg_parse.cuh) admits, against the oracle.

A v4 binary signature covers the literal BODY and the signature's hashed area, not the literal packet's framing, format
byte, FileName or date, so one signed (body, signature) pair can be re-framed in many ways without re-signing: one-pass
packet in new or old format, the literal as one definite run (1-, 2-, 5-byte or old-format lengths) or as partial-length
chunks split anywhere, FileNames of every nonce length with CR / LF anywhere.  Whatever framing the sender chose,
Client.Read must reach the same status, t and value.  The CPU half checks the generator below against the oracle
(pgp_oracle.read_response_status); the GPU half sends every framing class through bftq_read_responses_batch, one call per
class, and asserts from engine.stats() which of K0m and the host packer decided it — a K0m that flagged everything would
still answer correctly through the host packer and go unnoticed otherwise."""
import base64
import json
import os
import random
import struct
from dataclasses import dataclass, field
from typing import Dict, List, Tuple

import numpy as np
import pytest

from bftkv_b200 import workload
from oracle import packet_oracle, pgp_oracle as pgp, wotqs_oracle as wq
from oracle.wotqs_oracle import Node

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 10                                  # keys 0..9 are in the keyring and the quorum, key R signs as an outsider
NONCE8 = bytes.fromhex("9c0e5a7731f2b4d8")
BODY_LENS = list(range(201)) + [255, 256, 1000, 5000, 17000]
GOOD = (pgp.ST_OK, pgp.ST_UNVERIFIED)
READ_PIECE = 16384                      # bftq_read_responses_batch's default piece: K0m is launched per piece


# ---- the generator: (body, signature packet, FileName, framing) -> the decrypted transport message ----------------------

def new_len(form: str, n: int) -> bytes:
    """New-format length octets (RFC 4880 §4.2.2): 'p' partial (n a power of two), '1' / '2' / '5' definite."""
    if form == "p":
        assert n > 0 and n & (n - 1) == 0 and n <= 1 << 30
        return bytes([224 + n.bit_length() - 1])
    if form == "1":
        assert n < 192
        return bytes([n])
    if form == "2":
        assert 192 <= n <= 8383
        return bytes([192 + ((n - 192) >> 8), (n - 192) & 0xFF])
    assert form == "5"
    return b"\xff" + struct.pack(">I", n)


def pow2_runs(n: int) -> List[Tuple[str, int]]:
    """x/crypto's partialLengthWriter on one Write of n bytes: the largest power of two (<= 2^14) that fits, repeatedly."""
    out = []
    while n:
        e = min(14, n.bit_length() - 1)
        out.append(("p", 1 << e))
        n -= 1 << e
    return out


def lit_new(chunks):
    """A new-format (0xCB) literal written as the given (form, length) runs; the lengths must add up to the content."""
    def make(content: bytes, name_len: int) -> bytes:
        runs = chunks(len(content), name_len) if callable(chunks) else chunks
        out, p = bytearray(b"\xcb"), 0
        for form, n in runs:
            out += new_len(form, n) + content[p:p + n]
            p += n
        assert p == len(content), (p, len(content))
        return bytes(out)
    return make


def lit_old(lt: int):
    """An old-format literal 0xAC / 0xAD / 0xAE (1-, 2-, 4-byte length) or 0xAF (indeterminate: runs to the end)."""
    def make(content: bytes, name_len: int) -> bytes:
        if lt == 3:
            return b"\xaf" + content
        return bytes([0xAC | lt]) + len(content).to_bytes(1 << lt, "big") + content
    return make


def go_runs(total: int, name_len: int):
    """Go's framing: four Writes (format + name length, name, date, body), each in power-of-two chunks, then a zero length."""
    return pow2_runs(2) + pow2_runs(name_len) + pow2_runs(4) + pow2_runs(total - 6 - name_len) + [("1", 0)]


LIT_GO = lit_new(go_runs)


def def_form(n: int, form: str) -> bool:
    return {"1": n < 192, "2": 192 <= n <= 8383, "5": True}[form]


def one_pass(key_id: int, form: str = "C4", hash_id: int = 8) -> bytes:
    """A one-pass signature packet (v3, binary, RSA, last) with the given header."""
    body = bytes([3, 0, hash_id, 1]) + struct.pack(">Q", key_id) + b"\x01"
    return {"C4": b"\xc4\x0d", "90": b"\x90\x0d", "C4-5": b"\xc4\xff\x00\x00\x00\x0d", "91": b"\x91\x00\x0d",
            "92": b"\x92\x00\x00\x00\x0d"}[form] + body


def body_of_len(n: int) -> bytes:
    """A literal body of exactly n bytes: packet.Serialize(x, v, t) when n allows one, else a cut of one (which
    packet.Parse may reject: the signature still has to verify first)."""
    if n >= 25:
        v = bytes((i * 37 + n) & 0xFF for i in range(n - 25))
        return packet_oracle.serialize(b"x", v, n + 1)
    return packet_oracle.serialize(b"x", b"", n + 1)[:n]


@dataclass
class Ctx:
    keys: list
    kids: list
    ring: bytes
    ents: list
    qcs: list
    quorum: object
    sigs: Dict[tuple, bytes] = field(default_factory=dict)
    memo_status: Dict[tuple, tuple] = field(default_factory=dict)
    memo_plain: Dict[bytes, bytes] = field(default_factory=dict)

    def sig(self, body: bytes, signer: int, hash_id: int = 8) -> bytes:
        k = (body, signer, hash_id)
        if k not in self.sigs:
            self.sigs[k] = workload.go_signature_packet(self.keys[signer], self.kids[signer], hash_id, body, 0x5F000000 + signer)
        return self.sigs[k]

    def message(self, body: bytes, signer: int = 0, name: bytes = None, nonce: bytes = NONCE8, lit=LIT_GO, op: str = "C4",
                fmt: bytes = b"b", date: int = 0, hash_id: int = 8, between: bytes = b"", tail: bytes = b"", sig: bytes = None) -> bytes:
        name = base64.b64encode(nonce) if name is None else name
        content = fmt + bytes([len(name)]) + name + struct.pack(">I", date) + body
        sig = self.sig(body, signer, hash_id) if sig is None else sig
        return one_pass(self.kids[signer], op, hash_id) + lit(content, len(name)) + between + sig + tail

    def oracle(self, msg: bytes, nonce: bytes, pre: int = 0):
        """(status class, t, value, plain) as Client.Read sees the answer; memoised, many answers share their bytes."""
        k = (msg, nonce, pre)
        if k not in self.memo_status:
            st, t, v = pgp.read_response_status(self.ents, msg, nonce, pre)
            plain = None
            if st in GOOD:
                if msg not in self.memo_plain:
                    self.memo_plain[msg] = pgp.message_verify(self.ents, msg).plain
                plain = self.memo_plain[msg]
            self.memo_status[k] = (st, t, v, plain)
        return self.memo_status[k]


@pytest.fixture(scope="module")
def ctx():
    keys = workload.load_keys(R + 1)
    blocks, kids = [], []
    for i, k in enumerate(keys):
        b, kid = workload.pgp_public_key_block(k, workload._private_key(k), b"f%02d (http://localhost:58%02d) <f%02d@x>" % (i, i, i))
        blocks.append(b); kids.append(kid)
    ring = b"".join(blocks[:R])
    return Ctx(keys, kids, ring, pgp.read_entities(ring), [(3, 10, 4, 7, kids[:R])],
               wq.Quorum([wq.QC([Node(i) for i in kids[:R]], 3, 10, 4, 7)]))


@dataclass
class Answer:
    msg: bytes
    nonce: bytes
    want: object          # (status class, t, value) of the Go-framed original, or a status class


@dataclass
class Family:
    name: str
    on_gpu: bool          # True: K0m's shape check admits every answer; False: it must flag every one to the host packer
    nonce_len: int
    answers: List[Answer]


def original(c: Ctx, body: bytes, signer: int = 0, nonce: bytes = NONCE8):
    """What every accepted re-framing must reproduce: the oracle's (status, t, value) of the Go-framed message."""
    return c.oracle(c.message(body, signer, nonce=nonce), nonce)[:3]


def families(c: Ctx) -> List[Family]:
    rng = random.Random(0xF4A3)
    F: Dict[str, Family] = {}

    def add(name, on_gpu, msg, want, nonce=NONCE8):
        F.setdefault(name, Family(name, on_gpu, len(nonce), [])).answers.append(Answer(msg, nonce, want))

    # ---- body lengths: every residue mod 64 and the SHA-256 padding edges, in every framing that can carry them
    for n in BODY_LENS:
        body, s = body_of_len(n), n % R
        want = original(c, body, s)
        total = 2 + 12 + 4 + n                                      # format, name length, 12-character name, date, body
        add("partial: Go", True, c.message(body, s), want)
        for form in "125":
            if def_form(total, form):
                add("new definite %s-byte" % form, True, c.message(body, s, lit=lit_new([(form, total)])), want)
        for lt, cap in ((0, 255), (1, 65535), (2, 1 << 32)):
            if total <= cap:
                add("old %02X" % (0xAC | lt), True, c.message(body, s, lit=lit_old(lt)), want)
        if n <= 1000:
            add("partial: one byte per chunk", True, c.message(body, s, lit=lit_new([("p", 1)] * total + [("1", 0)])), want)
        runs, left = [], total
        while left and rng.random() < 0.9:
            e = rng.randrange(min(14, left.bit_length() - 1) + 1)
            runs.append(("p", 1 << e)); left -= 1 << e
        runs.append((rng.choice([f for f in "125" if def_form(left, f)]), left))
        add("partial: random powers of two", True, c.message(body, s, lit=lit_new(runs), date=rng.getrandbits(32)), want)
        if n >= 200:                                                 # final chunk of a partial sequence in every form
            for form, r in (("1", 0), ("1", 1), ("1", 191), ("2", 192), ("2", min(n, 8383)), ("5", 0), ("5", 17), ("5", n)):
                add("partial: final chunk %s-byte" % form, True, c.message(body, s, lit=lit_new(pow2_runs(total - r) + [(form, r)])), want)

    body = body_of_len(130)
    want = original(c, body)
    total = 18 + len(body)
    for cut in range(1, 20):                                         # a boundary at every byte of the literal header
        add("partial: header split", True, c.message(body, lit=lit_new(pow2_runs(cut) + pow2_runs(total - cut) + [("1", 0)])), want)
    for fmt in (b"t", b"u", b"\x00", b"\xff"):
        add("literal format byte / date", True, c.message(body, fmt=fmt, date=0xFFFFFFFF), want)

    # ---- one-pass packet headers
    for n in (0, 25, 100, 300):
        b = body_of_len(n)
        w = original(c, b)
        add("one-pass C4 0D", True, c.message(b, op="C4"), w)
        add("one-pass 90 0D", True, c.message(b, op="90"), w)
        add("one-pass 90 0D", True, c.message(b, op="90", lit=lit_old(1)), w)
        for op in ("C4-5", "91", "92"):                               # the same packet under longer length forms: flagged
            add("one-pass, other length forms", False, c.message(b, op=op), w)
        add("one-pass SHA-512", False, c.message(b, hash_id=10), w)

    # ---- old-format indeterminate length: the literal runs to the end and swallows the signature packet
    for n in (25, 100):
        add("old AF", False, c.message(body_of_len(n), lit=lit_old(3)), pgp.ST_INVALID)
    # ---- a 5-byte definite length in the middle of a partial sequence ends the literal there: the rest is not a signature
    add("partial: definite run mid-sequence", False, c.message(body, lit=lit_new(pow2_runs(64) + [("5", 40)] + pow2_runs(total - 104) + [("1", 0)])),
        pgp.ST_INVALID)
    add("partial: definite run mid-sequence", False, c.message(body, lit=lit_new([("p", 16), ("1", 2)] + pow2_runs(total - 18) + [("1", 0)])),
        pgp.ST_INVALID)

    # ---- FileName: every nonce length (one call each: nonce_len is per call), CR / LF anywhere, base64 corner cases
    for nl in (1, 2, 3, 8, 23, 24):
        nonce = bytes(rng.randrange(256) for _ in range(nl))
        other = bytes(rng.randrange(256) for _ in range(nl))
        resized = bytes(rng.randrange(256) for _ in range(nl + 1 if nl < 24 else nl - 1))
        w = original(c, body, nonce=nonce)
        assert w[0] == pgp.ST_OK
        add("FileName, nonce %d bytes" % nl, True, c.message(body, nonce=nonce), w, nonce)
        add("FileName, nonce %d bytes" % nl, True, c.message(body, nonce=other), pgp.ST_NONCE, nonce)
        add("FileName, nonce %d bytes" % nl, True, c.message(body, nonce=resized), pgp.ST_NONCE, nonce)
        add("FileName, nonce %d bytes" % nl, True, c.message(body, name=b""), pgp.ST_NONCE, nonce)
        name = base64.b64encode(nonce)
        if len(name) + 1 <= 32:
            for p in range(len(name) + 1):
                for ins in (b"\r", b"\n", b"\r\n"):
                    if len(name) + len(ins) <= 32:
                        add("FileName, nonce %d bytes" % nl, True, c.message(body, name=name[:p] + ins + name[p:]), w, nonce)
        pad = (b"\r\n" * 17)[:33 - len(name)]                        # 33 bytes: one past K0m's FileName limit
        add("FileName of 33 bytes, nonce %d bytes" % nl, False, c.message(body, name=name + pad), w, nonce)
        add("FileName of 33 bytes, nonce %d bytes" % nl, False, c.message(body, name=pad + name), w, nonce)
    nonce1 = b"A"                                                    # base64 "QQ=="
    w1 = original(c, body, nonce=nonce1)
    for name in (b"QR==", b"QX==", b"Q\nQ=\r\n=\n"):                   # trailing bits are not checked; CR / LF between the two '='
        add("FileName, nonce 1 bytes", True, c.message(body, name=name), w1, nonce1)
    for name in (b"QQ=", b"QQ=\n", b"QQ=A", b"QQ=\n\rA", b"Q===", b"=QQQ", b"Q=", b"QQ", b"Q", b"QUJ", b"QQ==QQ==", b"QQ==A",
                 b"QQ==\nA", b"QQ==\x00", b"QQ-=", b"QQ_=", b"Q Q==", b"QQ.=", b"QQ==" + b"=", b"Q\x80==", b"QUJD=", b"QUJDRA"):
        add("FileName, base64 errors", True, c.message(body, name=name), pgp.ST_OTHER, nonce1)
    nonce2 = b"AB"                                                   # base64 "QUI="
    w2 = original(c, body, nonce=nonce2)
    for name in (b"QUI=", b"QUJ=", b"QUI=\r\n", b"\nQUI=", b"Q\rU\nI=", b"QUI\n="):
        add("FileName, nonce 2 bytes", True, c.message(body, name=name), w2, nonce2)
    for name in (b"QUI==", b"QUI=QUI=", b"QUI=\nx", b"QU=I", b"QUI"):
        add("FileName, base64 errors (nonce 2 bytes)", True, c.message(body, name=name), pgp.ST_OTHER, nonce2)

    # ---- what follows the literal data
    unknown_pkt = b"\xfc\x03xyz"                                     # tag 60: skipped by packets.Next()
    marker = b"\xca\x03PGP"
    for s in (0, R):
        w = original(c, body, s)
        add("trailing data", False, c.message(body, s, tail=b"\x00"), w)
        add("trailing data", False, c.message(body, s, tail=marker), w)
        add("trailing data", False, c.message(body, s, tail=c.sig(body, (s + 1) % (R + 1))), w)
        add("trailing data", False, c.message(body, s, between=unknown_pkt), w)
        add("trailing data", False, c.message(body, s, between=unknown_pkt + unknown_pkt), w)

    # ---- signer: known, outsider (accepted unverified), one bit of the signature MPI or of its hash tag flipped
    for n in (0, 63, 64, 100, 300, 1000):
        b = body_of_len(n)
        add("signer outside the keyring", True, c.message(b, R), original(c, b, R))
        sig = c.sig(b, 1)
        for pos in (1, 2, 17, 100, 255):
            bad = bytearray(sig)
            bad[-pos] ^= 1 << (pos % 8)
            add("signature bit flipped", True, c.message(b, 1, sig=bytes(bad)), pgp.ST_INVALID)
        bad = bytearray(sig)
        bad[-259] ^= 0x01                                            # the two hash-tag bytes sit right before the MPI
        add("signature bit flipped", True, c.message(b, 1, sig=bytes(bad)), pgp.ST_INVALID)

    # ---- truncation at every byte of the last chunk and into the signature; lengths that claim more than remains
    for n, s in ((100, 2), (100, R), (300, 3)):
        b = body_of_len(n)
        m = c.message(b, s)
        w = original(c, b, s)
        op_len, lit_len = 15, len(LIT_GO(b"b\x0c" + base64.b64encode(NONCE8) + bytes(4) + b, 12))
        last = pow2_runs(n)[-1][1]
        lit_end = op_len + lit_len
        for cut in list(range(lit_end - 2 - last, lit_end)) + [lit_end, lit_end + 1, lit_end + 3, lit_end + 100, len(m) - 1]:
            want = pgp.ST_OTHER if cut < lit_end else (pgp.ST_INVALID if s < R else w)
            add("truncated", False, m[:cut], want)
    b = body_of_len(100)
    total = 18 + len(b)
    for head in (b"\xcb" + new_len("5", 0xFFFFFFFF), b"\xcb" + new_len("5", total + 400), b"\xcb" + new_len("2", 8383),
                 b"\xae" + struct.pack(">I", 0xFFFFFF00), b"\xad\xff\xff"):
        add("length octets past the end", False, c.message(b, lit=lambda content, nl, head=head: head + content), pgp.ST_OTHER)
    add("length octets past the end", False,
        c.message(b, lit=lambda content, nl: b"\xcb" + new_len("p", 64) + content[:64] + new_len("p", 1 << 30) + content[64:]), pgp.ST_OTHER)
    return list(F.values())


def status_class(st):
    return {0: pgp.ST_OK, 8: pgp.ST_UNVERIFIED, 7: pgp.ST_NONCE, 1: pgp.ST_INVALID, 2: pgp.ST_INVALID}.get(int(st), pgp.ST_OTHER)


def check_want(c: Ctx, a: Answer, ctx_name):
    st, t, v, _ = c.oracle(a.msg, a.nonce)
    if isinstance(a.want, tuple):
        assert (st, t, v) == a.want, (ctx_name, a.msg.hex())
    else:
        assert st == a.want, (ctx_name, st, a.msg.hex())


# ---- CPU half: the generator against the oracle -----------------------------------------------------------------------

def test_go_framing_is_the_writer_of_the_workload(ctx):
    """The generator's Go framing is byte for byte what workload.make_transport_message writes."""
    for n in (0, 1, 100, 5000):
        body = body_of_len(n)
        assert ctx.message(body, 3) == workload.make_transport_message(ctx.keys[3], ctx.kids[3], body, NONCE8, ctime=0x5F000003)
    assert lit_new([("p", 2), ("p", 1), ("5", 1)])(b"1234", 0) == b"\xcb\xe112\xe03\xff\x00\x00\x00\x014"
    assert lit_old(1)(b"1234", 0) == b"\xad\x00\x041234" and lit_old(3)(b"1234", 0) == b"\xaf1234"
    with pytest.raises(AssertionError):
        lit_new([("1", 3)])(b"1234", 0)                              # runs that do not cover the content are refused


def test_reframings_against_the_oracle(ctx):
    fams = families(ctx)
    seen = set()
    for f in fams:
        assert f.answers, f.name
        for a in f.answers:
            check_want(ctx, a, f.name)
            seen.add(a.want if isinstance(a.want, int) else a.want[0])
    assert seen == {pgp.ST_OK, pgp.ST_UNVERIFIED, pgp.ST_INVALID, pgp.ST_NONCE, pgp.ST_OTHER}, seen
    # the valid packets among the bodies read back as written, whatever their framing
    for n in BODY_LENS:
        st, t, v = original(ctx, body_of_len(n), n % R)
        if n >= 25:
            assert (st, t, len(v)) == (pgp.ST_OK, n + 1, n - 25), n


def test_gnupg_fixtures_oracle_agrees_with_gnupg():
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_messages.json")))
    ents = pgp.read_entities(bytes.fromhex(g["keyring"]))
    nonce = bytes.fromhex(g["nonce"])
    for c in g["cases"]:
        st, _, _ = pgp.read_response_status(ents, bytes.fromhex(c["msg"]), nonce)
        if c["signer"] == "m01" and c["name"] not in ("compressed-default", "name-not-base64"):
            assert (st != pgp.ST_INVALID) == c["gpg_good"], (c["name"], st)


# ---- GPU half: K0m (and the host packer for what it flags) against the oracle -----------------------------------------

@dataclass
class Call:
    """One bftq_read_responses_batch call: operations of (message, nonce, pre_status, peer id) answers."""
    nonce_len: int
    ops: List[list] = field(default_factory=list)
    offset: int = 0
    fillers: int = 0

    def filler_to(self, align: int):
        """A failed 1-3 byte answer in an operation of its own, so that the next answer starts at `align` mod 4."""
        pad = (align - self.offset) % 4
        if pad:
            self.ops.append([(b"\x00" * pad, bytes(self.nonce_len), 6, 0)])
            self.offset += pad
            self.fillers += 1

    def op(self, answers):
        self.ops.append(answers)
        self.offset += sum(len(a[0]) for a in answers)


def run_call(kr, c: Ctx, call: Call):
    """Runs the call and compares every status, t, value and decision with the oracle.
    Returns (answers K0m decided, answers the host packer decided, the call's status bytes)."""
    from bftkv_b200.crypto_gpu import read_responses_batch
    op_off, msgs, nonces, pre, peers = [0], [], [], [], []
    for op in call.ops:
        for m, n, p, peer in op:
            assert len(n) == call.nonce_len
            msgs.append(m); nonces.append(n); pre.append(p); peers.append(peer)
        op_off.append(len(msgs))
    s0 = kr.engine.stats()
    got = read_responses_batch(kr, c.qcs, np.array(op_off, np.uint32), np.array(peers, np.uint64), msgs,
                               np.frombuffer(b"".join(nonces), np.uint8).reshape(-1, call.nonce_len), pre_status=np.array(pre, np.uint8))
    s1 = kr.engine.stats()
    for i, (m, n, p) in enumerate(zip(msgs, nonces, pre)):
        st, t, v, plain = c.oracle(m, n, p)
        assert status_class(got["status"][i]) == st, (i, int(got["status"][i]), st, m.hex())
        if st in GOOD:
            vo, vl = int(got["value_off"][i]), int(got["value_len"][i])
            assert int(got["ts"][i]) == t and vl == len(v) and plain[vo:vo + vl] == v, (i, m.hex())
    for k in range(len(call.ops)):
        resp = []
        for i in range(op_off[k], op_off[k + 1]):
            st, t, v, _ = c.oracle(msgs[i], nonces[i], pre[i])
            resp.append((Node(peers[i]), st not in GOOD, t, v))
        kind, at, value, t = wq.read_decide(resp, c.quorum)
        assert (int(got["decision"][k]), int(got["decided_at"][k])) == (kind, at), (k, kind, at)
        if kind == wq.READ_VALUE:
            w = int(got["winner"][k])
            assert resp[w][2] == t and resp[w][3] == value and not resp[w][1], k
            assert not any(not r[1] and r[2] == t and r[3] == value for r in resp[:w]), k
        else:
            assert int(got["winner"][k]) == 0xFFFFFFFF, k
    return s1["msg_gpu_items"] - s0["msg_gpu_items"], s1["msg_host_items"] - s0["msg_host_items"], got["status"]


def aligned(call: Call, answers: List[Answer], reps: int = 4):
    """Every answer `reps` times, copy r at offset (index + r) mod 4 from the start of the call: every framing at every
    alignment of K0m's word loads."""
    for r in range(reps):
        for i, a in enumerate(answers):
            call.filler_to((i + r) % 4)
            call.op([(a.msg, a.nonce, 0, 0)])


@pytest.fixture(scope="module")
def kr(ctx, engine):
    from bftkv_b200.crypto_gpu import Keyring
    k = Keyring(engine)
    k.register(ctx.ring)
    yield k
    k.close()


@pytest.mark.gpu
def test_gnupg_fixtures_through_k0m(engine):
    from bftkv_b200.crypto_gpu import Keyring
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "golden_messages.json")))
    ring = bytes.fromhex(g["keyring"])
    c = Ctx([], [], ring, pgp.read_entities(ring), [(0, 1, 1, 1, [1])], wq.Quorum([wq.QC([Node(1)], 0, 1, 1, 1)]))
    k = Keyring(engine)
    k.register(ring)
    nonce = bytes.fromhex(g["nonce"])
    call = Call(len(nonce))
    for r in range(4):
        for i, case in enumerate(g["cases"]):
            call.filler_to((i + r) % 4)
            call.op([(bytes.fromhex(case["msg"]), nonce, 0, 1)])
    on_gpu, on_host, status = run_call(k, c, call)
    k.close()
    assert on_gpu + on_host == 4 * len(g["cases"]) + call.fillers and on_gpu > call.fillers, (on_gpu, on_host)
    by_msg = {bytes.fromhex(case["msg"]): case for case in g["cases"]}
    answers = [a for op in call.ops for a in op]
    assert len(answers) == len(status)
    for (m, _, pre, _), st in zip(answers, status):                  # GnuPG's own verdict on the signature
        case = by_msg.get(m) if pre == 0 else None
        if case and case["signer"] == "m01" and case["name"] not in ("compressed-default", "name-not-base64"):
            assert (status_class(st) != pgp.ST_INVALID) == case["gpg_good"], case["name"]


@pytest.mark.gpu
def test_every_framing_class_through_k0m(ctx, kr):
    """One call per framing class, every answer at all four alignments; K0m must decide exactly the classes its shape
    check admits and flag exactly the others."""
    table = []
    for f in families(ctx):
        call = Call(f.nonce_len)
        aligned(call, f.answers)
        on_gpu, on_host, _ = run_call(kr, ctx, call)
        n = 4 * len(f.answers)
        table.append((f.name, on_gpu - call.fillers, on_host))
        if f.on_gpu:
            assert (on_gpu, on_host) == (n + call.fillers, 0), (f.name, on_gpu, on_host, n, call.fillers)
        else:
            assert (on_gpu, on_host) == (call.fillers, n), (f.name, on_gpu, on_host, n, call.fillers)
    print("\nanswers decided per framing class (each answer at 4 alignments):  K0m / host")
    for name, g, h in table:
        print("  %-45s %6d / %d" % (name, g, h))


@pytest.mark.gpu
def test_two_pieces_in_one_call(ctx, kr):
    """More than one piece of answers in one call, the second piece starting at an offset that is not a multiple of 4."""
    fams = [f for f in families(ctx) if f.nonce_len == 8]
    want_gpu = want_host = 0
    call = Call(8)
    reps = 0
    while len([a for op in call.ops for a in op]) <= READ_PIECE + 2000:
        for f in fams:
            for i, a in enumerate(f.answers):
                call.filler_to((i + reps) % 4)
                call.op([(a.msg, a.nonce, 0, 0)])
                want_gpu += f.on_gpu
                want_host += not f.on_gpu
        reps += 1
    flat = [a for op in call.ops for a in op]
    while sum(len(a[0]) for a in flat[:READ_PIECE]) % 4 == 0:          # the second piece must start off a word boundary
        call.ops.insert(0, [(b"\x00", bytes(8), 6, 0)])
        call.fillers += 1
        flat.insert(0, call.ops[0][0])
    on_gpu, on_host, _ = run_call(kr, ctx, call)
    assert (on_gpu, on_host) == (want_gpu + call.fillers, want_host), (on_gpu, on_host, want_gpu, want_host, call.fillers)


@pytest.mark.gpu
def test_grouping_across_framings(ctx, kr):
    """Operations of ten responders that carry one value under different framings — some decided by K0m, some by the
    host packer — must land in one bucket; values that differ in one byte next to a chunk or hash-block boundary must not."""
    rng = random.Random(0x6A0)
    # value at body offset 17; Go's chunks and SHA-256 blocks of the body both break at body offsets 64, 128, 256
    bases = {100: (46, 47), 300: (111, 238, 239), 47: (46,)}
    bodies = {}
    for vlen, flips in bases.items():
        v = bytes((i * 11 + vlen) & 0xFF for i in range(vlen))
        bodies[vlen] = (packet_oracle.serialize(b"x", v, 9), [packet_oracle.serialize(b"x", v[:j] + bytes([v[j] ^ 0x01]) + v[j + 1:], 9) for j in flips])
    empty = packet_oracle.serialize(b"x", b"", 9)

    def framed(body, s):
        """-> (message, decided by K0m?)"""
        total = 18 + len(body)
        k = rng.randrange(12)
        if k == 0:
            return ctx.message(body, s), True
        if k == 1:
            return ctx.message(body, s, lit=lit_new([("p", 1)] * total + [("1", 0)])), True
        if k == 2:
            return ctx.message(body, s, lit=lit_new([("5", total)]), op="90"), True
        if k == 3:
            return ctx.message(body, s, lit=lit_old(rng.choice([1, 2]))), True
        if k == 4:
            cut = rng.randrange(1, total)
            return ctx.message(body, s, lit=lit_new(pow2_runs(cut) + pow2_runs(total - cut) + [("1", 0)])), True
        if k == 5:
            name = base64.b64encode(NONCE8)
            p = rng.randrange(len(name))
            return ctx.message(body, s, name=name[:p] + b"\r\n" + name[p:], lit=lit_new([("2", total + 2)] if total + 2 >= 192 else [("1", total + 2)])), True
        if k == 6:
            return ctx.message(body, s, name=base64.b64encode(NONCE8) + b"\n" * 21), False          # 33-byte FileName
        if k == 7:
            return ctx.message(body, s, hash_id=10), False                                          # SHA-512
        if k == 8:
            return ctx.message(body, s, between=b"\xfc\x01z"), False
        if k == 9:
            return ctx.message(body, s, op="91"), False
        if k == 10:
            return ctx.message(body, s, tail=b"\x00\x00"), False
        return ctx.message(body, s, lit=lit_new(pow2_runs(total - 5) + [("5", 5)])), True

    call = Call(8)
    want_gpu = want_host = 0
    for op in range(160):
        base, variants = bodies[rng.choice(list(bodies))] if op % 8 else (empty, [empty])
        order = list(range(R))
        rng.shuffle(order)
        if op % 2:
            alt = rng.choice(variants)
            chosen = [base if j % 2 else alt for j in range(R)]       # alternating: `alt` reaches the threshold (4) at answer 7
        else:
            chosen = [base] * R
        answers = []
        for j, s in enumerate(order):
            m, g = framed(chosen[j], s)
            want_gpu += g
            want_host += not g
            answers.append((m, NONCE8, 0, ctx.kids[s]))
        call.filler_to(rng.randrange(4))
        call.op(answers)
        # what run_call compares against: one bucket decides at the 4th answer, two buckets at the 7th
        resp = [(Node(peer), ctx.oracle(m, n)[0] not in GOOD, *ctx.oracle(m, n)[1:3]) for m, n, _, peer in answers]
        assert wq.read_decide(resp, ctx.quorum)[:2] == (wq.READ_VALUE, 7 if op % 2 else 4), op
    on_gpu, on_host, _ = run_call(kr, ctx, call)
    assert (on_gpu, on_host) == (want_gpu + call.fillers, want_host), (on_gpu, on_host, want_gpu, want_host)
