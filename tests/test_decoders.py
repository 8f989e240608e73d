"""N1 -- the databits decoders (minimodem_b200/csrc/fsk_b200_decode_core.h), CPU side.

The decoder source is compiled twice: into the k_decode kernels and, for these tests, into
liboracle.so (oracle/decode_oracle.c).  Here the host build is held against
  * the UNMODIFIED reference decoders (oracle/_ref/libfsk_ref.so: src/databits_*.c, src/baudot.c,
    src/uic_codes.c) on random and crafted word sequences, byte for byte, and
  * the stdout of the unmodified reference CLI on its own test invocations (tests/golden/),
    through the frame records of the rx-loop restatement.
The kernels are held against the host build in test_gpu_parity.py."""
import ctypes as C
import os
import shutil
import zlib

import numpy as np
import pytest

import golden_util as gu
import orc
import refcases


# --------------------------------------------------------------------------
# a private instance of the reference library: its decoders keep file-static state
# (src/baudot.c:197, src/databits_callerid.c:45-47), and these tests must see all of its history
# --------------------------------------------------------------------------
_priv = None


def private_ref(tmp_path_factory):
    """lib: the private copy, or None where oracle/_ref is not built (the decoders' recorded answers stand in)."""
    global _priv
    if _priv is None:
        L = None
        if orc.have_ref():
            d = tmp_path_factory.mktemp("refcopy")
            path = os.path.join(str(d), "libfsk_ref_private.so")
            shutil.copy(orc.LIBREF, path)
            L = C.CDLL(path)
        _priv = dict(lib=L, state=orc.DecoderState())      # our state with the same history
    return _priv


@pytest.mark.parametrize("kind,nbits", [("ascii8", 8), ("ascii8", 7), ("binary", 8), ("binary", 5), ("binary", 39),
                                        ("baudot", 5), ("uic-ground", 39), ("uic-train", 39)])
def test_words_against_reference_decoders(kind, nbits, tmp_path_factory):
    P = private_ref(tmp_path_factory)
    rng = np.random.default_rng(zlib.crc32(("%s/%d" % (kind, nbits)).encode()))
    n = 4000
    words = rng.integers(0, 1 << nbits, n, dtype=np.uint64)
    if kind == "baudot":
        # plenty of shifts and spaces
        words[::7] = 0x1B
        words[3::11] = 0x1F
        words[5::13] = 0x04
    if kind.startswith("uic"):
        codes = np.array([0x00, 0x02, 0x03, 0x04, 0x06, 0x08, 0x09, 0x0A, 0x0C, 0x55, 0x7F, 0xFF], np.uint64)
        # message byte sits bit-reversed in bits 24..31
        rev = np.array([int("{:08b}".format(int(c))[::-1], 2) for c in codes], np.uint64)
        pick = rng.integers(0, len(codes), n)
        words = (words & np.uint64(~(0xFF << 24) & ((1 << 39) - 1))) | (rev[pick] << np.uint64(24))
    resets = rng.random(n) < 0.02
    resets[0] = True
    st = P["state"]
    got = orc.decode_words(kind, nbits, words, resets, state=st)
    want = orc.ref_decode_words(kind, nbits, words, resets, L=P["lib"])
    assert got == want


def _mdmf(fields):
    body = b"".join(bytes([t, len(d)]) + d for t, d in fields)
    msg = bytes([0x80, len(body)]) + body
    return msg + bytes([(-sum(msg)) & 0xFF])


def _sdmf(date, number):
    body = date + number
    msg = bytes([0x04, len(body)]) + body
    return msg + bytes([(-sum(msg)) & 0xFF])


CRAFTED = [
    _mdmf([(1, b"03151045"), (2, b"8005551212"), (7, b"JOHN DOE")]),
    _mdmf([(1, b"12312359"), (4, b"P"), (8, b"O")]),
    _mdmf([(2, b"5551212"), (7, b"")]),                         # phone not 10 digits: printed plain
    _mdmf([(4, b"X"), (8, b"PP"), (3, b"abc"), (5, b""), (6, b"zz"), (0, b"q")]),   # unknown types, odd N/A
    _mdmf([(1, b"0315"), (7, b"A\x00B")]),                      # short date, NUL inside a field
    _mdmf([(7, b"OK"), (9, b"bad"), (7, b"never")]),            # bad type: the message's fields are dropped
    _mdmf([(7, b"x" * 40), (2, b"1234567890")]),
    _sdmf(b"03151045", b"8005551212"),
    _sdmf(b"03151045", b"5551212"),
    _sdmf(b"0315", b""),                                        # msglen < 8: the length wraps (no limit)
    bytes([0x80, 0x00]),                                         # empty MDMF completes at once
    bytes([0x04, 0x00]),
    b"\x11\x22\x80\x03\x07\x01Z\x55" + b"\x04\x12" + b"010203041234567890" + b"\x00",
]


def test_callerid_against_reference_decoder(tmp_path_factory):
    P = private_ref(tmp_path_factory)
    rng = np.random.default_rng(7)
    stream = bytearray()
    for m in CRAFTED:
        stream += m
        stream += bytes(rng.integers(0, 256, int(rng.integers(0, 4)), dtype=np.uint8))
    # random traffic: message starts are frequent, lengths stay below 200 so that the reference
    # never reads past its 256-byte array, zeros are frequent so that unbounded prints terminate
    for _ in range(400):
        t = int(rng.choice([0x80, 0x04]))
        ln = int(rng.integers(0, 200))
        body = rng.integers(0, 256, ln, dtype=np.uint8)
        body[rng.random(ln) < 0.15] = 0
        if t == 0x80 and ln >= 2 and rng.random() < 0.8:
            # plausible field headers
            i = 0
            while i + 2 <= ln:
                body[i] = int(rng.choice([0, 1, 2, 3, 4, 5, 6, 7, 8, 8, 7, 2, 1, 9]))
                fl = int(min(rng.integers(0, 16), ln - i - 2))
                body[i + 1] = fl
                i += 2 + fl
        stream += bytes([t, ln]) + bytes(body) + bytes([int(rng.integers(0, 256))])
    words = np.frombuffer(bytes(stream), np.uint8).astype(np.uint64)
    resets = rng.random(words.size) < 0.003
    resets[0] = True
    got = orc.decode_words("callerid", 8, words, resets, state=P["state"])
    want = orc.ref_decode_words("callerid", 8, words, resets, L=P["lib"])
    assert got == want
    assert got.count(b"CALLER-ID\n") > 300
    import minimodem_b200 as mm
    assert len(got) <= mm.decode_max_bytes(mm.DECODE_CALLERID, 8, words.size)
    assert b"Time:  03/15 10:45\nPhone: 800-555-1212\nName:  JOHN DOE\n" in got
    assert b"Phone: [blocked]\nName:  [N/A]\n" in got


def test_callerid_documented_output_without_reference():
    """The two messages of the reference's own tests (tests/testdata-callerid-*.txt), by value."""
    got = orc.decode_words("callerid", 8, list(_mdmf([(1, b"03151045"), (2, b"8005551212"), (7, b"JOHN DOE")])),
                           [True] + [False] * 40)
    assert got == b"CALLER-ID\nTime:  03/15 10:45\nPhone: 800-555-1212\nName:  JOHN DOE\n"
    got = orc.decode_words("callerid", 8, list(_sdmf(b"03151045", b"8005551212")), None)
    assert got == b"CALLER-ID\nTime:  03/15 10:45\nPhone: 800-555-1212\n"


def test_baudot_shift_state_by_value():
    # LTRS R Y FIGS 1 2 SPACE(unshift) R  -> "RY12 R"; a reset returns to letters
    w = [0x1F, 0x0A, 0x15, 0x1B, 0x17, 0x13, 0x04, 0x0A]
    assert orc.decode_words("baudot", 5, w, [True] + [False] * 7) == b"RY12 R"
    st = orc.DecoderState()
    assert orc.decode_words("baudot", 5, [0x1B, 0x17], None, state=st) == b"1"
    assert st.baudot_charset == 2
    assert orc.decode_words("baudot", 5, [0x17], None, state=st) == b"1"       # state carried over
    assert orc.decode_words("baudot", 5, [0x17], [True], state=st) == b"Q"     # reset -> letters
    # before any reset the reference's state is "unknown", which prints figures (src/baudot.c:197,236-239)
    assert orc.decode_words("baudot", 5, [0x17], None) == b"1"


def test_binary_and_uic_by_value():
    assert orc.decode_words("binary", 8, [0x41, 0xFF], None) == b"10000010\n11111111\n"
    assert orc.decode_words("binary", 5, [0x01], None) == b"10000\n"
    # train id nibbles 1..6 from bit 0, message 0x09 bit-reversed in bits 24..31
    word = 0x654321 | (int("{:08b}".format(0x09)[::-1], 2) << 24)
    assert orc.decode_words("uic-ground", 39, [word], None) == b"Train ID: 123456 - Message: 09 (Emergency stop)\n"
    assert orc.decode_words("uic-train", 39, [word], None) == \
        b"Train ID: 123456 - Message: 09 (Train staff wish to comm.)\n"
    word = 0xABCDEF | (int("{:08b}".format(0x7E)[::-1], 2) << 24)
    assert orc.decode_words("uic-train", 39, [word], None) == b"Train ID: FEDCBA - Message: 7E (Unknown)\n"


def test_output_cap_counts_are_clamped_by_the_caller():
    # the sink keeps counting past the capacity; only the first `cap` bytes are stored
    out = orc.decode_words("binary", 8, [0x41] * 4, None, cap=20)
    assert out == (b"10000010\n" * 3)[:20]


# --------------------------------------------------------------------------
# frame records of the rx-loop restatement -> the reference CLI's stdout
# --------------------------------------------------------------------------
GOLD = [c for c in refcases.ALL if c["name"] in (
    "01-self-test-1200", "03-self-test-rtty", "60-multibyte", "70-callerid-mdmf", "71-callerid-sdmf",
    "80-SAME", "81-ascii7", "81-tdd", "21-rate-slop-308", "40-noise-0.50", "small-rtty", "small-same")]
GOLD += refcases.OPTIONS + [c for c in refcases.MORE if not c["ring_limited"]]


@pytest.mark.parametrize("case", GOLD, ids=[c["name"] for c in GOLD])
def test_records_decode_to_reference_stdout(case):
    g = gu.load(case["name"])
    _, rx = gu.modes(case)
    a = gu.audio(case, g)
    r = orc.rx_run(rx, a, literal=False, rxnoise=case["rxnoise"], rx_one=case["rx_one"])
    rec = orc.frame_records(r["frames"])
    kind = refcases.decoder_of(case, rx)
    got = orc.decode_records(rx, kind, rec)
    assert got == bytes(g["stdout"])
    # a stream decoded in two batches continues where it stopped
    st = orc.DecoderState()
    k = rec.shape[0] // 2
    two = orc.decode_records(rx, kind, rec[:k], state=st) + orc.decode_records(rx, kind, rec[k:], state=st)
    assert two == got
    # session reports in the record stream are skipped
    mixed = np.insert(rec, k, np.array([1, 2, 3, 4, orc.FRAME_REPORT], np.uint32), axis=0)
    assert orc.decode_records(rx, kind, mixed) == got


def test_decoder_choice_follows_the_reference_main():
    import minimodem_b200 as mm
    assert mm.decoder_for_mode("1200") == mm.DECODE_ASCII                  # src/minimodem.c:552
    assert mm.decoder_for_mode("rtty", 5) == mm.DECODE_BAUDOT              # :820
    assert mm.decoder_for_mode("tdd", 5) == mm.DECODE_BAUDOT               # :828
    assert mm.decoder_for_mode("300", 5) == mm.DECODE_BAUDOT               # -5, :673-676
    assert mm.decoder_for_mode("callerid") == mm.DECODE_CALLERID           # :856
    assert mm.decoder_for_mode("uic-train", 39) == mm.DECODE_UIC_TRAIN     # :865-866
    assert mm.decoder_for_mode("uic-ground", 39) == mm.DECODE_UIC_GROUND   # :867-868
    assert mm.decoder_for_mode("rtty", 5, binary_output=True) == mm.DECODE_BINARY   # :891-892
    assert mm.decode_max_bytes_per_frame(mm.DECODE_BINARY, 8) == 9
    assert mm.decode_max_bytes_per_frame(mm.DECODE_UIC_TRAIN, 39) >= len(
        b"Train ID: 123456 - Message: 09 (Train staff wish to comm.)\n")
    assert C.sizeof(mm.DecoderState) == mm.DECODER_STATE_BYTES == C.sizeof(orc.DecoderState)
