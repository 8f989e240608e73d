"""ctypes bindings for the TEST-INFRASTRUCTURE oracle (oracle/liboracle.so, our
CPU restatement) and for oracle/_ref/libfsk_ref.so (the unmodified reference
src/fsk.c + databits decoders compiled in place).  Only tests/, bench.py's
cpu_baseline / --impl reference legs and __graft_entry__.smoke() import this.

Where oracle/_ref is not built, the reference's answers to the tests' inputs come
from tests/golden/reference_results.json (see `recorded`).

Also holds an independent Python restatement of the reference's mode presets
(src/minimodem.c:819-965) used to cross-check the product's host-side presets.
"""
import atexit
import base64
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIBORACLE = os.path.join(ORACLE_DIR, "liboracle.so")
LIBREF = os.path.join(ORACLE_DIR, "_ref", "libfsk_ref.so")
# the same unmodified src/fsk.c on MKL's DFTI FFT (oracle/shim/fftw3_dfti.c): timing only
LIBREF_DFTI = os.path.join(ORACLE_DIR, "_ref", "libfsk_ref_dfti.so")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "minimodem_ref")
REF_CLI_TRACE = os.path.join(ORACLE_DIR, "_ref", "minimodem_ref_trace")
REFERENCE_SRC = "/root/reference"
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
RECORDED = os.path.join(GOLDEN_DIR, "reference_results.json")

f32 = np.float32


def build_oracle(force=False):
    src = [os.path.join(ORACLE_DIR, f) for f in ("fsk_oracle.c", "fsk_oracle.h", "decode_oracle.c")]
    src.append(os.path.join(ROOT, "minimodem_b200", "csrc", "fsk_b200_decode_core.h"))
    if force or not os.path.exists(LIBORACLE) or any(
            os.path.getmtime(s) > os.path.getmtime(LIBORACLE) for s in src):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liboracle.so"])
    return LIBORACLE


def build_ref():
    """(Re)build oracle/_ref from /root/reference when that tree is present."""
    if os.path.isdir(os.path.join(REFERENCE_SRC, "src")):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "ref"])
    return os.path.exists(LIBREF)


def have_ref():
    return os.path.exists(LIBREF)


# --------------------------------------------------------------------------
# recorded answers of the unmodified reference
# --------------------------------------------------------------------------
_store = None
_new = {}


def _read_store():
    if not os.path.exists(RECORDED):
        return {}
    with open(RECORDED) as f:
        return json.load(f)


def _load_store():
    global _store
    if _store is None:
        _store = _read_store()
        if os.environ.get("FSK_RECORD_REFERENCE") == "1":
            atexit.register(_save_store)
    return _store


def _save_store():
    """Adds this process's answers to the file (other processes may have added theirs meanwhile)."""
    if _new:
        store = _read_store()
        store.update(_new)
        with open(RECORDED, "w") as f:
            f.write("{\n" + ",\n".join("%s:%s" % (json.dumps(k), json.dumps(store[k], separators=(",", ":")))
                                       for k in sorted(store)) + "\n}\n")


def record_key(*parts):
    """A stable name for one question put to the reference: its function and every input, byte for byte."""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, np.ndarray):
            b = p.dtype.str.encode() + repr(p.shape).encode() + np.ascontiguousarray(p).tobytes()
        elif isinstance(p, (bytes, bytearray)):
            b = bytes(p)
        elif isinstance(p, (float, np.floating)):
            b = np.float64(p).tobytes()
        else:
            b = repr(p).encode()
        h.update(len(b).to_bytes(8, "little") + b)
    return h.hexdigest()[:32]


def recorded(key, live):
    """The reference's answer to the question `key`.  Where oracle/_ref is built, `live()` asks the
    compiled reference (and FSK_RECORD_REFERENCE=1 writes the answer to tests/golden/reference_results.json);
    elsewhere the answer comes from that file.  A question it has no answer for is an error: the input
    the test put to the reference is not the one it was recorded with."""
    store = _load_store()
    if have_ref():
        value = live()
        if os.environ.get("FSK_RECORD_REFERENCE") == "1":
            _new[key] = value
        return value
    assert key in store, "no recorded reference answer for this input (%s); oracle/_ref is not built" % key
    return store[key]


class RecordedBytes:
    """A long output of the reference, recorded as its length and sha256: equal to exactly those bytes."""

    def __init__(self, n, sha256):
        self.n, self.sha256 = n, sha256

    def __eq__(self, other):
        if isinstance(other, RecordedBytes):
            return (self.n, self.sha256) == (other.n, other.sha256)
        return (isinstance(other, (bytes, bytearray)) and len(other) == self.n
                and hashlib.sha256(other).hexdigest() == self.sha256)

    __hash__ = None

    def __len__(self):
        return self.n

    def __repr__(self):
        return "<%d bytes of reference output, sha256 %s>" % (self.n, self.sha256)


def _enc_bytes(b, verbatim=256):
    if len(b) <= verbatim:
        return base64.b64encode(bytes(b)).decode()
    return {"len": len(b), "sha256": hashlib.sha256(b).hexdigest()}


def _dec_bytes(v):
    return base64.b64decode(v) if isinstance(v, str) else RecordedBytes(v["len"], v["sha256"])


# --------------------------------------------------------------------------
# struct mirrors of oracle/fsk_oracle.h
# --------------------------------------------------------------------------
class OrcPlan(C.Structure):
    _fields_ = [("sample_rate", C.c_float), ("f_mark", C.c_float), ("f_space", C.c_float),
                ("band_width", C.c_float), ("fftsize", C.c_int), ("nbands", C.c_uint),
                ("b_mark", C.c_uint), ("b_space", C.c_uint), ("tw_n", C.c_uint),
                ("tw", C.c_void_p)]


class OrcRxConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_float), ("data_rate", C.c_float),
                ("f_mark", C.c_float), ("f_space", C.c_float), ("band_width", C.c_float),
                ("n_data_bits", C.c_uint), ("nstartbits", C.c_int), ("nstopbits", C.c_float),
                ("invert_start_stop", C.c_int), ("msb_first", C.c_int),
                ("do_rx_sync", C.c_int), ("sync_byte", C.c_ulonglong),
                ("confidence_threshold", C.c_float), ("confidence_search_limit", C.c_float),
                ("expect_data_string", C.c_char_p)]


class OrcRxDerived(C.Structure):
    _fields_ = [("nsamples_per_bit", C.c_float), ("frame_n_bits", C.c_uint),
                ("frame_nsamples", C.c_uint), ("expect_n_bits", C.c_uint),
                ("expect_nsamples", C.c_uint), ("nsamples_overscan", C.c_uint),
                ("samplebuf_size", C.c_size_t), ("expect_data", C.c_char * 68),
                ("expect_sync", C.c_char * 68)]


class OrcRxFrame(C.Structure):
    _fields_ = [("bits", C.c_ulonglong), ("confidence", C.c_float), ("amplitude", C.c_float),
                ("frame_start", C.c_uint), ("acquired", C.c_uint), ("pos", C.c_ulonglong)]


class OrcRxReport(C.Structure):
    _fields_ = [("nframes_decoded", C.c_uint), ("carrier_nsamples", C.c_ulonglong),
                ("confidence_total", C.c_float), ("amplitude_total", C.c_float),
                ("after_frame", C.c_uint)]


class OrcRxCall(C.Structure):
    _fields_ = [("frame_nsamples", C.c_uint), ("try_first", C.c_uint), ("try_max", C.c_uint),
                ("try_step", C.c_uint), ("limit", C.c_float), ("use_sync_string", C.c_int),
                ("confidence", C.c_float), ("bits", C.c_ulonglong), ("ampl", C.c_float),
                ("frame_start", C.c_uint), ("pos", C.c_ulonglong)]


class OrcRxResult(C.Structure):
    _fields_ = [("frames", C.POINTER(OrcRxFrame)), ("nframes", C.c_size_t), ("cap_frames", C.c_size_t),
                ("reports", C.POINTER(OrcRxReport)), ("nreports", C.c_size_t), ("cap_reports", C.c_size_t),
                ("calls", C.POINTER(OrcRxCall)), ("ncalls", C.c_size_t), ("cap_calls", C.c_size_t),
                ("n_find_frame_calls", C.c_ulonglong)]


class OrcTxConfig(C.Structure):
    _fields_ = [("sample_rate", C.c_float), ("data_rate", C.c_float),
                ("f_mark", C.c_float), ("f_space", C.c_float), ("n_data_bits", C.c_uint),
                ("nstartbits", C.c_float), ("nstopbits", C.c_float),
                ("invert_start_stop", C.c_int), ("msb_first", C.c_int),
                ("do_tx_sync_bytes", C.c_uint), ("sync_byte", C.c_uint),
                ("leader_bits", C.c_int), ("trailer_bits", C.c_int),
                ("amplitude", C.c_float), ("sin_table_len", C.c_uint), ("s16", C.c_int)]


FIND_FRAME_FN = C.CFUNCTYPE(C.c_float, C.c_void_p, C.POINTER(C.c_float), C.c_uint, C.c_uint,
                            C.c_uint, C.c_uint, C.c_float, C.c_char_p,
                            C.POINTER(C.c_ulonglong), C.POINTER(C.c_float), C.POINTER(C.c_uint))

_lib = None


def lib():
    global _lib
    if _lib is None:
        build_oracle()
        L = C.CDLL(LIBORACLE)
        fp = C.POINTER(C.c_float)
        L.orc_plan_init.argtypes = [C.POINTER(OrcPlan), C.c_float, C.c_float, C.c_float, C.c_float]
        L.orc_plan_init.restype = C.c_int
        L.orc_plan_free.argtypes = [C.POINTER(OrcPlan)]
        L.orc_bit_mags.argtypes = [C.POINTER(OrcPlan), fp, C.c_uint, fp, fp]
        L.orc_frame_analyze.argtypes = [C.POINTER(OrcPlan), fp, C.c_float, C.c_int, C.c_char_p,
                                        C.POINTER(C.c_ulonglong), fp, fp, fp, C.POINTER(C.c_uint)]
        L.orc_frame_analyze.restype = C.c_float
        L.orc_find_frame.argtypes = [C.POINTER(OrcPlan), fp, C.c_uint, C.c_uint, C.c_uint, C.c_uint,
                                     C.c_float, C.c_char_p, C.POINTER(C.c_ulonglong), fp,
                                     C.POINTER(C.c_uint)]
        L.orc_find_frame.restype = C.c_float
        L.orc_rx_derive.argtypes = [C.POINTER(OrcRxConfig), C.POINTER(OrcRxDerived)]
        L.orc_rx_run.argtypes = [C.POINTER(OrcRxConfig), fp, C.c_size_t, C.c_int, C.c_float,
                                 C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(OrcRxResult)]
        L.orc_rx_run.restype = C.c_int
        L.orc_rx_result_free.argtypes = [C.POINTER(OrcRxResult)]
        L.orc_rx_databits.argtypes = [C.POINTER(OrcRxConfig), C.c_ulonglong]
        L.orc_rx_databits.restype = C.c_ulonglong
        L.orc_decode_words.argtypes = [C.c_int, C.c_uint, C.c_void_p, C.POINTER(C.c_ulonglong), C.c_uint,
                                       C.c_char_p, C.c_char_p, C.c_uint]
        L.orc_decode_words.restype = C.c_uint
        L.orc_decode_records.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_int, C.c_int, C.c_ulonglong,
                                         C.c_void_p, C.c_void_p, C.c_uint, C.c_char_p, C.c_uint]
        L.orc_decode_records.restype = C.c_uint
        L.orc_rx_many.argtypes = [C.POINTER(OrcRxConfig), fp, C.c_size_t, C.c_size_t, C.c_size_t,
                                  C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(C.c_uint), C.POINTER(C.c_ulonglong)]
        L.orc_rx_many.restype = C.c_ulonglong
        L.orc_pool_new.argtypes = [C.POINTER(OrcRxConfig), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_pool_new.restype = C.c_void_p
        L.orc_pool_load.argtypes = [C.c_void_p, fp, C.c_size_t, C.c_size_t, C.c_size_t]
        L.orc_pool_load.restype = C.c_int
        L.orc_pool_run.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(C.c_uint),
                                   C.POINTER(C.c_ulonglong)]
        L.orc_pool_run.restype = C.c_double
        L.orc_pool_free.argtypes = [C.c_void_p]
        L.orc_tx_nsamples.argtypes = [C.POINTER(OrcTxConfig), C.c_size_t]
        L.orc_tx_nsamples.restype = C.c_size_t
        L.orc_tx_words.argtypes = [C.POINTER(OrcTxConfig), C.POINTER(C.c_uint), C.c_size_t, fp, C.c_size_t]
        L.orc_tx_words.restype = C.c_size_t
        L.orc_build_expect_bits_string.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_float, C.c_int,
                                                   C.c_int, C.c_ulonglong]
        L.orc_build_expect_bits_string.restype = C.c_int
        _lib = L
    return _lib


def fptr(a):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_float))


# --------------------------------------------------------------------------
# mode presets: Python restatement of src/minimodem.c:819-965
# --------------------------------------------------------------------------
class Mode:
    """Everything main() derives from `{baudmode}` and the options the reference
    tests use.  Field names follow the reference's variables."""

    def __init__(self, mode, sample_rate=48000, mark=0.0, space=0.0, n_data_bits=0,
                 startbits=-1, stopbits=-1.0, bandwidth=0.0, inverted=False,
                 invert_start_stop=False, msb_first=False, sync_byte=None,
                 confidence=1.5, limit=2.3, baudot=False):
        self.mode = str(mode)
        self.sample_rate = int(sample_rate)
        band_width = f32(bandwidth)
        mark_f = f32(mark)
        space_f = f32(space)
        nstartbits = int(startbits)
        nstopbits = f32(stopbits)
        do_rx_sync = 0
        do_tx_sync_bytes = 0
        sb = (1 << 64) - 1            # (unsigned long long)-1, :501
        if sync_byte is not None:     # :716-720
            do_rx_sync, do_tx_sync_bytes, sb = 1, 16, int(sync_byte)
        self.decoder = "baudot" if baudot else "ascii8"
        if baudot:
            n_data_bits = 5           # :673-677
        self.expect_data_string = None
        m = self.mode.lower()
        if m == "rtty":                               # :819-826
            self.decoder = "baudot"
            data_rate = f32(45.45)
            n_data_bits = n_data_bits or 5
            if nstopbits < 0:
                nstopbits = f32(1.5)
        elif m == "tdd":                              # :827-836
            self.decoder = "baudot"
            data_rate = f32(45.45)
            n_data_bits = n_data_bits or 5
            if nstopbits < 0:
                nstopbits = f32(2.0)
            mark_f, space_f = f32(1400), f32(1800)
        elif m == "same":                             # :837-848
            data_rate = f32(520.0 + 5 / 6.0)
            n_data_bits = 8
            nstartbits, nstopbits = 0, f32(0)
            do_rx_sync, do_tx_sync_bytes, sb = 1, 16, 0xAB
            mark_f = f32(2083.0 + 1 / 3.0)
            space_f = f32(1562.5)
            band_width = data_rate
        elif m.startswith("caller"):                  # :849-858
            self.decoder = "callerid"
            data_rate = f32(1200)
            n_data_bits = 8
        elif m.startswith("uic"):                     # :859-876
            self.decoder = "uic-train" if (len(m) > 4 and m[4] == "t") else "uic-ground"
            data_rate = f32(600)
            n_data_bits = 39
            mark_f, space_f = f32(1300), f32(1700)
            nstartbits, nstopbits = 8, f32(0)
            self.expect_data_string = b"11110010" + b"d" * 39
        elif m.startswith("v.21"):                    # :877-881
            data_rate = f32(300)
            mark_f, space_f = f32(980), f32(1180)
            n_data_bits = 8
        else:                                         # :882-886
            data_rate = f32(float(self.mode))
            n_data_bits = n_data_bits or 8
        assert data_rate != 0
        if data_rate >= 400:                          # :900-910
            shift = -int(f32(f32(data_rate * f32(5)) / f32(6)))
            if mark_f == 0:
                mark_f = f32(f32(data_rate / f32(2)) + f32(600))
            if space_f == 0:
                space_f = f32(mark_f - f32(shift))
            if band_width == 0:
                band_width = f32(200)
        elif data_rate >= 100:                        # :911-921
            shift = 200
            if mark_f == 0:
                mark_f = f32(1270)
            if space_f == 0:
                space_f = f32(mark_f - f32(shift))
            if band_width == 0:
                band_width = f32(50)
        else:                                         # :922-934
            shift = 170
            if mark_f == 0:
                mark_f = f32(1585)
            if space_f == 0:
                space_f = f32(mark_f - f32(shift))
            if band_width == 0:
                band_width = f32(10)
        self.autodetect_shift = shift
        if nstartbits < 0:                            # :937-940
            nstartbits = 1
        if nstopbits < 0:
            nstopbits = f32(1.0)
        self.frame_n_bits = int(f32(f32(n_data_bits + nstartbits) + nstopbits))   # :943
        self.leader_bits = 0 if nstartbits == 0 else 2    # :950-951, :51
        self.trailer_bits = 2                             # :52
        if inverted:                                      # :953-957
            mark_f, space_f = space_f, mark_f
        if band_width > data_rate:                        # :960-961
            band_width = data_rate
        limit = f32(limit)
        confidence = f32(confidence)
        if limit < confidence:                            # :964-965
            limit = confidence
        self.data_rate = f32(data_rate)
        self.mark_f, self.space_f, self.band_width = f32(mark_f), f32(space_f), f32(band_width)
        self.n_data_bits, self.nstartbits, self.nstopbits = int(n_data_bits), nstartbits, f32(nstopbits)
        self.invert_start_stop, self.msb_first = int(invert_start_stop), int(msb_first)
        self.do_rx_sync, self.do_tx_sync_bytes, self.sync_byte = do_rx_sync, do_tx_sync_bytes, sb
        self.confidence_threshold, self.confidence_search_limit = confidence, limit

    def rx_config(self):
        c = OrcRxConfig()
        c.sample_rate = self.sample_rate
        c.data_rate = self.data_rate
        c.f_mark, c.f_space, c.band_width = self.mark_f, self.space_f, self.band_width
        c.n_data_bits, c.nstartbits, c.nstopbits = self.n_data_bits, self.nstartbits, self.nstopbits
        c.invert_start_stop, c.msb_first = self.invert_start_stop, self.msb_first
        c.do_rx_sync, c.sync_byte = self.do_rx_sync, self.sync_byte
        c.confidence_threshold = self.confidence_threshold
        c.confidence_search_limit = self.confidence_search_limit
        c.expect_data_string = self.expect_data_string
        return c

    def tx_config(self, amplitude=1.0, lut=4096, float_samples=False):
        c = OrcTxConfig()
        c.sample_rate = self.sample_rate
        c.data_rate = self.data_rate
        c.f_mark, c.f_space = self.mark_f, self.space_f
        c.n_data_bits = self.n_data_bits
        c.nstartbits, c.nstopbits = self.nstartbits, self.nstopbits
        c.invert_start_stop, c.msb_first = self.invert_start_stop, self.msb_first
        c.do_tx_sync_bytes = self.do_tx_sync_bytes
        c.sync_byte = self.sync_byte & 0xFFFFFFFF
        c.leader_bits, c.trailer_bits = self.leader_bits, self.trailer_bits
        c.amplitude = amplitude
        c.sin_table_len = lut
        c.s16 = 0 if float_samples else 1
        return c

    def derived(self):
        d = OrcRxDerived()
        cfg = self.rx_config()
        lib().orc_rx_derive(C.byref(cfg), C.byref(d))
        return d


# --------------------------------------------------------------------------
# convenience wrappers
# --------------------------------------------------------------------------
class Plan:
    def __init__(self, sample_rate, f_mark, f_space, bw):
        self.p = OrcPlan()
        if lib().orc_plan_init(C.byref(self.p), sample_rate, f_mark, f_space, bw) != 0:
            raise ValueError("orc_plan_init: EINVAL")

    def __del__(self):
        try:
            lib().orc_plan_free(C.byref(self.p))
        except Exception:
            pass

    def find_frame(self, samples, frame_nsamples, try_first, try_max, try_step, limit, expect):
        bits, ampl, start = C.c_ulonglong(0), C.c_float(0), C.c_uint(0)
        if isinstance(expect, str):
            expect = expect.encode()
        c = lib().orc_find_frame(C.byref(self.p), fptr(samples), frame_nsamples, try_first,
                                 try_max, try_step, limit, expect,
                                 C.byref(bits), C.byref(ampl), C.byref(start))
        return f32(c), bits.value, f32(ampl.value), start.value

    def frame_analyze(self, samples, spb, expect):
        if isinstance(expect, str):
            expect = expect.encode()
        n = len(expect)
        sig = np.zeros(n, np.float32)
        noise = np.zeros(n, np.float32)
        val = np.zeros(n, np.uint32)
        bits, ampl = C.c_ulonglong(0), C.c_float(0)
        c = lib().orc_frame_analyze(C.byref(self.p), fptr(samples), spb, n, expect, C.byref(bits),
                                    C.byref(ampl), fptr(sig), fptr(noise),
                                    val.ctypes.data_as(C.POINTER(C.c_uint)))
        return f32(c), bits.value, f32(ampl.value), sig, noise, val

    def bit_mags(self, samples, n):
        a, b = C.c_float(0), C.c_float(0)
        lib().orc_bit_mags(C.byref(self.p), fptr(samples), n, C.byref(a), C.byref(b))
        return f32(a.value), f32(b.value)


def rx_run(mode, samples, literal=False, rxnoise=0.0, rx_one=False, want_calls=False,
           find_frame=None):
    """Run the oracle rx loop; returns dict of numpy arrays."""
    samples = np.ascontiguousarray(samples, np.float32)
    cfg = mode.rx_config()
    res = OrcRxResult()
    cb = None
    if find_frame is not None:
        cb = FIND_FRAME_FN(find_frame)
    rc = lib().orc_rx_run(C.byref(cfg), fptr(samples), samples.size, 0 if literal else 1,
                          rxnoise, int(rx_one), int(want_calls),
                          C.cast(cb, C.c_void_p) if cb else None, None, C.byref(res))
    if rc != 0:
        raise ValueError("orc_rx_run failed")
    out = {
        "frames": [(r.bits, f32(r.confidence), f32(r.amplitude), r.frame_start, r.acquired, r.pos)
                   for r in (res.frames[i] for i in range(res.nframes))],
        "reports": [(r.nframes_decoded, r.carrier_nsamples, f32(r.confidence_total),
                     f32(r.amplitude_total), r.after_frame)
                    for r in (res.reports[i] for i in range(res.nreports))],
        "calls": [(r.frame_nsamples, r.try_first, r.try_max, r.try_step, f32(r.limit),
                   r.use_sync_string, f32(r.confidence), r.bits, f32(r.ampl), r.frame_start, r.pos)
                  for r in (res.calls[i] for i in range(res.ncalls))],
        "n_calls": res.n_find_frame_calls,
    }
    lib().orc_rx_result_free(C.byref(res))
    return out


def tx_words(mode, words, amplitude=1.0, lut=4096, float_samples=False):
    cfg = mode.tx_config(amplitude, lut, float_samples)
    words = np.ascontiguousarray(words, np.uint32)
    n = lib().orc_tx_nsamples(C.byref(cfg), words.size)
    out = np.zeros(n, np.float32)
    got = lib().orc_tx_words(C.byref(cfg), words.ctypes.data_as(C.POINTER(C.c_uint)), words.size,
                             fptr(out), n)
    assert got == n, (got, n)
    return out


def databits(mode, bits):
    cfg = mode.rx_config()
    return lib().orc_rx_databits(C.byref(cfg), bits)


# ---- N1: the host build of the product's decoder source (oracle/decode_oracle.c) ------------
DECODE_KINDS = {"ascii8": 0, "binary": 1, "baudot": 2, "callerid": 3, "uic-ground": 4, "uic-train": 5}
FRAME_ACQUIRED = 0x80000000
FRAME_REPORT = 0xFFFFFFFF


class DecoderState(C.Structure):
    """fsk_b200_decoder_state (include/fsk_b200.h)"""
    _fields_ = [("baudot_charset", C.c_uint32), ("cid_msgtype", C.c_uint32), ("cid_ndata", C.c_uint32),
                ("reserved", C.c_uint32), ("cid_buf", C.c_uint8 * 256)]


def decode_words(kind, n_data_bits, words, resets=None, state=None, cap=1 << 20):
    """data words -> bytes through decoder `kind` (name or number); resets[i] = a decoder reset
    before word i.  `state` (DecoderState) persists across calls when given."""
    k = DECODE_KINDS.get(kind, kind)
    st = state if state is not None else DecoderState()
    w = (C.c_ulonglong * max(len(words), 1))(*[int(x) for x in words])
    rb = bytes(1 if r else 0 for r in resets) if resets is not None else None
    buf = C.create_string_buffer(cap)
    n = lib().orc_decode_words(k, n_data_bits, C.addressof(st), w, len(words), rb, buf, cap)
    return buf.raw[:min(n, cap)]


def frame_records(frames, reports_at=None):
    """oracle frames [(bits, conf, ampl, start, acquired, pos)...] -> uint32 [n, 5] records as
    rx_batch writes them (include/fsk_b200.h fsk_b200_frame)."""
    rec = np.zeros((len(frames), 5), np.uint32)
    for i, fr in enumerate(frames):
        rec[i, 0] = fr[0] & 0xFFFFFFFF
        rec[i, 1] = fr[0] >> 32
        rec[i, 2] = np.float32(fr[1]).view(np.uint32)
        rec[i, 3] = np.float32(fr[2]).view(np.uint32)
        rec[i, 4] = fr[3] | (FRAME_ACQUIRED if fr[4] else 0)
    return rec


def decode_records(mode, kind, records, state=None, cap=1 << 20):
    """uint32 [n, 5] frame records -> bytes, the walk k_decode does per stream."""
    k = DECODE_KINDS.get(kind, kind)
    st = state if state is not None else DecoderState()
    rec = np.ascontiguousarray(records, np.uint32).reshape(-1, 5)
    shift = (1 if mode.nstopbits != 0.0 else 0) + int(mode.nstartbits)
    sync = mode.sync_byte if mode.sync_byte is not None else 0xFFFFFFFFFFFFFFFF
    buf = C.create_string_buffer(cap)
    n = lib().orc_decode_records(k, shift, mode.n_data_bits, int(mode.msb_first), int(mode.do_rx_sync),
                                 sync & 0xFFFFFFFFFFFFFFFF, C.addressof(st), rec.ctypes.data, rec.shape[0],
                                 buf, cap)
    return buf.raw[:min(n, cap)]


def report_line(mode, report):
    """Format a report the way report_no_carrier does (src/minimodem.c:253-291)."""
    nframes, carrier_nsamples, ctot, atot, _ = report
    frame_n_bits = f32(mode.frame_n_bits)
    nbits_decoded = f32(f32(nframes) * frame_n_bits)
    sr = mode.sample_rate
    with np.errstate(all="ignore"):
        rate = f32(f32(nbits_decoded * f32(sr)) / f32(carrier_nsamples))
        conf = float(f32(ctot) / f32(nframes))
        ampl = float(f32(atot) / f32(nframes))
    s = "### NOCARRIER ndata=%u confidence=%.3f ampl=%.3f bps=%.2f" % (nframes, conf, ampl, float(rate))
    lhs = int(f32(f32(nbits_decoded * f32(sr)) + f32(0.5)))
    rhs = int(f32(mode.data_rate * f32(carrier_nsamples)))
    if lhs == rhs:
        s += " (rate perfect) ###"
    else:
        skew = f32(f32(rate - mode.data_rate) / mode.data_rate)
        s += " (%.1f%% %s) ###" % (float(abs(skew) * f32(100.0)), "slow" if np.signbit(skew) else "fast")
    return s


# --------------------------------------------------------------------------
# the unmodified reference, as a library (oracle/_ref/libfsk_ref.so)
# --------------------------------------------------------------------------
_ref = None


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(LIBREF)
        fp = C.POINTER(C.c_float)
        L.fsk_plan_new.argtypes = [C.c_float] * 4
        L.fsk_plan_new.restype = C.c_void_p
        L.fsk_plan_destroy.argtypes = [C.c_void_p]
        L.fsk_find_frame.argtypes = [C.c_void_p, fp, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_float,
                                     C.c_char_p, C.POINTER(C.c_ulonglong), fp, C.POINTER(C.c_uint)]
        L.fsk_find_frame.restype = C.c_float
        for name in ("databits_decode_ascii8", "databits_decode_baudot", "databits_decode_callerid",
                     "databits_decode_binary", "databits_decode_uic_ground", "databits_decode_uic_train"):
            fn = getattr(L, name)
            fn.argtypes = [C.c_char_p, C.c_uint, C.c_ulonglong, C.c_uint]
            fn.restype = C.c_uint
        # databits.h:65: databits_encode_baudot is a macro for baudot_encode
        for name in ("databits_encode_ascii8", "baudot_encode"):
            fn = getattr(L, name)
            fn.argtypes = [C.POINTER(C.c_uint), C.c_char]
            fn.restype = C.c_int
        _ref = L
    return _ref


_ref_dfti = None


def have_ref_dfti():
    return os.path.exists(LIBREF_DFTI)


def ref_dfti():
    """oracle/_ref/libfsk_ref_dfti.so: needs PyTorch's libraries (MKL lives in libtorch_cpu.so)."""
    global _ref_dfti
    if _ref_dfti is None:
        os.environ.setdefault("MKL_NUM_THREADS", "1")        # one transform per caller thread
        import torch  # noqa: F401  (loads libtorch_cpu.so with its dependencies)
        L = C.CDLL(LIBREF_DFTI)
        fp = C.POINTER(C.c_float)
        L.fsk_plan_new.argtypes = [C.c_float] * 4
        L.fsk_plan_new.restype = C.c_void_p
        L.fsk_plan_destroy.argtypes = [C.c_void_p]
        L.fsk_find_frame.argtypes = [C.c_void_p, fp, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_float,
                                     C.c_char_p, C.POINTER(C.c_ulonglong), fp, C.POINTER(C.c_uint)]
        L.fsk_find_frame.restype = C.c_float
        _ref_dfti = L
    return _ref_dfti


class RefPlan:
    """fsk_plan of the unmodified reference (src/fsk.c:33); recorded answers where oracle/_ref is not built."""

    def __init__(self, sample_rate, f_mark, f_space, bw):
        self.args = tuple(float(f32(x)) for x in (sample_rate, f_mark, f_space, bw))
        self.h = None
        if have_ref():
            self.h = ref().fsk_plan_new(sample_rate, f_mark, f_space, bw)
            if not self.h:
                raise ValueError("fsk_plan_new failed")

    def __del__(self):
        try:
            if self.h:
                ref().fsk_plan_destroy(self.h)
        except Exception:
            pass

    def find_frame(self, samples, frame_nsamples, try_first, try_max, try_step, limit, expect):
        if isinstance(expect, str):
            expect = expect.encode()
        args = (int(frame_nsamples), int(try_first), int(try_max), int(try_step), float(f32(limit)), bytes(expect))

        def live():
            bits, ampl, start = C.c_ulonglong(0), C.c_float(0), C.c_uint(0)
            c = ref().fsk_find_frame(self.h, fptr(samples), frame_nsamples, try_first, try_max, try_step,
                                     limit, expect, C.byref(bits), C.byref(ampl), C.byref(start))
            return [float(f32(c)), int(bits.value), float(f32(ampl.value)), int(start.value)]
        c, bits, ampl, start = recorded(record_key("fsk_find_frame", self.args, samples, args), live)
        return f32(c), bits, f32(ampl), start

    def detect_carrier(self, samples, nsamples, threshold):
        def live():
            fn = ref().fsk_detect_carrier
            fn.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_uint, C.c_float]
            fn.restype = C.c_int
            return int(fn(self.h, fptr(samples), nsamples, threshold))
        return recorded(record_key("fsk_detect_carrier", self.args, samples, int(nsamples), float(f32(threshold))),
                        live)


def ref_encode(decoder, data):
    """bytes -> frame data words through the reference's databits encoder."""
    def live():
        L = ref()
        enc = L.baudot_encode if decoder == "baudot" else L.databits_encode_ascii8
        words = []
        buf = (C.c_uint * 2)()
        for ch in data:
            n = enc(buf, C.c_char(bytes([ch])))
            words.extend(int(buf[i]) for i in range(n))
        return words
    return np.array(recorded(record_key("databits_encode", decoder, bytes(data)), live), np.uint32)


REF_DECODERS = {"ascii8": "databits_decode_ascii8", "baudot": "databits_decode_baudot",
                "callerid": "databits_decode_callerid", "binary": "databits_decode_binary",
                "uic-ground": "databits_decode_uic_ground", "uic-train": "databits_decode_uic_train"}


def ref_decode_words(kind, n_data_bits, words, resets, L=None):
    """data words -> output bytes through the reference's databits decoder `kind`, with a decoder reset
    before word i where resets[i].  L: the reference library to call (default: oracle/_ref/libfsk_ref.so)."""
    words = np.ascontiguousarray(words, np.uint64)
    resets = np.ascontiguousarray(resets, np.bool_)

    def live():
        fn = getattr(L or ref(), REF_DECODERS[kind])
        fn.argtypes = [C.c_char_p, C.c_uint, C.c_ulonglong, C.c_uint]
        fn.restype = C.c_uint
        buf = C.create_string_buffer(8192)
        out = bytearray()
        for w, r in zip(words, resets):
            if r:
                fn(None, 0, 0, 0)
            n = fn(buf, 8192, int(w), n_data_bits)
            out += buf.raw[:n]
        return _enc_bytes(out)
    return _dec_bytes(recorded(record_key("databits_decode", kind, int(n_data_bits), words, resets), live))


def ref_decode(mode, frames, decoder=None):
    """frame records -> output bytes through the reference's databits decoder,
    following src/minimodem.c:1351 (reset on acquire) and :1415-1446."""
    words, resets = [], []
    reset = False
    for fr in frames:
        bits, acquired = fr[0], fr[4]
        reset = reset or bool(acquired)
        data = databits(mode, bits)
        if mode.do_rx_sync and data == mode.sync_byte:      # :1436-1439 (a reset there acts on the next word)
            continue
        words.append(data)
        resets.append(reset)
        reset = False
    return ref_decode_words(decoder or mode.decoder, mode.n_data_bits, words, resets)


def ref_cli(tx_args, rx_args, text):
    """The unmodified reference CLI: `--tx tx_args` writes `text` to a WAV file, `--rx rx_args` reads it back.
    Returns what the tests compare with: the length and sha256 of the float32 samples the receiver saw, its
    stdout and its NOCARRIER stat lines."""
    def live():
        if GOLDEN_DIR not in sys.path:
            sys.path.insert(0, GOLDEN_DIR)
        from make_golden import read_wav
        with tempfile.TemporaryDirectory() as d:
            wav = os.path.join(d, "x.wav")
            subprocess.run([REF_CLI, "--tx", "--file", wav] + list(tx_args), input=text, check=True)
            r = subprocess.run([REF_CLI, "--rx", "--file", wav] + list(rx_args), stdout=subprocess.PIPE,
                               stderr=subprocess.PIPE, check=True)
            audio, _, _ = read_wav(wav)
        return {"audio_len": int(audio.size),
                "audio_sha256": hashlib.sha256(np.ascontiguousarray(audio, np.float32).tobytes()).hexdigest(),
                "stdout": _enc_bytes(r.stdout),
                "nocarrier": [ln.strip() for ln in r.stderr.decode().splitlines() if ln.startswith("### NOCARRIER")]}
    v = recorded(record_key("minimodem", list(tx_args), list(rx_args), bytes(text)), live)
    return dict(v, stdout=_dec_bytes(v["stdout"]))


def ref_cli_tx_image(tx_args, text, keep=256):
    """The first `keep` bytes and the length of the WAV file the reference CLI's `--tx tx_args` writes for `text`."""
    def live():
        with tempfile.TemporaryDirectory() as d:
            wav = os.path.join(d, "t.wav")
            subprocess.run([REF_CLI, "--tx", "--file", wav] + list(tx_args), input=text, check=True)
            image = open(wav, "rb").read()
        return {"head": _enc_bytes(image[:keep]), "len": len(image)}
    v = recorded(record_key("minimodem_tx_image", list(tx_args), bytes(text), keep), live)
    return _dec_bytes(v["head"]), v["len"]


def rx_many(mode, samples, nsamples=None, nthreads=1, kind="port"):
    """CPU baseline driver: kind="port" = the oracle's two-bin analyzer, kind="reference" =
    the unmodified src/fsk.c from oracle/_ref behind the same rx-loop restatement.
    samples: [nstreams, stride] float32.  Returns (total_frames, frames_per_stream, bits_xor)."""
    samples = np.ascontiguousarray(samples, np.float32)
    nstreams, stride = samples.shape
    n = int(nsamples if nsamples is not None else stride)
    cfg = mode.rx_config()
    fps = np.zeros(nstreams, np.uint32)
    bx = np.zeros(nstreams, np.uint64)
    pn = ff = pd = None
    if kind in ("reference", "reference-dfti"):
        R = ref() if kind == "reference" else ref_dfti()
        pn = C.cast(R.fsk_plan_new, C.c_void_p)
        ff = C.cast(R.fsk_find_frame, C.c_void_p)
        pd = C.cast(R.fsk_plan_destroy, C.c_void_p)
    total = lib().orc_rx_many(C.byref(cfg), fptr(samples.reshape(-1)), nstreams, stride, n, int(nthreads),
                              pn, ff, pd, fps.ctypes.data_as(C.POINTER(C.c_uint)),
                              bx.ctypes.data_as(C.POINTER(C.c_ulonglong)))
    return int(total), fps, bx


class RxPool:
    """Persistent CPU worker pool for the timing arms (oracle/fsk_oracle.c, orc_pool_*): `nthreads`
    workers pinned one per allowed CPU, one plan per worker built once, each worker owns a contiguous
    block of streams that it copied into pool memory itself (first touch).  kind as in rx_many."""

    def __init__(self, mode, nthreads=1, kind="port"):
        self.cfg = mode.rx_config()
        pn = ff = pd = None
        if kind in ("reference", "reference-dfti"):
            R = ref() if kind == "reference" else ref_dfti()
            pn = C.cast(R.fsk_plan_new, C.c_void_p)
            ff = C.cast(R.fsk_find_frame, C.c_void_p)
            pd = C.cast(R.fsk_plan_destroy, C.c_void_p)
        self._keep = (pn, ff, pd)
        self.nthreads = int(nthreads)
        self.h = lib().orc_pool_new(C.byref(self.cfg), self.nthreads, pn, ff, pd)
        assert self.h
        self.nstreams = 0

    def load(self, samples, nsamples=None):
        samples = np.ascontiguousarray(samples, np.float32)
        self.nstreams, stride = samples.shape
        self.nsamples = int(nsamples if nsamples is not None else stride)
        rc = lib().orc_pool_load(self.h, fptr(samples.reshape(-1)), self.nstreams, stride, self.nsamples)
        assert rc == 0

    def run(self):
        """One pass over the loaded streams: (seconds, total_frames, frames_per_stream, bits_xor)."""
        fps = np.zeros(self.nstreams, np.uint32)
        bx = np.zeros(self.nstreams, np.uint64)
        total = C.c_ulonglong(0)
        dt = lib().orc_pool_run(self.h, C.byref(total), fps.ctypes.data_as(C.POINTER(C.c_uint)),
                                bx.ctypes.data_as(C.POINTER(C.c_ulonglong)))
        assert dt >= 0.0, "a worker could not build its plan"
        return float(dt), int(total.value), fps, bx

    def close(self):
        if self.h:
            lib().orc_pool_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
