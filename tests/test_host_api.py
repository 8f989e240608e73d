"""CPU-only checks of the product's host layer (no compute calls): the C-ABI
library loads and exports every symbol include/fsk_b200.h declares; the mode
presets and frame geometry it derives equal the oracle's restatement of
src/minimodem.c:819-1131 for every mode the reference tests use; without a CUDA
device the engine refuses to start (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import minimodem_b200 as mm
import orc
import refcases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _built():
    if not os.path.exists(mm.LIB_PATH):
        mm.build()


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "fsk_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(fsk_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations found"
    L = C.CDLL(mm.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert declared == set(mm.EXPORTS)
    assert "sm_100a" in mm.version()


MODES = [("1200", {}), ("300", {}), ("rtty", {}), ("tdd", {}), ("same", {}), ("callerid", {}),
         ("uic-train", {}), ("uic-ground", {}), ("V.21", {}), ("0.5", {}), ("12000", {}),
         ("1200", dict(sample_rate=24000, mark=1200, space=2400)), ("1200", dict(n_data_bits=7)),
         ("rtty", dict(sample_rate=8000)), ("292", {}), ("308", {}), ("110", {}), ("2400", dict(bandwidth=100)),
         ("1200", dict(inverted=True)), ("1200", dict(msb_first=True, startbits=2, stopbits=2.0)),
         ("600", dict(sync_byte=0x7E))]


# the option combinations minted from the reference CLI (tests/refcases.py OPTIONS), rx side
MODES += [(c["rx_mode"], c["rx_mkw"]) for c in refcases.OPTIONS + refcases.MORE]


def overrides_for(kw):
    """orc.Mode keyword names -> fsk_b200_rx_config override names (the -5 option is n_data_bits 5)."""
    names = dict(mark="f_mark", space="f_space", bandwidth="band_width", startbits="nstartbits",
                 stopbits="nstopbits", confidence="confidence_threshold", limit="confidence_search_limit")
    ov = {names.get(k, k): v for k, v in kw.items() if k not in ("sample_rate", "baudot")}
    if kw.get("baudot"):
        ov["n_data_bits"] = 5
    return ov


@pytest.mark.parametrize("mode,kw", MODES, ids=["%s-%d" % (m, i) for i, (m, _) in enumerate(MODES)])
def test_presets_and_geometry_match_oracle(mode, kw):
    om = orc.Mode(mode, **kw)
    od = om.derived()
    ov = overrides_for(kw)
    cfg = mm.rx_config_for_mode(mode, kw.get("sample_rate", 48000), **ov)
    assert np.float32(cfg.data_rate) == om.data_rate
    assert (np.float32(cfg.f_mark), np.float32(cfg.f_space)) == (om.mark_f, om.space_f)
    assert np.float32(cfg.band_width) == om.band_width
    assert (cfg.n_data_bits, cfg.nstartbits, np.float32(cfg.nstopbits)) == (om.n_data_bits, om.nstartbits, om.nstopbits)
    assert (cfg.do_rx_sync, cfg.sync_byte) == (om.do_rx_sync, om.sync_byte)
    assert (cfg.invert_start_stop, cfg.msb_first) == (om.invert_start_stop, om.msb_first)
    assert (np.float32(cfg.confidence_threshold), np.float32(cfg.confidence_search_limit)) == \
        (om.confidence_threshold, om.confidence_search_limit)
    p = mm.rx_params(cfg)
    op = orc.Plan(om.sample_rate, om.mark_f, om.space_f, om.band_width).p
    assert (p.fftsize, p.nbands, p.b_mark, p.b_space) == (op.fftsize, op.nbands, op.b_mark, op.b_space)
    assert np.float32(p.nsamples_per_bit) == np.float32(od.nsamples_per_bit)
    assert (p.frame_n_bits, p.frame_nsamples, p.expect_n_bits, p.expect_nsamples, p.nsamples_overscan) == \
        (od.frame_n_bits, od.frame_nsamples, od.expect_n_bits, od.expect_nsamples, od.nsamples_overscan)
    assert p.expect_data == od.expect_data and p.expect_sync == od.expect_sync
    spb = np.float32(p.expect_nsamples) / np.float32(p.expect_n_bits)
    assert p.bit_nsamples == int(np.float32(spb + np.float32(0.5)))
    for b in range(p.expect_n_bits):
        assert p.bit_begin[b] == int(np.float32(np.float32(spb * np.float32(b)) + np.float32(0.5)))
    tm_c = int(np.float32(np.float32(od.nsamples_per_bit) * np.float32(0.75) + np.float32(0.5))) + od.nsamples_overscan
    tm_n = int(np.float32(od.nsamples_per_bit)) + od.nsamples_overscan
    assert (p.try_max_carrier, p.try_max_nocarrier) == (tm_c, tm_n)
    # data word extraction, src/minimodem.c:1415-1428
    rng = np.random.default_rng(7)
    for _ in range(50):
        bits = int(rng.integers(0, 1 << 62))
        rec = dict(bits_lo=bits & 0xFFFFFFFF, bits_hi=bits >> 32, confidence=1.0, amplitude=1.0, frame_start=0)
        assert mm.frame_databits(p, rec) == orc.databits(om, bits)


def test_survey_table_values():
    """SURVEY.md 8(d): the derived integers of the BASELINE configs."""
    want = {
        ("1200", 48000): dict(fftsize=240, b=(6, 11), expect=440, frame=400, over=20, tmn=60, tmc=50, N=40, span=440),
        ("rtty", 8000): dict(fftsize=800, b=(159, 142), expect=1408, frame=1232, over=88, tmn=264, tmc=220, N=176, span=1408),
        ("300", 48000): dict(fftsize=960, b=(25, 21), expect=1760, frame=1600, over=80, tmn=240, tmc=200, N=160, span=1760),
        ("same", 48000): dict(fftsize=92, b=(4, 3), expect=737, frame=737, over=46, tmn=138, tmc=115, N=92, span=737),
    }
    for (mode, sr), w in want.items():
        p = mm.rx_params(mm.rx_config_for_mode(mode, sr))
        assert p.fftsize == w["fftsize"] and (p.b_mark, p.b_space) == w["b"]
        assert (p.expect_nsamples, p.frame_nsamples, p.nsamples_overscan) == (w["expect"], w["frame"], w["over"])
        assert (p.try_max_nocarrier, p.try_max_carrier) == (w["tmn"], w["tmc"])
        assert (p.bit_nsamples, p.span_nsamples) == (w["N"], w["span"])
    p = mm.rx_params(mm.rx_config_for_mode("same", 48000))
    assert list(p.bit_begin[:8]) == [0, 92, 184, 276, 369, 461, 553, 645]


def test_bad_plan_is_rejected_like_the_reference():
    cfg = mm.rx_config_for_mode("1200", 48000, f_mark=30000.0)   # band beyond nbands, src/fsk.c:58-64
    with pytest.raises(RuntimeError):
        mm.rx_params(cfg)
    with pytest.raises(RuntimeError):
        mm.rx_config_for_mode("0", 48000)                        # usage() at :887


def test_no_cpu_fallback_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = mm.rx_params(mm.rx_config_for_mode("1200"))
    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        mm.RxEngine(p)
    with pytest.raises(ValueError):
        mm.FskPlan(48000, 1200, 2200, 200)


def test_binding_refuses_the_emulation_build():
    """tests/emu builds the kernels' source for a host SIMT emulator behind the same C ABI; it is
    test infrastructure, and the product binding must not accept it in the library's place."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    import emu_mode
    lib = emu_mode.build()
    r = subprocess.run([sys.executable, "-c", "import minimodem_b200 as mm; mm.lib()"], cwd=ROOT,
                       env=dict(os.environ, FSK_B200_LIB=lib), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert r.returncode != 0 and b"HOST-EMULATION" in r.stdout and b"refuses" in r.stdout


def test_wav_locate_on_the_reference_transmitters_files():
    """N2, the file side: the WAV images the reference's own transmitter writes (S16 by default,
    float32 with --float-samples) are located exactly; what is not mono PCM16/float32 is refused."""
    import struct
    import golden_util as gu
    g = gu.load("small-1200")
    a = gu.audio(refcases.BY_NAME["small-1200"], g)

    def wav(samples, rate, fmt, bits, channels=1, junk=b""):
        data = samples.astype("<f4").tobytes() if fmt == 3 else np.round(samples * 32768).astype("<i2").tobytes()
        body = b"WAVE" + junk + b"fmt " + struct.pack("<IHHIIHH", 16, fmt, channels, rate, rate * bits // 8 * channels,
                                                      bits // 8 * channels, bits) + b"data" + struct.pack("<I", len(data)) + data
        return b"RIFF" + struct.pack("<I", len(body)) + body

    off, n, rate, isf = mm.wav_locate(wav(a, 48000, 1, 16))
    assert (off, n, rate, isf) == (44, a.size, 48000, False)
    off, n, rate, isf = mm.wav_locate(wav(a, 8000, 3, 32, junk=b"LIST" + struct.pack("<I", 5) + b"abcde\0"))
    assert (n, rate, isf) == (a.size, 8000, True) and off == 44 + 14
    img = wav(a, 48000, 1, 16)
    off, n, _, _ = mm.wav_locate(img[:44 + 100])              # truncated file: clipped, not refused
    assert (off, n) == (44, 50)
    for bad in (b"", b"RIFFxxxxWAVX", wav(a, 48000, 1, 16, channels=2), wav(a, 48000, 1, 8), img[:30]):
        with pytest.raises(RuntimeError):
            mm.wav_locate(bad)
    # a file written by the unmodified reference CLI: its header as recorded, the samples' bytes zeroed
    for extra, isfloat in (([], False), (["--float-samples"], True)):
        head, size = orc.ref_cli_tx_image(["1200"] + extra, b"wav header\n")
        image = head + bytes(size - len(head))
        off, n, rate, isf = mm.wav_locate(image)
        assert rate == 48000 and isf == isfloat and off + n * (4 if isfloat else 2) == len(image)
