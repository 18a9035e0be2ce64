"""The C++ host-side mirror (waveform_b200/host/SpectrumSourceCUDA: ring buffers, A/V sync, timeout, live ticks through
the C-ABI) against the compiled reference driven with the SAME packet / tick schedule (what it produced is stored in
tests/golden/ref_gpu_host.npz by tests/golden/make_golden.py: silent flags and the DB_MIN pattern as digests, spectra as a
fixed sample of bins that includes every tick's first, last and strongest)."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from helpers import ReferenceOutputs, digest, parity_report, sample_rows, synth_pcm, take_sample

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def _build_driver(tmp_path):
    exe = tmp_path / "live_driver"
    lib = ROOT / "waveform_b200" / "lib"
    subprocess.run(["g++", "-std=c++17", "-O2", f"-I{ROOT/'include'}", f"-I{ROOT/'waveform_b200'/'host'}",
                    str(ROOT / "tests" / "host" / "live_driver.cpp"), str(ROOT / "waveform_b200" / "host" / "spectrum_source.cpp"),
                    f"-L{lib}", "-lwfstft", f"-Wl,-rpath,{lib}", "-o", str(exe)], check=True)
    return exe


def _reference_live(settings, cc, pcm, N, packet, fps, ticks):
    from oracle import refbind
    ref = refbind.RefSource(settings, impl=refbind.IMPL_GENERIC, channels=cc)
    L, h = ref.L, ref.h
    now = 10 * 10**9
    tick_ns, pkt_ns = 10**9 // fps, packet * 10**9 // 48000
    next_pkt, pos = now, 0
    clock = now
    ns = pcm.shape[1]
    out, sil = [], []

    def set_clock(t):
        nonlocal clock
        assert t >= clock
        L.wfref_advance_clock_ns(h, t - clock)
        clock = t

    for _ in range(ticks):
        now += tick_ns
        while next_pkt + pkt_ns <= now and pos + packet <= ns:
            next_pkt += pkt_ns
            set_clock(next_pkt)
            ref.push(pcm[0, pos:pos + packet], pcm[1, pos:pos + packet] if cc > 1 else None)
            pos += packet
        set_clock(now)
        ref.tick(np.float32(1.0) / np.float32(fps))
        out.append(np.stack([ref.decibels(c) for c in range(ref.display_channels)]))
        sil.append(ref.last_silent)
    return np.stack(out), np.array(sil, dtype=np.uint8)


LIVE_CASES = [(4096, 2, 1, 0), (2048, 1, 0, 0), (1024, 2, 0, 0), (2048, 2, 1, 1), (800, 1, 0, 1)]
PACKET, FPS, TICKS, NS = 480, 60, 45, 48000


def _live_case(N, cc, stereo, normalize):
    pcm = synth_pcm(1, cc, NS, seed=21)[0]
    pcm[:, 20000:] = 0.0  # goes silent: EMA decay, then the gate
    settings = {"fft_size": N, "channel_mode": "stereo" if stereo else "mono"}
    if normalize:  # the RMS feed runs live in both: capture_audio pre-accumulate + update_input_rms (not forced)
        settings["normalize_volume"] = True
    return pcm, settings


@pytest.mark.parametrize("N,cc,stereo,normalize", LIVE_CASES)
def test_live_adapter_matches_reference_plugin(tmp_path, N, cc, stereo, normalize):
    exe = _build_driver(tmp_path)
    pcm, settings = _live_case(N, cc, stereo, normalize)
    rec = ReferenceOutputs("gpu_host")[f"N{N}_cc{cc}_stereo{stereo}_norm{normalize}"]
    assert digest(pcm) == rec["inputs"], "inputs differ from the ones the reference was run on"
    inp, outp = tmp_path / "pcm.f32", tmp_path / "out.f32"
    pcm.astype(np.float32).tofile(inp)
    r = subprocess.run([str(exe), str(inp), str(cc), str(NS), str(N), str(PACKET), str(FPS), str(TICKS), str(outp),
                        str(stereo), str(normalize)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    B = N // 2
    dch = 2 if stereo else 1
    raw = np.fromfile(outp, dtype=np.uint8).reshape(TICKS, dch * B * 4 + 1)
    got = raw[:, :-1].copy().view(np.float32).reshape(TICKS, dch, B)
    got_sil = raw[:, -1]
    assert digest(got_sil) == rec["silent"]
    assert digest(got <= -758.0 + 1.0) == rec["floor"], "DB_MIN pattern"
    rep = parity_report(take_sample(got, rec["db_sample"]), rec["db"])
    assert rep["ok"], rep


def reference_records():
    """The compiled reference (oracle/_ref) driven live for each case above; tests/golden/make_golden.py stores the result."""
    recs = {}
    for i, (N, cc, stereo, normalize) in enumerate(LIVE_CASES):
        pcm, settings = _live_case(N, cc, stereo, normalize)
        ref, ref_sil = _reference_live(settings, cc, pcm, N, PACKET, FPS, TICKS)
        values, sample = sample_rows(ref, max(1, 384 // (ref.shape[0] * ref.shape[1])), seed=i)
        recs[f"N{N}_cc{cc}_stereo{stereo}_norm{normalize}"] = {
            "inputs": digest(pcm), "silent": digest(ref_sil), "floor": digest(ref <= -758.0 + 1.0), "db": values,
            "db_sample": sample}
    return recs
