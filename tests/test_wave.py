"""Waveform (oscilloscope) mode, tick_waveform: SURVEY.md §8(f) rank 4.

CPU: the oracle restatement (oracle/wf_oracle_meter.c, wfo_wave_*) bit-exact against what the compiled reference produced
(tests/golden/ref_wave.npz, digests of every tick's output) and against the committed golden fixtures.  GPU: the CUDA
path (wf_wave_* through the C-ABI) against the oracle — which points are emitted and which sample each takes is integer arithmetic and must match exactly (checked through the DB_MIN pattern and the silent
flags); the dBFS values agree to 1e-4 dB (log10f last-bit differences between glibc and CUDA).
"""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import pytest

from helpers import ReferenceOutputs, digest, synth_pcm

GOLD = sorted((Path(__file__).parent / "golden").glob("wave_*.npz"))

WAVE_CASES = [
    ({"width": 800, "meter_buf": 150}, 2, 800),                                   # defaults, two channels mixed to mono
    ({"width": 800, "meter_buf": 150, "channel_mode": "stereo"}, 2, 800),
    ({"width": 300, "meter_buf": 50}, 1, 441),
    ({"width": 200, "meter_buf": 10}, 1, 1600),                                   # packet longer than the window: silent rule fires
    ({"width": 640, "meter_buf": 500, "channel_mode": "stereo", "normalize_volume": True}, 2, 1024),
    ({"width": 1000, "meter_buf": 20, "channel_mode": "stereo"}, 1, 333),         # mono capture shown as two channels: the
                                                                                  # copy's newest points stay RAW (quirk)
]


def _case(settings, ch, hop, T=50, S=1):
    pcm = synth_pcm(S, ch, T * hop)
    pcm[:, :, 20 * hop: 30 * hop] = 0.0
    pcm[:, :, 33 * hop: 35 * hop] = 1.0  # |x| == 1 -> exactly 0.0 dBFS entries (the all-zero "silent" quirk's raw material)
    rms = (0.05 + 0.2 * np.random.default_rng(3).uniform(size=(S, T))).astype(np.float32) \
        if settings.get("normalize_volume") else None
    return pcm, rms


@pytest.fixture(scope="module")
def ref():
    return ReferenceOutputs("wave")


@pytest.mark.parametrize("settings,ch,hop", WAVE_CASES)
def test_wave_oracle_is_bit_exact_vs_compiled_reference(settings, ch, hop, ref):
    rec = ref[f"case{WAVE_CASES.index((settings, ch, hop))}"]
    _check_bit_exact(rec, settings, ch, hop, *_case(settings, ch, hop, T=50))


def _random_case(seed):
    rng = np.random.default_rng(7000 + seed)
    ch = int(rng.choice([1, 2]))
    settings = {"width": int(rng.choice([64, 200, 301, 640, 800, 1000, 1920])), "meter_buf": int(rng.choice([5, 10, 20, 50, 150, 500]))}
    if rng.uniform() < 0.5:
        settings["channel_mode"] = "stereo"
    if rng.uniform() < 0.3:
        settings["normalize_volume"] = True
    hop = int(rng.choice([97, 333, 441, 480, 800, 1024, 1600, 2000]))
    T = 60
    pcm = synth_pcm(1, ch, T * hop, seed=seed)
    a, b = sorted(int(v) for v in rng.integers(0, T, size=2))
    pcm[:, :, a * hop: (a + (b - a) // 2) * hop] = 1.0
    pcm[:, :, (a + (b - a) // 2) * hop: b * hop] = 0.0
    if ch == 2 and rng.uniform() < 0.4:
        pcm[:, 1] = 0.0
    rms = (0.05 + 0.2 * rng.uniform(size=(1, T))).astype(np.float32) if settings.get("normalize_volume") else None
    return settings, ch, hop, pcm, rms


@pytest.mark.parametrize("seed", range(30))
def test_wave_oracle_randomised_settings_bit_exact_vs_compiled_reference(seed, ref):
    """Differential fuzz of the waveform-mode oracle against the unmodified reference: random width, window length, packet size,
    channel layout, volume normalisation, stretches of zeros and of full-scale samples (the all-zero silent rule's raw material)."""
    _check_bit_exact(ref[f"random{seed}"], *_random_case(seed))


def _check_bit_exact(rec, settings, ch, hop, pcm, rms):
    from oracle.oraclebind import OracleWave

    assert digest(pcm) + digest(rms) == rec["inputs"], "inputs differ from the ones the reference was run on"
    T = pcm.shape[-1] // hop
    out = OracleWave(settings, channels=ch).run(pcm[0], T, hop, rms=None if rms is None else rms[0])
    assert digest(out["out"]) == rec["out"], settings
    assert digest(out["silent"]) == rec["silent"], settings


def reference_records():
    """m_decibels and m_last_silent of the compiled reference (oracle/_ref) after every tick of each case above, as digests;
    tests/golden/make_golden.py stores them."""
    from oracle import refbind

    recs = {}
    for name, (settings, ch, hop, pcm, rms) in [(f"case{i}", (s, c, h) + _case(s, c, h, T=50)) for i, (s, c, h) in enumerate(WAVE_CASES)] \
            + [(f"random{seed}", _random_case(seed)) for seed in range(30)]:
        T = pcm.shape[-1] // hop
        r = refbind.RefSource({"display_mode": "waveform", **settings}, channels=ch).run_wave(
            pcm[0], T, hop, rms=None if rms is None else rms[0])
        recs[name] = {"inputs": digest(pcm) + digest(rms), "out": digest(r["out"]), "silent": digest(r["silent"])}
    return recs


@pytest.mark.parametrize("path", GOLD, ids=[p.stem for p in GOLD])
def test_wave_oracle_against_reference_golden_vectors(path):
    from oracle.oraclebind import OracleWave

    z = np.load(path, allow_pickle=False)
    settings = json.loads(str(z["settings"]))
    rms = z["rms"] if z["rms"].size else None
    out = OracleWave(settings, channels=int(z["channels"])).run(z["pcm"], int(z["n_ticks"]), int(z["hop"]), rms=rms)
    assert np.array_equal(out["out"], z["out"]) and np.array_equal(out["silent"], z["silent"])


@pytest.mark.parametrize("width,meter_ms,hop", [(800, 150, 800), (300, 50, 441), (1000, 20, 333), (200, 10, 1600), (640, 500, 1024)])
def test_engine_timestamp_walk_equals_the_reference(width, meter_ms, hop):
    """No GPU needed: libwfstft's host-side plan (which points a tick emits, which sample each takes) against the oracle.
    A mono capture shown as two channels leaves the RAW new samples in the second channel (reference quirk), so a ramp input
    reveals the sample index the reference picked for every point."""
    from oracle.oraclebind import OracleWave
    from waveform_b200.engine import make_wave_config, preview_wave_plan

    T = 40
    settings = {"width": width, "meter_buf": meter_ms, "channel_mode": "stereo"}
    ramp = ((np.arange(T * hop, dtype=np.float64) + 1.0) * 2.0 ** -20).astype(np.float32)[None, :]  # exact, never 0
    ref = OracleWave(settings, channels=1).run(ramp, T, hop)["out"][:, 1, :]
    counts, src = preview_wave_plan(make_wave_config(settings, channels=1), T, hop)
    assert counts.min() >= 0 and counts.max() <= width and counts.sum() == len(src)
    o = 0
    for t in range(T):
        c = int(counts[t])
        want = np.where(src[o: o + c] >= 0, ramp[0, np.maximum(src[o: o + c], 0)], np.float32(0.0))
        assert np.array_equal(ref[t, width - c:], want), t
        o += c


def _oracle_batch(settings, ch, pcm, T, hop, rms):
    from oracle.oraclebind import OracleWave

    outs = [OracleWave(settings, channels=ch).run(pcm[s], T, hop, rms=None if rms is None else rms[s]) for s in range(pcm.shape[0])]
    return np.stack([o["out"] for o in outs]), np.stack([o["silent"] for o in outs])


@pytest.mark.gpu
@pytest.mark.parametrize("device_ptrs", [False, True])
@pytest.mark.parametrize("settings,ch,hop", WAVE_CASES)
def test_gpu_wave_parity_vs_oracle(settings, ch, hop, device_ptrs):
    from waveform_b200 import WaveEngine

    S, T = 4, 50
    pcm, rms = _case(settings, ch, hop, T, S)
    ref, ref_sil = _oracle_batch(settings, ch, pcm, T, hop, rms)
    eng = WaveEngine(settings, channels=ch, max_streams=S)
    if device_ptrs:
        import torch
        o = eng.process(torch.from_numpy(pcm).cuda(), T, hop, input_rms=None if rms is None else torch.from_numpy(rms))
        out, sil = o["out"].cpu().numpy(), o["silent"].cpu().numpy()
    else:
        o = eng.process(pcm, T, hop, input_rms=rms)
        out, sil = o["out"], o["silent"]
    assert np.array_equal(sil, ref_sil)
    lo = ref < -700.0                     # DB_MIN entries: which points exist / took a zero sample — integer arithmetic
    assert np.array_equal(out < -700.0, lo)
    untouched = ref == np.float32(-758.59564)  # never-converted or zero-sample entries without volume compensation
    assert np.array_equal(out[untouched], ref[untouched])
    raw = (~lo) & (np.abs(ref) <= 1.0) & (ref == out)  # raw samples kept by the reference (gathers are exact)
    # DB_MIN + volume compensation: the compensation itself goes through log10f (1 ulp between glibc and CUDA)
    assert np.max(np.abs(out[lo] - ref[lo]), initial=0.0) < 1e-3
    assert np.max(np.abs(out[~lo & ~raw] - ref[~lo & ~raw]), initial=0.0) < 1e-4
    # state continues across calls (the clock, the scrolling buffer, m_last_silent)
    eng2 = WaveEngine(settings, channels=ch, max_streams=S)
    a = eng2.process(pcm[:, :, : 7 * hop], 7, hop, input_rms=None if rms is None else rms[:, :7])
    b = eng2.process(pcm[:, :, 7 * hop:], T - 7, hop, input_rms=None if rms is None else rms[:, 7:])
    assert np.array_equal(np.concatenate([a["out"], b["out"]], axis=1), o["out"] if not device_ptrs else out)
    assert np.array_equal(np.concatenate([a["silent"], b["silent"]], axis=1), sil)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(16))
def test_gpu_wave_randomised_settings_vs_oracle(seed):
    """Differential fuzz of the chunked waveform kernel against the oracle (itself bit-exact against the reference over the
    same settings space, test_wave_oracle_randomised_settings_bit_exact_vs_compiled_reference): point pattern and silent flags
    exactly, dB values to 1e-4 dB; three streams: plain signal, full-scale / zero stretches, a silent second channel."""
    from waveform_b200 import WaveEngine

    rng = np.random.default_rng(7000 + seed)
    ch = int(rng.choice([1, 2]))
    settings = {"width": int(rng.choice([64, 200, 301, 640, 800, 1000, 1920])), "meter_buf": int(rng.choice([5, 10, 20, 50, 150, 500]))}
    if rng.uniform() < 0.5:
        settings["channel_mode"] = "stereo"
    if rng.uniform() < 0.3:
        settings["normalize_volume"] = True
    hop = int(rng.choice([97, 333, 441, 480, 800, 1024, 1600, 2000]))
    S, T = 3, 40
    pcm = synth_pcm(S, ch, T * hop, seed=seed)
    a, b = sorted(int(v) for v in rng.integers(0, T, size=2))
    pcm[1, :, a * hop: (a + (b - a) // 2) * hop] = 1.0
    pcm[1, :, (a + (b - a) // 2) * hop: b * hop] = 0.0
    pcm[2, -1] = 0.0
    rms = (0.05 + 0.2 * rng.uniform(size=(S, T))).astype(np.float32) if settings.get("normalize_volume") else None
    ref, ref_sil = _oracle_batch(settings, ch, pcm, T, hop, rms)
    cut = int(rng.integers(1, T))
    eng = WaveEngine(settings, channels=ch, max_streams=S)
    p1 = eng.process(pcm[:, :, : cut * hop], cut, hop, input_rms=None if rms is None else rms[:, :cut])
    p2 = eng.process(pcm[:, :, cut * hop:], T - cut, hop, input_rms=None if rms is None else rms[:, cut:])
    out = np.concatenate([p1["out"], p2["out"]], axis=1)
    sil = np.concatenate([p1["silent"], p2["silent"]], axis=1)
    assert np.array_equal(sil, ref_sil), (settings, ch, hop)
    lo = ref < -700.0
    assert np.array_equal(out < -700.0, lo), (settings, ch, hop)
    untouched = ref == np.float32(-758.59564)
    assert np.array_equal(out[untouched], ref[untouched])
    raw = (~lo) & (np.abs(ref) <= 1.0) & (ref == out)
    assert np.max(np.abs(out[lo] - ref[lo]), initial=0.0) < 1e-3, (settings, ch, hop)
    assert np.max(np.abs(out[~lo & ~raw] - ref[~lo & ~raw]), initial=0.0) < 1e-4, (settings, ch, hop)


@pytest.mark.gpu
def test_gpu_wave_requires_all_streams_and_reset():
    from waveform_b200 import WaveEngine, WfError

    eng = WaveEngine({"width": 256, "meter_buf": 100}, channels=1, max_streams=3)
    pcm = synth_pcm(3, 1, 4 * 800)
    with pytest.raises(WfError):
        eng.process(pcm[:2], 4, 800)        # a subset of the streams would desynchronise the shared clock
    eng.process(pcm, 4, 800)
    eng.reset()                              # hidden / capture-timeout branch: buffers := DB_MIN, m_last_silent := true
    out = eng.process(np.zeros((3, 1, 800), np.float32), 1, 800)
    assert out["out"].min() < -700.0


CHUNK_CASES = WAVE_CASES + [
    ({"width": 301, "meter_buf": 40}, 2, 97),                                       # width % 4 != 0: the scalar row path; many ticks per chunk
    ({"width": 301, "meter_buf": 40, "channel_mode": "stereo"}, 1, 97),
    ({"width": 1024, "meter_buf": 1000}, 1, 64),                                    # ~1.4 points per tick: chunks of 32 ticks, some ticks without points
    ({"width": 4096, "meter_buf": 300, "channel_mode": "stereo"}, 2, 480),          # wide buffer (opt-in shared memory)
    ({"width": 64, "meter_buf": 5, "channel_mode": "stereo", "normalize_volume": True}, 2, 2000),  # every tick replaces the whole buffer
]


@pytest.mark.gpu
@pytest.mark.parametrize("settings,ch,hop", CHUNK_CASES)
def test_gpu_wave_chunked_kernel_is_bit_identical_to_the_per_tick_kernel(settings, ch, hop, monkeypatch):
    """wave_chunk_kernel (several ticks per barrier, sliding windows over an extended buffer) against wave_kernel (the
    tick-by-tick restatement of src/source_generic.cpp:272-390): same rows, same silent flags, same state across calls —
    including input built to trip the all-zero rule (|x| == 1 -> 0.0 dBFS entries followed by zeros)."""
    from waveform_b200 import WaveEngine

    _chunk_vs_per_tick(settings, ch, hop, 5, 90, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("settings,ch,hop", [CHUNK_CASES[0], CHUNK_CASES[1], CHUNK_CASES[5]])
def test_gpu_wave_chunked_kernel_many_streams(settings, ch, hop, monkeypatch):
    """More streams than resident CTAs (148 SMs x 5): every CTA walks several streams, its shared-memory state is rebuilt per stream."""
    _chunk_vs_per_tick(settings, ch, hop, 1700, 24, monkeypatch)


def _chunk_vs_per_tick(settings, ch, hop, S, T, monkeypatch):
    from waveform_b200 import WaveEngine

    pcm, rms = _case(settings, ch, hop, T, S)
    pcm[1] = 0.0
    pcm[2, :, : 40 * hop] = 1.0          # a buffer full of exactly 0.0 dB ...
    pcm[2, :, 40 * hop: 70 * hop] = 0.0  # ... then zeros: the silent rule fires, repeatedly
    pcm[3, -1] = 0.0                     # a silent second channel (the raw m_decibels[1] of the mono branch)
    if rms is not None:
        rms = np.repeat(rms[:, :1], T, axis=1) * np.linspace(0.5, 2.0, T, dtype=np.float32)[None, :]
        rms[2] = 10.0 ** (settings.get("volume_target", -8.0) / 20.0)  # compensation of exactly... whatever log10f gives
    outs = {}
    for chunk in ("1", "0"):
        monkeypatch.setenv("WF_WAVE_CHUNK", chunk)
        eng = WaveEngine(settings, channels=ch, max_streams=S)
        a = eng.process(pcm[:, :, : 13 * hop], 13, hop, input_rms=None if rms is None else rms[:, :13])
        b = eng.process(pcm[:, :, 13 * hop:], T - 13, hop, input_rms=None if rms is None else rms[:, 13:])
        outs[chunk] = (np.concatenate([a["out"], b["out"]], axis=1), np.concatenate([a["silent"], b["silent"]], axis=1))
    assert np.array_equal(outs["1"][1], outs["0"][1])
    assert np.array_equal(outs["1"][0].view(np.uint32), outs["0"][0].view(np.uint32))
