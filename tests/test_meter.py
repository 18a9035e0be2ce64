"""Level meter (tick_meter) and RMS feed (update_input_rms): SURVEY.md §8(f) rank 4 / §8(a) a9.

CPU: the oracle restatement (oracle/wf_oracle_meter.c) bit-exact against what the compiled reference produced
(tests/golden/ref_meter.npz, digests of every tick's values) and against the committed golden fixtures.  GPU: the CUDA
path (wf_meter_* through the C-ABI) against the oracle — bit-exact for peak values and silent flags, 1e-5 relative for
RMS values: an fp32 sum of W squares depends on the order of the additions — the reference's own AVX path (src/source_avx.cpp:257-268, 16 partial sums) differs from its generic path (ring order,
one accumulator) by 1.8e-6 on this data; the CUDA path sums 256-sample blocks.
"""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import pytest

from helpers import ReferenceOutputs, digest, synth_pcm

GOLD = sorted((Path(__file__).parent / "golden").glob("meter_*.npz"))

METER_CASES = [
    ({"meter_buf": 150, "rms_mode": True}, 2, 800),
    ({"meter_buf": 100, "rms_mode": False, "fast_peaks": True}, 2, 800),
    ({"meter_buf": 20, "rms_mode": True, "temporal_smoothing": "none"}, 1, 441),
    ({"meter_buf": 50, "rms_mode": False, "temporal_smoothing": "tv_exp_moving_avg", "gravity": 0.4}, 2, 1024),
    ({"meter_buf": 10, "rms_mode": True, "gravity": 0.2, "floor": -40}, 1, 1601),  # hop > window
]


def _case_pcm(ch, T, hop, S=1):
    pcm = synth_pcm(S, ch, T * hop)
    pcm[:, :, (T // 2) * hop: (3 * T // 4) * hop] = 0.0  # a silent stretch: decay, m_last_silent, wake-up
    return pcm


# ---- CPU: oracle pinned to the reference -------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ref():
    return ReferenceOutputs("meter")


@pytest.mark.parametrize("settings,ch,hop", METER_CASES)
def test_meter_oracle_is_bit_exact_vs_compiled_reference(settings, ch, hop, ref):
    from oracle.oraclebind import OracleMeter

    T = 60
    pcm = _case_pcm(ch, T, hop)[0]
    rec = ref[f"case{METER_CASES.index((settings, ch, hop))}"]
    assert digest(pcm) == rec["inputs"], "inputs differ from the ones the reference was run on"
    o = OracleMeter(settings, channels=ch)
    assert o.window == rec["window"]
    out = o.run(pcm, T, hop)
    for key in ("db", "lin", "silent"):
        assert digest(out[key]) == rec[key], key
    assert out["silent"].sum() > 0 or settings.get("floor", -65) < -60


def _random_case(seed):
    rng = np.random.default_rng(9000 + seed)
    ch = int(rng.choice([1, 2]))
    settings = {"meter_buf": int(rng.choice([5, 10, 20, 50, 100, 150, 300])), "rms_mode": bool(rng.uniform() < 0.5),
                "temporal_smoothing": str(rng.choice(["none", "exp_moving_avg", "tv_exp_moving_avg"])),
                "gravity": float(rng.choice([0.2, 0.4, 0.65, 0.9])), "floor": int(rng.choice([-30, -40, -65])),
                "fast_peaks": bool(rng.uniform() < 0.4)}
    hop = int(rng.choice([97, 441, 480, 800, 801, 1024, 1601]))
    T = 50
    pcm = _case_pcm(ch, T, hop)[0] * np.float32(rng.choice([1.0, 0.1, 0.01]))
    return settings, ch, hop, T, pcm


@pytest.mark.parametrize("seed", range(30))
def test_meter_oracle_randomised_settings_bit_exact_vs_compiled_reference(seed, ref):
    """Differential fuzz of the level-meter oracle against the unmodified reference (generic path): random window, mode,
    smoothing, gravity, floor, packet size and channel count, with a silent stretch."""
    from oracle.oraclebind import OracleMeter

    settings, ch, hop, T, pcm = _random_case(seed)
    rec = ref[f"random{seed}"]
    assert digest(pcm) == rec["inputs"], "inputs differ from the ones the reference was run on"
    o = OracleMeter(settings, channels=ch)
    assert o.window == rec["window"]
    out = o.run(pcm, T, hop)
    for key in ("db", "lin", "silent"):
        assert digest(out[key]) == rec[key], (key, settings, hop)


@pytest.mark.parametrize("ch", [1, 2])
def test_rms_feed_oracle_is_bit_exact_vs_compiled_reference(ch, ref):
    from oracle.oraclebind import OracleMeter

    T, hop = 90, 800
    pcm = _case_pcm(ch, T, hop)[0]
    rec = ref[f"rms_feed{ch}"]
    assert digest(pcm) == rec["inputs"], "inputs differ from the ones the reference was run on"
    out = OracleMeter({}, channels=ch).run(pcm, T, hop, meter=False, rms=True)["rms"]
    assert digest(out) == rec["rms"]


def reference_records():
    """What the compiled reference's tick_meter / update_input_rms (oracle/_ref) produced for each case above, as digests;
    tests/golden/make_golden.py stores them."""
    from oracle import refbind

    recs = {}
    cases = [(f"case{i}", (s, c, h, 60, _case_pcm(c, 60, h)[0])) for i, (s, c, h) in enumerate(METER_CASES)] \
        + [(f"random{seed}", _random_case(seed)) for seed in range(30)]
    for name, (settings, ch, hop, T, pcm) in cases:
        r = refbind.RefSource({"display_mode": "level_meter", **settings}, channels=ch)
        out = r.run_meter(pcm, T, hop)
        recs[name] = {"inputs": digest(pcm), "window": r.fft_size, **{k: digest(out[k]) for k in ("db", "lin", "silent")}}
    for ch in (1, 2):
        T, hop = 90, 800
        pcm = _case_pcm(ch, T, hop)[0]
        r = refbind.RefSource({"normalize_volume": True, "fft_size": 1024}, channels=ch)
        recs[f"rms_feed{ch}"] = {"inputs": digest(pcm), "rms": digest(r.run_meter(pcm, T, hop)["rms"])}
    return recs


@pytest.mark.parametrize("path", GOLD, ids=[p.stem for p in GOLD])
def test_meter_oracle_against_reference_golden_vectors(path):
    from oracle.oraclebind import OracleMeter

    z = np.load(path, allow_pickle=False)
    settings = json.loads(str(z["settings"]))
    ch, T, hop = int(z["channels"]), int(z["n_ticks"]), int(z["hop"])
    o = OracleMeter(settings, channels=ch)
    if str(z["kind"]) == "rms_feed":
        assert np.array_equal(o.run(z["pcm"], T, hop, meter=False, rms=True)["rms"], z["rms"])
    else:
        out = o.run(z["pcm"], T, hop)
        assert np.array_equal(out["db"], z["db"]) and np.array_equal(out["lin"], z["lin"])
        assert np.array_equal(out["silent"], z["silent"])


def test_meter_abi_symbols_and_config_defaults():
    """No GPU needed: the library exports the meter entry points and the defaults are the plugin's."""
    from waveform_b200.engine import EXPORTS, WfMeterConfig, load_library
    import ctypes as C

    L = load_library()
    for name in EXPORTS:
        assert hasattr(L, name), name
    c = WfMeterConfig()
    L.wf_meter_config_init(C.byref(c))
    assert (c.struct_size, c.meter_ms, c.mode, c.floor_db) == (C.sizeof(WfMeterConfig), 150, 1, -65)
    assert abs(c.gravity - 0.65) < 1e-7


# ---- GPU: the CUDA path against the oracle ---------------------------------------------------------------------

def _oracle_meter_batch(settings, ch, pcm, T, hop, **kw):
    from oracle.oraclebind import OracleMeter

    outs = [OracleMeter(settings, channels=ch).run(pcm[s], T, hop, **kw) for s in range(pcm.shape[0])]
    return {k: np.stack([o[k] for o in outs]) for k in outs[0] if outs[0][k] is not None}


RMS_TOL = 1e-5  # see the module docstring


def _close(a, b, rel):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(b), 1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("device_ptrs", [False, True])
@pytest.mark.parametrize("settings,ch,hop", METER_CASES)
def test_gpu_meter_parity_vs_oracle(settings, ch, hop, device_ptrs):
    from waveform_b200 import MeterEngine

    S, T = 5, 48
    pcm = _case_pcm(ch, T, hop, S=S)
    ref = _oracle_meter_batch(settings, ch, pcm, T, hop)
    eng = MeterEngine(settings, channels=ch, max_streams=S)
    if device_ptrs:
        import torch
        out = {k: v.cpu().numpy() for k, v in eng.process(torch.from_numpy(pcm).cuda(), T, hop).items()}
    else:
        out = eng.process(pcm, T, hop)
    assert np.array_equal(out["silent"], ref["silent"])
    if settings.get("rms_mode", True):
        assert _close(out["lin"], ref["lin"], RMS_TOL)
        fin = ref["db"] > -700
        assert np.array_equal(fin, out["db"] > -700)
        assert np.max(np.abs(out["db"][fin] - ref["db"][fin])) < 2e-4  # dB (1e-5 relative = 8.7e-5 dB)
    else:
        assert np.array_equal(out["lin"], ref["lin"])  # max and the EMA are exact
        assert np.max(np.abs(out["db"] - ref["db"])) < 1e-4
    assert eng.launch_count >= 1  # one-pass kernel (hop divides the window) or the three-kernel path


@pytest.mark.gpu
def test_gpu_meter_state_continues_across_calls_and_reset():
    from waveform_b200 import MeterEngine

    settings, ch, hop, S, T = {"meter_buf": 100, "rms_mode": True}, 2, 800, 3, 40
    pcm = _case_pcm(ch, T, hop, S=S)
    whole = MeterEngine(settings, channels=ch, max_streams=S).process(pcm, T, hop)
    eng = MeterEngine(settings, channels=ch, max_streams=S)
    a = eng.process(pcm[:, :, : 3 * hop], 3, hop)          # 3 ticks: shorter than the ring (history path)
    b = eng.process(pcm[:, :, 3 * hop:], T - 3, hop)
    for k in ("silent",):
        assert np.array_equal(np.concatenate([a[k], b[k]], axis=1), whole[k])
    assert _close(np.concatenate([a["lin"], b["lin"]], axis=1), whole["lin"], RMS_TOL)
    # capture-timeout branch: ring zeroed, m_meter_buf = 0 -> the next tick of silence reports DB_MIN and stays silent
    from oracle.oraclebind import OracleMeter
    eng.reset()
    z = np.zeros((S, ch, 2 * hop), np.float32)
    z[:, :, hop:] = 0.25
    out = eng.process(z, 2, hop)
    o = OracleMeter(settings, channels=ch)
    o.run(pcm[0], T, hop)
    o.reset()
    ref = o.run(z[0], 2, hop)
    assert np.array_equal(out["silent"][0], ref["silent"])
    assert _close(out["lin"][0], ref["lin"], RMS_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("ch", [1, 2])
def test_gpu_rms_feed_parity_and_feeds_volume_normalisation(ch):
    """wf_meter INPUT_RMS reproduces m_input_rms tick by tick; its output is what wf_batch.input_rms expects."""
    from waveform_b200 import Engine, MeterEngine
    from waveform_b200.engine import METER_INPUT_RMS

    S, T, hop = 4, 70, 800
    pcm = _case_pcm(ch, T, hop, S=S)
    ref = _oracle_meter_batch({}, ch, pcm, T, hop, meter=False, rms=True)["rms"]
    feed = MeterEngine({}, channels=ch, max_streams=S, mode=METER_INPUT_RMS)
    assert feed.window == 48000
    got = feed.process(pcm, T, hop)["rms"]
    assert _close(got, ref, RMS_TOL)
    # downstream: the spectrum engine accepts it as its per-tick input_rms
    N = 1024
    Tf = (T * hop - N) // hop + 1
    eng = Engine({"fft_size": N, "normalize_volume": True}, channels=ch, max_streams=S)
    out = eng.process(pcm, Tf, hop, input_rms=got[:, :Tf])
    assert np.isfinite(out["db"][:, :, :, 1:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["rms", "peak", "feed"])
def test_gpu_meter_one_pass_path_carries_block_partials(mode, monkeypatch):
    """The one-pass kernel (hop divides the window) keeps the ring's block partials across calls instead of re-reading the
    ring; a hop change, a call on a subset of the streams and a reset fall back to reducing the ring.  Every sequence of
    calls must equal the three-kernel path (WF_METER_FUSED=0) on the same calls, and the oracle."""
    from waveform_b200 import MeterEngine
    from waveform_b200.engine import METER_INPUT_RMS

    settings = {"meter_buf": 100, "rms_mode": mode != "peak"}
    eng_mode = METER_INPUT_RMS if mode == "feed" else None
    ch, S = 2, 6
    plan = [(800, 7, slice(0, S)), (800, 3, slice(0, S)), (800, 5, slice(2, 5)), (800, 9, slice(0, S)),
            (400, 6, slice(0, S)), (400, 20, slice(0, S)), (800, 4, slice(0, S))]
    total = sum(h * t for h, t, _ in plan)
    pcm = synth_pcm(S, ch, total, seed=3)
    pcm[:, :, total // 3: total // 2] = 0.0
    outs = {}
    for name, env in (("fused", "1"), ("general", "0")):
        monkeypatch.setenv("WF_METER_FUSED", env)
        eng = MeterEngine(settings, channels=ch, max_streams=S, mode=eng_mode)
        pos, res = 0, []
        for i, (hop, T, sl) in enumerate(plan):
            x = np.ascontiguousarray(pcm[sl, :, pos: pos + hop * T])
            res.append(eng.process(x, T, hop, first_stream=sl.start))
            if sl.start == 0 and sl.stop == S:
                pos += hop * T     # (the subset call re-feeds a stretch the other streams have not seen: fine, both paths do)
            if i == 3:
                eng.reset(1, 2)
        outs[name] = res
    for a, b in zip(outs["fused"], outs["general"]):
        for k in a:
            if k == "silent":
                assert np.array_equal(a[k], b[k])
            else:
                fin = np.isfinite(b[k]) & (b[k] > -700)
                assert _close(a[k][fin], b[k][fin], 2 * RMS_TOL), k
