#!/usr/bin/env python
"""Generate golden input/output vectors from the UNMODIFIED reference compiled into oracle/_ref
(make -C oracle/ref_build).  Run in the dev container where /root/reference exists:

    python tests/golden/make_golden.py
    python tests/golden/make_golden.py --reference-outputs     # only the ref_*.npz files (see main_reference_outputs)

Each case_*.npz holds: settings (json), channels, hop, pcm [cc, samples] float32, and what the reference's
WAVSourceGeneric produced tick by tick: db [T, dch, B], points [T, dch, P] (generic interpolation path),
silent [T], plus the tables WAVSource::update() built (window, slope, rolloff, interp indices / weights / band widths).
The PCM is stored (not regenerated) so the fixtures do not depend on any RNG implementation.
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from helpers import synth_pcm  # noqa: E402
from oracle.refbind import IMPL_GENERIC, RefSource  # noqa: E402

OUT = Path(__file__).resolve().parent

CASES = {
    # BASELINE.json configs[0]: 1 mono channel, N=1024 Hann, bars mode, generic CPU path
    "c1_mono_1024_hann_bars": dict(settings={"fft_size": 1024, "window": "hann", "display_mode": "bars",
                                             "interp_mode": "catmull_rom"}, channels=1, T=12, hop=800),
    # configs[1] shape: stereo, N=4096 Blackman-Harris, dBFS + temporal smoothing, 60 fps hop
    "c2_stereo_4096_bh": dict(settings={"fft_size": 4096, "window": "blackman_harris", "channel_mode": "stereo"},
                              channels=2, T=8, hop=800),
    # configs[2] shape: mono N=2048 Hann EMA dB
    "c3_mono_2048_hann": dict(settings={"fft_size": 2048, "window": "hann"}, channels=1, T=10, hop=2048),
    # configs[3] shape (scaled down): 75 % overlap, log-frequency Lanczos curve
    "c4_mono_2048_overlap_lanczos": dict(settings={"fft_size": 2048, "window": "hann", "interp_mode": "lanczos",
                                                   "width": 400}, channels=1, T=10, hop=512),
    # everything on: slope, roll-off, fast peaks, gaussian, 2ch->mono mix, volume normalisation
    "mix_1024_all_options": dict(settings={"fft_size": 1024, "window": "hamming", "slope": 0.75, "rolloff_q": 1.5,
                                           "rolloff_rate": 9.0, "fast_peaks": True, "filter_mode": "gauss",
                                           "filter_radius": 2.0, "interp_mode": "lanczos", "width": 256,
                                           "normalize_volume": True}, channels=2, T=10, hop=512, rms=True),
    # silence gate: decay, freeze, wake-up
    "gate_1024_silence": dict(settings={"fft_size": 1024, "window": "hann", "gravity": 0.3, "floor": -40},
                              channels=1, T=40, hop=1024, silence=(4, 30)),
    # non-power-of-two size the plugin's auto mode produces at 48 kHz / 60 fps (src/source.cpp:1161-1167)
    "auto_800_tvexp": dict(settings={"fft_size": 800, "window": "blackman", "temporal_smoothing": "tv_exp_moving_avg",
                                     "gravity": 0.5, "log_scale": False, "interp_mode": "point", "width": 200},
                           channels=1, T=8, hop=800),
}


def main():
    for name, c in CASES.items():
        ref = RefSource(c["settings"], impl=IMPL_GENERIC, channels=c["channels"])
        N, T, hop = ref.fft_size, c["T"], c["hop"]
        cc = ref.capture_channels
        pcm = synth_pcm(1, cc, (T - 1) * hop + N, seed=0xB200 + len(name))[0]
        if "silence" in c:
            a, b = c["silence"]
            pcm[:, a * hop:] = 0.0
            pcm[:, b * hop: (b + 2) * hop] = 0.05
        rms = None
        if c.get("rms"):
            rms = (0.02 + 0.3 * np.random.default_rng(7).uniform(size=T)).astype(np.float32)
        r = ref.run_stft(pcm, T, hop, seconds=1.0 / 60.0, rms=rms, want_points=True, fma3=False)
        taps, weights = ref.interp_kernel()
        gk, gr, gs = ref.gauss_kernel()
        np.savez_compressed(
            OUT / f"case_{name}.npz",
            settings=json.dumps(c["settings"]), channels=c["channels"], hop=hop, n_frames=T, seconds=1.0 / 60.0,
            pcm=pcm, rms=rms if rms is not None else np.zeros(0, np.float32),
            db=r["db"], points=r["points"], silent=r["silent"],
            window=ref.window() if ref.window() is not None else np.zeros(0, np.float32),
            window_sum=np.float32(ref.window_sum),
            slope=ref.slope() if ref.slope() is not None else np.zeros(0, np.float32),
            rolloff=ref.rolloff() if ref.rolloff() is not None else np.zeros(0, np.float32),
            interp_indices=ref.interp_indices(), band_widths=ref.band_widths(),
            interp_weights=weights if weights is not None else np.zeros((0, 0), np.float32),
            gauss=gk, gauss_sum=np.float32(gs), db_min=np.float32(ref.db_min),
        )
        print(name, "N", N, "db", r["db"].shape, "points", r["points"].shape, "silent ticks", int(r["silent"].sum()))


# Level meter / RMS feed fixtures (SURVEY.md §8(f) rank 4): what the unmodified reference's tick_meter /
# update_input_rms produce tick by tick (src/source_generic.cpp:182-270, :392-403).
METER_CASES = {
    "rms_150ms_stereo": dict(kind="meter", settings={"meter_buf": 150, "rms_mode": True}, channels=2, T=50, hop=800),
    "peak_fast_100ms": dict(kind="meter", settings={"meter_buf": 100, "rms_mode": False, "fast_peaks": True}, channels=2,
                            T=50, hop=800),
    "rms_20ms_mono_nosmooth": dict(kind="meter", settings={"meter_buf": 20, "rms_mode": True, "temporal_smoothing": "none"},
                                   channels=1, T=64, hop=441),
    "rms_feed_stereo": dict(kind="rms_feed", settings={}, channels=2, T=75, hop=800),
}


def main_meter():
    for name, c in METER_CASES.items():
        T, hop, ch = c["T"], c["hop"], c["channels"]
        pcm = synth_pcm(1, ch, T * hop, seed=0xB200 + len(name))[0]
        pcm[:, (T // 2) * hop: (3 * T // 4) * hop] = 0.0
        if c["kind"] == "meter":
            ref = RefSource({"display_mode": "level_meter", **c["settings"]}, impl=IMPL_GENERIC, channels=ch)
        else:
            ref = RefSource({"normalize_volume": True, "fft_size": 1024}, impl=IMPL_GENERIC, channels=ch)
        r = ref.run_meter(pcm, T, hop)
        np.savez_compressed(OUT / f"meter_{name}.npz", kind=c["kind"], settings=json.dumps(c["settings"]), channels=ch,
                            hop=hop, n_ticks=T, pcm=pcm, db=r["db"], lin=r["lin"], silent=r["silent"], rms=r["rms"])
        print("meter", name, "window", ref.fft_size, "silent ticks", int(r["silent"].sum()), "rms[-1]", float(r["rms"][-1]))


# Waveform (oscilloscope) mode fixtures: m_decibels after every tick of the unmodified reference's tick_waveform
# (src/source_generic.cpp:272-390).
WAVE_CASES = {
    "mono_mix_800_150ms": dict(settings={"width": 800, "meter_buf": 150}, channels=2, T=30, hop=800),
    "stereo_300_50ms": dict(settings={"width": 300, "meter_buf": 50, "channel_mode": "stereo"}, channels=2, T=40, hop=441),
    "silent_200_10ms": dict(settings={"width": 200, "meter_buf": 10}, channels=1, T=40, hop=1600),
    "normalized_640_500ms": dict(settings={"width": 640, "meter_buf": 500, "channel_mode": "stereo",
                                           "normalize_volume": True}, channels=2, T=30, hop=1024),
}


def main_wave():
    for name, c in WAVE_CASES.items():
        T, hop, ch = c["T"], c["hop"], c["channels"]
        pcm = synth_pcm(1, ch, T * hop, seed=0xB200 + len(name))[0]
        pcm[:, (T // 2) * hop: (2 * T // 3) * hop] = 0.0
        rms = (0.05 + 0.2 * np.random.default_rng(5).uniform(size=T)).astype(np.float32) \
            if c["settings"].get("normalize_volume") else None
        ref = RefSource({"display_mode": "waveform", **c["settings"]}, impl=IMPL_GENERIC, channels=ch)
        r = ref.run_wave(pcm, T, hop, rms=rms)
        np.savez_compressed(OUT / f"wave_{name}.npz", settings=json.dumps(c["settings"]), channels=ch, hop=hop, n_ticks=T,
                            pcm=pcm, rms=rms if rms is not None else np.zeros(0, np.float32), out=r["out"], silent=r["silent"])
        print("wave", name, r["out"].shape, "silent ticks", int(r["silent"].sum()))


# "Not enough audio" (src/source_generic.cpp:55-61): the only way the plugin's public API produces it is audio that is
# stamped AHEAD of the tick clock (positive get_audio_sync, src/source.hpp:279-285): the tick then wants delay + N samples
# and the ring, trimmed to N by the earlier in-sync packets, needs a few ticks to refill.  During those ticks the channel
# `continue`s while m_last_silent is false, so the stale dB values are pushed through dbfs() again (SURVEY appendix A quirk).
# The fixture stores the sample stream the ticks see (`pcm`, with the N start-up zeros update() leaves in the ring) and,
# per engine call, the offset of frame 0, the number of ticks and the skip mask; frame t of a call = pcm[offset + t*hop ...+N).
STALL_CASES = {
    "2048_avsync_jump": dict(settings={"fft_size": 2048, "window": "hann"}, channels=1, T=14, hop=800, jump_at=5,
                             ahead_ms=50),
    "1024_stereo_jump_rolloff": dict(settings={"fft_size": 1024, "window": "hamming", "channel_mode": "stereo",
                                               "rolloff_q": 1.0, "rolloff_rate": 6.0}, channels=2, T=16, hop=512,
                                     jump_at=6, ahead_ms=32),
}


def main_stall():
    for name, c in STALL_CASES.items():
        ref = RefSource(c["settings"], impl=IMPL_GENERIC, channels=c["channels"])
        N, T, hop, J = ref.fft_size, c["T"], c["hop"], c["jump_at"]
        cc = ref.capture_channels
        audio = synth_pcm(1, cc, T * hop, seed=0xB200 + len(name))[0]
        delay = int(round(c["ahead_ms"] * 1e-3 * 48000))
        assert delay % hop == 0, "keep the delayed frames on the hop grid"
        dbs, sil = [], []
        for t in range(T):
            ref.advance(hop / 48000.0)
            ref.push(audio[0, t * hop:(t + 1) * hop], audio[1, t * hop:(t + 1) * hop] if cc > 1 else None,
                     ts_adjust_ns=0 if t < J else int(c["ahead_ms"] * 1e6))
            ref.tick(1.0 / 60.0)
            dbs.append(np.stack([ref.decibels(ch) for ch in range(ref.display_channels)]))
            sil.append(ref.last_silent)
        db = np.stack(dbs)
        # what the ticks saw: ring = [N zeros][audio]; in sync, tick t takes the newest N samples = ring[(t+1)*hop ...);
        # delayed, the oldest N of the newest delay+N = ring[(t+1)*hop - delay ...), once the ring holds that much
        ring = np.concatenate([np.zeros((cc, N), np.float32), audio], axis=1)
        k = delay // hop
        calls = [dict(offset=hop, n_frames=J, skip=[0] * J),
                 dict(offset=(J + 1 - k) * hop, n_frames=T - J, skip=[1] * (k - 1) + [0] * (T - J - k + 1))]
        skipped = [t for t in range(J, J + k - 1)]  # the first delayed push already counts towards the refill
        assert all((db[t] <= ref.db_min + 1).all() for t in skipped) and (db[J + k - 1] > ref.db_min + 1).any()
        np.savez_compressed(OUT / f"stall_{name}.npz", settings=json.dumps(c["settings"]), channels=c["channels"], hop=hop,
                            n_frames=T, seconds=1.0 / 60.0, pcm=ring, calls=json.dumps(calls), db=db,
                            silent=np.array(sil, np.uint8), db_min=np.float32(ref.db_min))
        print("stall", name, "N", N, "skipped ticks", skipped, "db at first skipped tick: max", float(db[J].max()))


# What the tests that compare with the reference on their own inputs need from it (test_oracle_vs_reference, test_wave,
# test_meter, test_gpu_host): each of those modules builds its inputs and runs the reference in reference_records(); the
# result goes to ref_<name>.npz, read back by helpers.ReferenceOutputs.
REFERENCE_OUTPUTS = {"oracle_vs_reference": "test_oracle_vs_reference", "wave": "test_wave", "meter": "test_meter",
                     "gpu_host": "test_gpu_host"}


def main_reference_outputs():
    import importlib

    from helpers import ReferenceOutputs

    for name, module in REFERENCE_OUTPUTS.items():
        recs = importlib.import_module(module).reference_records()
        ReferenceOutputs.save(name, recs)
        print("reference outputs", name, len(recs), "cases", (OUT / f"ref_{name}.npz").stat().st_size, "bytes")


if __name__ == "__main__":
    import sys
    if "--reference-outputs" in sys.argv:
        main_reference_outputs()
        sys.exit(0)
    if "--stall-only" in sys.argv:
        main_stall()
        sys.exit(0)
    if "--meter-only" not in sys.argv and "--wave-only" not in sys.argv:
        main()
    if "--wave-only" not in sys.argv:
        main_meter()
    if "--meter-only" not in sys.argv:
        main_wave()
    if "--meter-only" not in sys.argv and "--wave-only" not in sys.argv:
        main_stall()
