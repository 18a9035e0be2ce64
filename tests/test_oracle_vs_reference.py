"""The oracle against the UNMODIFIED reference (oracle/ref_build compiles it into oracle/_ref/libwaveform_ref.so), on fresh
inputs — including the AVX2 path the plugin really executes.  What the reference produced is stored in
tests/golden/ref_oracle_vs_reference.npz (reference_records() below, run by tests/golden/make_golden.py): tables, silent
flags and the DB_MIN pattern as digests, spectra and display points as a fixed sample of entries."""
import numpy as np
import pytest

from helpers import ReferenceOutputs, digest, parity_report, sample_rows, synth_pcm, take_sample
from oracle.oraclebind import OracleSource

NAME = "oracle_vs_reference"
CASES = [
    ({"fft_size": 1024, "window": "hann", "display_mode": "bars", "interp_mode": "catmull_rom"}, 1),
    ({"fft_size": 4096, "window": "blackman_harris", "channel_mode": "stereo"}, 2),
    ({"fft_size": 2048, "window": "hann"}, 1),
    ({"fft_size": 2048, "window": "hamming", "slope": 0.5, "rolloff_q": 1.0, "rolloff_rate": 6.0, "fast_peaks": True}, 2),
    ({"fft_size": 8192, "window": "blackman", "interp_mode": "lanczos", "filter_mode": "gauss", "filter_radius": 2.5}, 2),
    ({"fft_size": 800, "window": "power_of_sine", "sine_exponent": 3, "temporal_smoothing": "tv_exp_moving_avg",
      "gravity": 0.4, "log_scale": False, "interp_mode": "point"}, 1),
    ({"fft_size": 2048, "window": "none", "temporal_smoothing": "none", "display_mode": "bars", "interp_mode": "point",
      "normalize_volume": True}, 2),
    ({"fft_size": 1024, "display_mode": "bars", "interp_mode": "lanczos", "bar_width": 4, "bar_gap": 1,
      "filter_mode": "gauss", "mirror_freq_axis": True}, 2),
    ({"fft_size": 16384, "window": "hann"}, 1),
    ({"fft_size": 1024, "channel_mode": "stereo", "gravity": 0.2, "floor": -30}, 2),
]
DB_SAMPLES, POINT_SAMPLES = 192, 96  # drawn entries per case, at least one per frame and channel besides the fixed three


@pytest.fixture(scope="module")
def ref():
    return ReferenceOutputs(NAME)


@pytest.mark.parametrize("settings,channels", CASES)
def test_oracle_matches_compiled_reference(settings, channels, ref):
    _check(ref[f"case{CASES.index((settings, channels))}"], settings, channels)


def _random_case(seed):
    rng = np.random.default_rng(4000 + seed)
    N = int(rng.choice([128, 512, 1024, 2048, 4096, 8192, 800, 720, 1600, 1920, 1456, 352, 2000, 4160, 1088]))
    mode = str(rng.choice(["mono", "mono", "stereo"]))
    channels = 2 if mode == "stereo" or rng.uniform() < 0.25 else 1
    settings = {"fft_size": N, "channel_mode": mode,
                "window": str(rng.choice(["none", "hann", "hamming", "blackman", "blackman_harris", "power_of_sine"])),
                "temporal_smoothing": str(rng.choice(["none", "exp_moving_avg", "exp_moving_avg", "tv_exp_moving_avg"])),
                "gravity": float(rng.choice([0.2, 0.5, 0.65, 0.9])), "floor": int(rng.choice([-30, -45, -65])),
                "display_mode": str(rng.choice(["curve", "curve", "bars"])),
                "interp_mode": str(rng.choice(["point", "lanczos", "catmull_rom"])),
                "log_scale": bool(rng.uniform() < 0.8)}
    if settings["window"] == "power_of_sine":
        settings["sine_exponent"] = int(rng.choice([1, 2, 3, 4]))
    if rng.uniform() < 0.3:
        settings.update(slope=float(rng.choice([0.25, 1.0])), fast_peaks=bool(rng.uniform() < 0.5))
    if rng.uniform() < 0.3:
        settings.update(rolloff_q=1.0, rolloff_rate=float(rng.choice([3.0, 9.0])))
    if rng.uniform() < 0.3:
        settings.update(filter_mode="gauss", filter_radius=float(rng.choice([1.5, 2.5])))
    if rng.uniform() < 0.2:
        settings["normalize_volume"] = True
    if settings["display_mode"] == "bars" and rng.uniform() < 0.5:
        settings.update(bar_width=int(rng.choice([2, 4, 24])), bar_gap=int(rng.choice([0, 1, 6])))
    hop_div = int(rng.choice([1, 2, 4]))
    return settings, channels, dict(T=int(rng.choice([6, 14, 30])), hop_div=hop_div, seed=seed)


@pytest.mark.parametrize("seed", range(40))
def test_randomised_settings_oracle_vs_compiled_reference(seed, ref):
    """Differential fuzz of the oracle against the unmodified reference over the settings space the GPU fuzz
    (tests/test_gpu_scale.py::test_randomised_configs_against_oracle) draws from, plus the display options: every table bit for bit,
    every tick's spectrum within the parity criterion, silent flags and points."""
    settings, channels, kw = _random_case(seed)
    _check(ref[f"random{seed}"], settings, channels, **kw)


def _inputs(settings, N, cc, T=30, hop_div=2, seed=11):
    hop = N // hop_div
    x = synth_pcm(1, cc, (T - 1) * hop + N, seed=seed)[0]
    x[:, 6 * hop: 6 * hop + 4 * N] = 0
    if cc == 2:
        x[1, 12 * hop:] = 0  # one channel goes silent: exercises the stale-dB quirk
    rms = (0.05 + 0.3 * np.random.default_rng(1).uniform(size=T)).astype(np.float32) if settings.get("normalize_volume") else None
    return x, hop, rms


def _observe(src, settings, N, cc, T=30, hop_div=2, seed=11):
    """What the comparison looks at, from a reference RefSource or an OracleSource (the same method names)."""
    x, hop, rms = _inputs(settings, N, cc, T, hop_div, seed)
    r = src.run_stft(x, T, hop, rms=rms, want_points=True)
    taps, weights = src.interp_kernel()
    obs = {name: getattr(src, name)() for name in ("window", "slope", "rolloff", "interp_indices")}
    obs.update(inputs=digest(x) + digest(rms), window_sum=src.window_sum, taps=taps, interp_weights=weights,
               db=r["db"], silent=r["silent"], points=r["points"])
    return obs


def _record(obs, db_min, seed):
    rows = obs["db"].shape[0] * obs["db"].shape[1]
    rec = {k: digest(obs[k]) for k in ("window", "slope", "rolloff", "interp_indices", "interp_weights", "silent")}
    rec.update(inputs=obs["inputs"], window_sum=obs["window_sum"], taps=obs["taps"], floor=digest(obs["db"] <= db_min + 1.0))
    rec["db"], rec["db_sample"] = sample_rows(obs["db"], max(1, DB_SAMPLES // rows), seed)
    rec["points"], rec["points_sample"] = sample_rows(obs["points"], max(1, POINT_SAMPLES // rows), seed + 1)
    return rec


def _check(rec, settings, channels, **kw):
    orc = OracleSource(settings, channels=channels)
    N, cc = 2 * orc.bins, orc.cfg.capture_channels
    assert (N, cc) == (rec["fft_size"], rec["capture_channels"])
    obs = _observe(orc, settings, N, cc, **kw)
    assert obs["inputs"] == rec["inputs"], "inputs differ from the ones the reference was run on"
    for name in ("window", "slope", "rolloff", "interp_indices", "interp_weights"):
        assert digest(obs[name]) == rec[name], name
    assert obs["window_sum"] == rec["window_sum"] and obs["taps"] == rec["taps"]
    rep = parity_report(take_sample(obs["db"], rec["db_sample"]), rec["db"], db_min=orc.db_min)
    assert rep["ok"] and rep["normwise"] < 1e-6, rep
    assert digest(obs["db"] <= orc.db_min + 1.0) == rec["floor"], "DB_MIN pattern"
    assert digest(obs["silent"]) == rec["silent"]
    d = np.abs(take_sample(obs["points"], rec["points_sample"]).astype(np.float64) - rec["points"])
    assert d.max() < 5e-3 and np.median(d) < 1e-4


def test_avx2_path_is_within_the_same_tolerance(ref):
    """What the plugin runs on any recent x86 (WAVSourceAVX2, FMA EMA, sqrt(fma)) is held to the same parity criterion as
    the generic path (the parity target): the oracle against both."""
    s = {"fft_size": 2048, "window": "hann"}
    x = synth_pcm(1, 1, 20 * 2048, seed=5)[0]
    o = OracleSource(s, channels=1).run_stft(x, 20, 2048)["db"]
    rec = ref["avx2"]
    assert rec["inputs"] == digest(x)
    for impl in ("generic", "avx2"):
        rep = parity_report(take_sample(o, rec[impl + "_sample"]), rec[impl], db_min=-758.59564)
        assert rep["ok"], (impl, rep)
        assert digest(o <= -758.59564 + 1.0) == rec[impl + "_floor"], impl


def test_av_sync_offset_selects_older_frame(ref):
    """Positive audio/video delay: tick_spectrum takes the OLDEST N of the last delay+N samples
    (src/source_generic.cpp:50-59)."""
    s = {"fft_size": 1024, "window": "hann", "temporal_smoothing": "none"}
    N = 1024
    x = synth_pcm(1, 1, 4 * N, seed=9)[0]
    rec = ref["av_sync"]
    assert rec["inputs"] == digest(x)
    o = OracleSource(s, channels=1)
    o.tick([x[0, -N:]])
    assert parity_report(rec["latest"], o.decibels(0))["ok"]


PX_CASES = [
    ({"fft_size": 1024, "display_mode": "curve", "interp_mode": "lanczos", "height": 300}, 1),
    ({"fft_size": 2048, "display_mode": "bars", "interp_mode": "catmull_rom", "rounded_caps": True, "min_bar_height": 5,
      "bar_width": 10, "bar_gap": 2}, 1),
    ({"fft_size": 1024, "display_mode": "curve", "channel_mode": "stereo", "channel_spacing": 20, "mirror_freq_axis": True,
      "filter_mode": "gauss", "height": 400}, 2),
    ({"fft_size": 1024, "display_mode": "bars", "channel_mode": "stereo", "channel_spacing": 10, "rounded_caps": True,
      "mirror_freq_axis": True, "interp_mode": "point"}, 2),
]


@pytest.mark.parametrize("settings,channels", PX_CASES)
def test_display_stage_matches_reference_render(settings, channels, ref):
    """dB -> pixel lerp/clamp, mirroring and (miny, minpos): the oracle against WAVSource::render() itself
    (src/source.cpp:1346-1565 run verbatim behind the fake graphics API)."""
    rec = ref[f"px{PX_CASES.index((settings, channels))}"]
    orc = OracleSource(settings, channels=channels)
    N, T, cc = 2 * orc.bins, 6, orc.cfg.capture_channels
    x = synth_pcm(1, cc, T * N, seed=4)[0]
    assert rec["inputs"] == digest(x)
    for t in range(T):
        orc.tick([x[c, t * N:(t + 1) * N] for c in range(cc)])
    px, miny, minpos = orc.render_pixels()
    assert px.shape[0] == rec["render"].shape[0]
    assert np.abs(take_sample(px, rec["render_sample"]) - rec["render"]).max() < 5e-4
    # fed with the reference's own m_decibels only the interpolation's summation order differs: on an AVX machine
    # render() takes apply_interp_filter_fma3 (src/source.cpp:1383-1387), the oracle restates the generic template
    px2, _ = orc.pixels_of(rec["decibels"])
    assert np.abs(take_sample(px2, rec["render_sample"]) - rec["render"]).max() < 1e-4


def reference_records():
    """Run the compiled reference (oracle/_ref) on every case above; tests/golden/make_golden.py stores the result."""
    from oracle import refbind

    recs = {}
    for name, settings, channels, kw in [(f"case{i}", s, c, {}) for i, (s, c) in enumerate(CASES)] + \
            [(f"random{seed}",) + _random_case(seed) for seed in range(40)]:
        r = refbind.RefSource(settings, impl=refbind.IMPL_GENERIC, channels=channels)
        N, cc = r.fft_size, r.capture_channels
        recs[name] = dict(_record(_observe(r, settings, N, cc, **kw), r.db_min, seed=len(recs)),
                          fft_size=N, capture_channels=cc)

    s = {"fft_size": 2048, "window": "hann"}
    x = synth_pcm(1, 1, 20 * 2048, seed=5)[0]
    recs["avx2"] = {"inputs": digest(x)}
    for impl, which in (("generic", refbind.IMPL_GENERIC), ("avx2", refbind.IMPL_AVX2)):
        db = refbind.RefSource(s, impl=which, channels=1).run_stft(x, 20, 2048)["db"]
        recs["avx2"][impl], recs["avx2"][impl + "_sample"] = sample_rows(db, DB_SAMPLES // 20, seed=5)
        recs["avx2"][impl + "_floor"] = digest(db <= -758.59564 + 1.0)

    s = {"fft_size": 1024, "window": "hann", "temporal_smoothing": "none", "audio_sync_offset": 0}
    N = 1024
    x = synth_pcm(1, 1, 4 * N, seed=9)[0]
    r = refbind.RefSource(s, impl=refbind.IMPL_GENERIC, channels=1)
    r.advance(4 * N / 48000)
    r.push(x[0])                      # packet ends "now"
    r.tick()
    recs["av_sync"] = {"inputs": digest(x), "latest": r.decibels(0)}

    for case, (settings, channels) in enumerate(PX_CASES):
        r = refbind.RefSource(settings, impl=refbind.IMPL_GENERIC, channels=channels)
        N, T = r.fft_size, 6
        x = synth_pcm(1, r.capture_channels, T * N, seed=4)[0]
        for t in range(T):
            r.advance(N / 48000)
            r.push(x[0, t * N:(t + 1) * N], x[1, t * N:(t + 1) * N] if r.capture_channels > 1 else None)
            r.tick()
        r.render()
        render = np.stack([r.render_buf(c) for c in range(r.display_channels)])
        values, sample = sample_rows(render, 256, seed=case)
        recs[f"px{case}"] = {"inputs": digest(x), "render": values, "render_sample": sample,
                             "decibels": np.stack([r.decibels(c) for c in range(r.display_channels)])}
    return recs
