"""Shared test helpers: synthetic PCM (SURVEY.md §8d) and the parity metric (DESIGN.md §Parity)."""
from __future__ import annotations

import hashlib
import json
from pathlib import Path

import numpy as np

SR = 48000
GOLDEN = Path(__file__).resolve().parent / "golden"


def synth_pcm(n_streams: int, channels: int, n_samples: int, seed: int = 0xB200, zero_frames=(), frame_len=0,
              hop=0) -> np.ndarray:
    """[n_streams, channels, n_samples] float32: 0.25*U(-1,1) + 0.5 sin(2 pi f_c n/48k) + 0.1 sin(2 pi 3.01 f_c n/48k),
    f_c = 110 * 2^((c mod 60)/12), counter-based Philox so every shard regenerates identical data."""
    out = np.empty((n_streams, channels, n_samples), dtype=np.float32)
    n = np.arange(n_samples, dtype=np.float64)
    for s in range(n_streams):
        for c in range(channels):
            idx = s * channels + c
            rng = np.random.Generator(np.random.Philox(key=seed + idx))
            fc = 110.0 * 2.0 ** ((idx % 60) / 12.0)
            x = 0.25 * rng.uniform(-1.0, 1.0, n_samples) + 0.5 * np.sin(2 * np.pi * fc * n / SR) \
                + 0.1 * np.sin(2 * np.pi * fc * 3.01 * n / SR)
            out[s, c] = x.astype(np.float32)
    for (s, t0, t1) in zero_frames:  # zero the samples covered by frames [t0, t1) of stream s
        out[s, :, t0 * hop: (t1 - 1) * hop + frame_len] = 0.0
    return out


def db_to_lin(db):
    return np.power(10.0, np.asarray(db, dtype=np.float64) / 20.0)


def parity_report(got_db, ref_db, db_min=-758.0):
    """Compare dB spectra in the LINEAR domain (what the 1e-5 relative bar of the north star is about).

    A pure per-bin relative test is meaningless for an fp32 FFT (bins far below the frame's energy carry the
    rounding noise of the big bins; the real FFTW has the same property against an fp64 DFT), so the criterion is
        |gpu - ref| <= 1e-5 * |ref| + 1e-6 * frame_peak        (linear magnitudes)
    and we also report: normwise error (max|d| / frame peak), fraction of bins inside the pure 1e-5 relative test,
    and max |d dB| over the bins within 60 dB of the frame peak.
    """
    got_db = np.asarray(got_db, dtype=np.float64)
    ref_db = np.asarray(ref_db, dtype=np.float64)
    floor_mask = (ref_db <= db_min + 1.0) | (got_db <= db_min + 1.0)
    same_floor = np.array_equal(ref_db <= db_min + 1.0, got_db <= db_min + 1.0)
    g, r = db_to_lin(got_db), db_to_lin(ref_db)
    g[floor_mask] = 0.0
    r[floor_mask] = 0.0
    peak = np.maximum(r.max(axis=-1, keepdims=True), 1e-300)
    d = np.abs(g - r)
    tol = 1e-5 * r + 1e-6 * peak
    strong = (r >= peak * 1e-3) & ~floor_mask
    return {
        "ok": bool(np.all(d <= tol) and same_floor),
        "normwise": float((d / peak).max()),
        "frac_rel_1e5": float(np.mean(d[~floor_mask] <= 1e-5 * r[~floor_mask])) if (~floor_mask).any() else 1.0,
        "max_db_strong": float(np.abs(got_db - ref_db)[strong].max()) if strong.any() else 0.0,
        "worst_excess": float((d / tol).max()),
        "same_floor": same_floor,
    }


def check_points(settings, channels, got_db, got_points):
    """Display points are a linear map of the dB spectrum (interpolation + Gaussian, src/filter.hpp:133-211): check the
    CUDA epilogue against the oracle's interpolation applied to the CUDA path's OWN dB spectrum, so that this test
    isolates the interpolation arithmetic (the spectrum itself is judged by parity_report)."""
    from oracle.oraclebind import OracleSource

    o = OracleSource(settings, channels=channels)
    exp = o.interp_of(got_db)
    d = np.abs(np.asarray(got_points, dtype=np.float64) - exp.astype(np.float64))
    scale = np.maximum(np.abs(exp).max(axis=-1, keepdims=True), 1.0)
    return float((d / scale).max())


def device_pcm(n_streams: int, channels: int, n_samples: int, seed: int = 0xB200, zero_every: int = 0, frame_len: int = 0):
    """The same signal family generated ON THE DEVICE (torch) for shapes too large for synth_pcm: noise + two sines per
    (stream, channel); with zero_every > 0 every zero_every-th aligned block of frame_len samples of a stream-dependent
    phase is digital silence, so that the silence gate runs at scale.  Returns a CUDA tensor [S, cc, ns]."""
    import torch

    dev = torch.device("cuda")
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    n = torch.arange(n_samples, device=dev, dtype=torch.float32)
    pcm = torch.empty((n_streams, channels, n_samples), device=dev, dtype=torch.float32)
    rows = n_streams * channels
    flat = pcm.view(rows, n_samples)
    chunk = max(1, (1 << 26) // max(1, n_samples))
    for r0 in range(0, rows, chunk):
        r1 = min(rows, r0 + chunk)
        idx = torch.arange(r0, r1, device=dev, dtype=torch.float32)
        fc = 110.0 * torch.pow(2.0, torch.remainder(idx, 60.0) / 12.0)
        ph = 2.0 * torch.pi * fc[:, None] * n[None, :] / SR
        x = 0.25 * (2.0 * torch.rand((r1 - r0, n_samples), device=dev, generator=g) - 1.0)
        x += 0.5 * torch.sin(ph) + 0.1 * torch.sin(3.01 * ph)
        flat[r0:r1] = x
    if zero_every > 0 and frame_len > 0:
        nb = n_samples // frame_len
        blk = pcm[:, :, : nb * frame_len].view(n_streams, channels, nb, frame_len)
        s = torch.arange(n_streams, device=dev)[:, None]
        b = torch.arange(nb, device=dev)[None, :]
        zero = ((b + 3 * s) % zero_every) == 0          # [S, nb]
        blk[zero[:, None, :].expand(n_streams, channels, nb)] = 0.0
    return pcm


def fp64_truth_db(pcm, window, window_sum, n_frames, hop, g, db_min=-758.59564):
    """Double-precision ground truth of the plain pipeline (window -> DFT -> |X| 2/sum(w) -> EMA -> dBFS) for one mono
    stream, from the SAME float32 window table (so that only the arithmetic differs): SURVEY.md §7 'both
    implementations' error vs fp64 truth'.  pcm: [samples] float32."""
    N = len(window)
    w = window.astype(np.float64)
    coef = 2.0 / float(window_sum)
    state = np.zeros(N // 2)
    out = np.empty((n_frames, N // 2))
    for t in range(n_frames):
        x = pcm[t * hop: t * hop + N].astype(np.float64) * w
        mag = np.abs(np.fft.rfft(x)[: N // 2]) * coef
        state = g * state + (1.0 - g) * mag
        with np.errstate(divide="ignore"):
            out[t] = np.where(state > 0, 20.0 * np.log10(np.maximum(state, 1e-300)), db_min)
    return out


# ---- what the compiled reference produced, stored under tests/golden/ref_*.npz by make_golden.py --reference-outputs ----
#
# Arrays the tests compare bit for bit are stored as digests; arrays compared within a tolerance are stored as a fixed
# sample of entries per row: the first and the last entry, the row's largest (so that a spectrum's frame peak is in its
# sample) and k more drawn with a seed.  Only the values and the rows' peak positions are stored; the other positions
# are drawn again when the sample is compared.

def digest(a) -> str:
    """Short content hash of an array (dtype, shape and bytes); "none" for None."""
    if a is None:
        return "none"
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:16]


def sample_columns(n: int, peaks, k: int, seed: int) -> np.ndarray:
    """[rows, k+3] positions of a sample of rows of n entries: 0, n-1, the row's peak, then k distinct positions."""
    rng = np.random.default_rng(seed)
    k = min(k, n)
    return np.array([[0, n - 1, p, *rng.choice(n, k, replace=False)] for p in peaks], dtype=np.intp)


def sample_rows(a, k: int, seed: int):
    """(values [rows, k+3], record) of a sample of a[..., n] viewed as rows of n; the record (JSON-able) lets
    take_sample() find the same positions again."""
    rows = np.asarray(a).reshape(-1, a.shape[-1])
    peaks = [int(i) for i in rows.argmax(axis=1)]
    cols = sample_columns(rows.shape[1], peaks, k, seed)
    return np.take_along_axis(rows, cols, axis=1), {"peaks": peaks, "k": k, "seed": seed, "cols": digest(cols)}


def take_sample(a, record: dict) -> np.ndarray:
    """The entries of a[..., n] at the positions of a sample_rows() sample, as [rows, k+3]."""
    rows = np.asarray(a).reshape(-1, a.shape[-1])
    cols = sample_columns(rows.shape[1], record["peaks"], record["k"], record["seed"])
    assert digest(cols) == record["cols"], "the sampled positions differ from the stored ones"
    return np.take_along_axis(rows, cols, axis=1)


class ReferenceOutputs:
    """tests/golden/ref_<name>.npz: per case, a JSON record (digests, scalars) and the sampled arrays "<case>__<key>"."""

    def __init__(self, name: str):
        self.path = GOLDEN / f"ref_{name}.npz"
        z = np.load(self.path, allow_pickle=False)
        self.meta = json.loads(str(z["meta"]))
        self.arrays = {k: z[k] for k in z.files if k != "meta"}

    def __getitem__(self, case: str) -> dict:
        rec = dict(self.meta[case])
        pre = case + "__"
        rec.update({k[len(pre):]: v for k, v in self.arrays.items() if k.startswith(pre)})
        return rec

    @staticmethod
    def save(name: str, records: dict):
        """records: {case: {key: json-able value or np.ndarray}}; ndarrays go to their own members."""
        meta, arrays = {}, {}
        for case, rec in records.items():
            meta[case] = {k: v for k, v in rec.items() if not isinstance(v, np.ndarray)}
            arrays.update({f"{case}__{k}": v for k, v in rec.items() if isinstance(v, np.ndarray)})
        np.savez_compressed(GOLDEN / f"ref_{name}.npz", meta=json.dumps(meta, sort_keys=True), **arrays)
