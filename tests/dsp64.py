"""float64 references of the signal ends of the engine (dsp.cu): forward STFT, inverse STFT, the int16 output rule and the
post-mix outputs.  Each restates its operation from the definition, so that the kernels can be compared with it
elementwise at any batch size; tests/test_dsp64.py checks them against the oracle's own versions."""
import numpy as np

from oracle import nhans_oracle as O

WIN, HOP, NBIN = O.WIN, O.HOP, O.NBIN
LOG_EPS = O.LOG_EPS
_HANN = O.hann_periodic().astype(np.float64)          # the float32 window values the kernels read, exactly
_W2 = np.concatenate([_HANN * _HANN, np.zeros(3 * HOP - WIN)])
_WINV = _HANN / np.tile(_W2.reshape(3, HOP).sum(axis=0), 3)[:WIN]     # w / sum_j w^2[n mod 160 + 160 j]


def n_frames(n_samples):
    return 1 + (n_samples - WIN) // HOP if n_samples >= WIN else 0


def normalise_i16(pcm, peak=None):
    """The int16 entry's normalisation: float32(float64(pcm) * (1 / (peak + 1e-6))), the reciprocal multiply of
    stft_kernel.  peak defaults to numpy's max|pcm| (abs(-32768) wraps, so that sample never wins)."""
    pcm = np.asarray(pcm, np.int16)
    if peak is None:
        peak = O.peak_of(pcm)
    return (pcm.astype(np.float64) * (1.0 / (float(peak) + 0.000001))).astype(np.float32)


def stft64(x):
    """Frames x[160 t : 160 t + 400] of float32 samples times the periodic Hann window, rfft-400 in float64
    -> complex [T, 201]."""
    x = np.asarray(x, np.float32).astype(np.float64)
    T = n_frames(len(x))
    if T == 0:
        return np.zeros((0, NBIN), np.complex128)
    frames = np.lib.stride_tricks.as_strided(x, (T, WIN), (HOP * x.strides[0], x.strides[0]))
    return np.fft.rfft(frames * _HANN, n=WIN, axis=1)


def istft64(mag, phasor):
    """irfft-400 of mag * phasor ([T, 201] each; the imaginary parts of DC and Nyquist are ignored), the
    inverse window w / sum w^2 and overlap-add, in float64 -> (T - 1) * 160 + 400 samples."""
    T = mag.shape[0]
    if T == 0:
        return np.zeros(0, np.float64)
    frames = np.fft.irfft(np.asarray(mag, np.float64) * np.asarray(phasor, np.complex128), n=WIN, axis=1) * _WINV
    frames = np.concatenate([frames, np.zeros((T, 3 * HOP - WIN))], axis=1)
    out = np.zeros((T + 2) * HOP)
    for j in range(3):                                   # hop h sums frames h, h - 1, h - 2
        out[j * HOP:(j + T) * HOP] += frames[:, j * HOP:(j + 1) * HOP].reshape(-1)
    return out[:(T - 1) * HOP + WIN]


def i16_rule(y_f32, peak):
    """int16 output of the engine: round half to even of y * float32(peak + 1e-6), computed in float32, saturated."""
    v = np.asarray(y_f32, np.float32) * np.float32(float(peak) + 0.000001)
    return np.clip(np.rint(v), -32768, 32767).astype(np.int16)


def postmix64(den, mixed, compensate=0.0, ac=False):
    """Post-mix of one clip from its float32 denoised and mixed_processed samples: removed = mixed - den in float32,
    snr_est = sum(den^2) / sum(removed^2) in float64 (+inf when removed is all zero, including an empty clip), and
    compensated = den + removed * factor with factor = float32(snr_est / 20) (ac) or the constant, 0 when not finite.
    -> (removed, snr_est, compensated, factor)"""
    den = np.asarray(den, np.float32)
    removed = np.asarray(mixed, np.float32) - den
    e_den = float(np.sum(den.astype(np.float64) ** 2))
    e_rem = float(np.sum(removed.astype(np.float64) ** 2))
    snr = e_den / e_rem if e_rem > 0 else np.inf
    with np.errstate(over="ignore"):
        factor = np.float32(snr / 20.0) if ac else np.float32(compensate)
    if not np.isfinite(factor):
        factor = np.float32(0.0)
    return removed, snr, (den + removed * factor).astype(np.float32), factor
