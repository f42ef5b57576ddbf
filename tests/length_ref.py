"""librosa's Griffin-Lim loop with ``length=``, composed from the restated oracle's own ``istft`` (which restates
librosa's ``length`` crop / zero padding) and ``stft``.  librosa hands ``length`` to every istft of
``librosa.griffinlim``, the loop's included, so the re-analysed signal has exactly ``length`` samples; with
``length=None`` this is ``oracle.librosa_restated.griffinlim`` step for step.

It lives here rather than as a ``length`` argument of the oracle's ``griffinlim_step`` / ``griffinlim`` /
``mel_to_audio`` so that the oracle the existing parity tests measure against stays byte for byte what it was.
tests/test_oracle_length.py pins it to the oracle (bit-identical at ``length=None`` and at ``length=(T-1)*256``) and to
torchaudio's independent griffinlim(length=...)."""
import numpy as np

from oracle import librosa_restated as lr


def griffinlim_step(angles, tprev, S, *, length=None, momentum=0.99):
    """One body of the loop (hop 256, n_fft 1024).  Returns (new_angles, rebuilt, inverse)."""
    eps = np.finfo(np.float32).tiny
    inverse = lr.istft(angles, hop_length=256, n_fft=1024, dtype=np.float32, length=length)
    rebuilt = lr.stft(inverse, n_fft=1024, hop_length=256)      # looked up at call time: tests may swap it
    new = rebuilt.copy()
    if tprev is not None:
        new -= (momentum / (1 + momentum)) * tprev
    new /= np.abs(new) + eps
    new *= S
    return new, rebuilt, inverse


def griffinlim(S, *, n_iter, init_phase, length=None, momentum=0.99):
    S = np.asarray(S, dtype=np.float32)
    angles = np.empty(S.shape, dtype=np.complex64)
    angles[:] = lr.phasor(init_phase)
    angles *= S
    tprev = None
    for _ in range(n_iter):
        angles, tprev, _ = griffinlim_step(angles, tprev, S, length=length, momentum=momentum)
    return lr.istft(angles, hop_length=256, n_fft=1024, dtype=np.float32, length=length)
