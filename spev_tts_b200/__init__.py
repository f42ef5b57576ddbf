"""spev_tts_b200 -- B200-native (sm_100a) spectral hot path for SPEV-TTS.

Drop-in surface (reference call sites in ``/root/reference/spev_real_metrics.py``):
  melspectrogram / logmel   <- librosa.feature.melspectrogram + log/clip      (:363-367)
  mel_to_audio / Vocoder    <- Vocoder.infer Griffin-Lim branch                (:725-733)
  LengthRegulator           <- class LengthRegulator                           (:122-146)
  duration_rule             <- clamp((exp(ld)-1)*d,0,500).round().long()       (:215)
  bucketize_embed           <- torch.bucketize + nn.Embedding (north-star; no in-tree site)

Everything dispatches to ``libspev_b200.so`` (C ABI in ``include/spev_b200.h``).  There is no
CPU, PyTorch-eager or Triton fallback: without the library or without an sm_100 GPU the calls
raise ``RuntimeError``.
"""
from ._lib import EXPORTED_SYMBOLS, LIB_PATH, load  # noqa: F401
from .batch import Context, FlatBatch, make_batch, out_layout, plan_chunk_tiles, plan_frame_tiles  # noqa: F401
from .dataset import (ResidentCache, read_reference_cache, write_metadata, write_records,  # noqa: F401
                      write_reference_cache)
from .features import frame_features_flat, rms, segment_pool, spectral_centroid  # noqa: F401
from .install import install, patch_model, uninstall  # noqa: F401
from .pitch import PyinContext, pyin, pyin_flat  # noqa: F401
from .records import (build_cache_sharded, build_records, corpus_stats, plan_records, scale_durations,  # noqa: F401
                      uniform_durations)  # noqa: F401
from .length_regulator import (LengthRegulator, VARIANCE_CLAMPS, expand, mel_mask, plan,  # noqa: F401
                               regulate_variances, variance_adaptor)
from .spectral import (griffinlim, griffinlim_flat, istft, logmel, logmel_flat, mel_project,  # noqa: F401
                       mel_to_audio, mel_to_mag_flat, mel_to_stft, melspectrogram, stft,
                       stft_power_flat)
from .variance import bucketize, bucketize_embed, duration_rule  # noqa: F401
from .vocoder import CONFIG, Vocoder  # noqa: F401

__version__ = "0.1.0"
