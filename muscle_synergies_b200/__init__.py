"""muscle_synergies_b200: the Vicon Nexus CSV loader and trial windowing of
elvis-sik/muscle_synergies, rebuilt for NVIDIA B200 (sm_100a).

    import muscle_synergies_b200 as muscle_synergies
    data = muscle_synergies.load_vicon_file("trial.csv")     # same call as the reference
    data.emg.df            # pandas DataFrame, bit-identical to the reference loader's
    data.emg.tensor        # (channels, rows) float64 CUDA tensor, zero-copy

The data path is hand-written CUDA behind a C ABI (include/ms_b200.h, libms_b200.so);
there is no CPU fallback.
"""
__version__ = "0.1.0"

from .analysis import (SynergyMatch, SynergyRunResult, find_synergies, match_synergies_batched,  # noqa: F401
                       nmf_beta_batched, nmf_cd_batched, nmf_mu_batched, nmf_transform_batched, vaf)
from .cache import load_trial, load_vicon_file_cached, save_trial  # noqa: F401
from .emg import (  # noqa: F401
    digital_filter,
    envelope_windows,
    linear_envelope,
    normalize,
    rms,
    time_normalize,
    zero_center,
)
from .pipeline import (cross_cycle_vaf, synergies_for_files, synergies_for_files_sharded,  # noqa: F401
                       synergy_similarity, trial_synergies)
from .vicon_data import (  # noqa: F401
    DeviceData,
    DeviceType,
    ViconLoader,
    ViconNexusData,
    load_vicon_bytes,
    load_vicon_file,
)

__all__ = (
    "load_vicon_file",
    "load_vicon_bytes",
    "ViconLoader",
    "ViconNexusData",
    "DeviceData",
    "DeviceType",
    # analysis.py names of the reference that have a CUDA implementation here
    "zero_center",
    "linear_envelope",
    "digital_filter",
    "rms",
    "normalize",
    "time_normalize",
    "vaf",
    "find_synergies",
    # extensions
    "match_synergies_batched",
    "nmf_beta_batched",
    "nmf_cd_batched",
    "nmf_mu_batched",
    "nmf_transform_batched",
    "envelope_windows",
    "save_trial",
    "load_trial",
    "load_vicon_file_cached",
    "trial_synergies",
    "cross_cycle_vaf",
    "synergy_similarity",
    "synergies_for_files",
    "synergies_for_files_sharded",
)
