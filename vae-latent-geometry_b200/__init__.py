"""vlg_b200 -- B200-native engine for the geodesic curve-energy hot path of
johannefranck/vae-latent-geometry (see DESIGN.md).  Import name: ``vlg_b200`` (the directory
is called ``vae-latent-geometry_b200``; ``vlg_b200.py`` at the repo root is the import shim).
"""
from . import _lib, build, formats, sharding  # noqa: F401
from .api import (DEFAULT_PRECISION, DecoderEnsemble, GeodesicSplineBatch, compute_energy, compute_energy_mc,  # noqa: F401
                  compute_geodesic_lengths, construct_nullspace_basis, ensemble_std_norm, expected_curve_energy,
                  fit_splines_to_paths, optimize_single_decoder, optimize_splines)
from ._lib import VlgError  # noqa: F401

__all__ = ["DEFAULT_PRECISION", "DecoderEnsemble", "GeodesicSplineBatch", "compute_energy", "compute_energy_mc",
           "compute_geodesic_lengths", "construct_nullspace_basis", "ensemble_std_norm", "expected_curve_energy",
           "fit_splines_to_paths", "optimize_single_decoder", "optimize_splines", "VlgError"]
