"""astrild_b200: B200-native matter/halo power-spectrum path of astrild.

Drop-in host side (Python, mirrors astrild's interfaces for this path) over a C-ABI CUDA
library (include/astrild_pk.h, astrild_b200/csrc).  Only what the path needs lives here.
"""
from .lab import ArrayMesh, CatalogMesh, FFTBispectrum, FFTCorr, FFTPower, ParticleMesh, TaylorFourierMesh  # noqa: F401
from .engine import PkEngine, get_engine  # noqa: F401
from .power_spectrum_3d import PowerSpectrum3D, PowerSpectrum3DWarning  # noqa: F401
from .stats_subfind import SubFind  # noqa: F401
from .catalog import PkBatch, read_table, subfind_stats, write_table  # noqa: F401

__all__ = ["ArrayMesh", "CatalogMesh", "FFTBispectrum", "FFTCorr", "FFTPower", "ParticleMesh", "TaylorFourierMesh", "PkEngine", "get_engine",
           "PowerSpectrum3D", "PowerSpectrum3DWarning", "SubFind", "PkBatch", "read_table", "subfind_stats", "write_table"]
