"""blmm_b200 — B200-native engine for BulkLMM.jl's multi-trait LMM genome-scan path.

Host-side mirror of the reference's API (see api.py) over libblmm_b200.so (csrc/, include/)."""
from .api import (BlmmError, Engine, bulkscan, bulkscan_alt_grid, bulkscan_null, bulkscan_null_grid,  # noqa: F401
                  bulkscan_peaks,
                  calcKinship, default_engine, get_thresholds, lod2log10p, scan, thresholds_from_max,
                  transform_rotation, DeviceMatrix, read_csv_matrix, readBXDpheno, readBXDgeno,
                  readGenoProb_ExcludeComplements)
