"""radar-b200: B200-native (sm_100a) per-frame detection hot path for radar point-cloud tracking.

Drop-in for the hot functions of ``4_temporal_object_tracker.py`` / ``radar_pipeline``:

* :mod:`.tracker`     ``load_radar_csv``, ``build_frame``, ``build_occupancy_grid``,
  ``identify_land_cells``, ``filter_land_from_frame``, ``st_dbscan`` and :func:`tracker.install`
* :mod:`.clustering`  flat-label ``st_dbscan(coords, times, ...)``
* :mod:`.transforms`  ``polar_to_cartesian``, ``sweep_to_point_cloud``
* :mod:`.fusion`      concat / grid-max gain fusion
* :mod:`.pipeline`    device-resident batch pipeline (what ``bench.py`` times)
* :mod:`.recording`   a whole recording fed block by block: one land grid, one ST-DBSCAN labelling (windowed)
* :mod:`.sharded`     time-sharded multi-GPU driver (one process per GPU, NCCL)

All compute is hand-written CUDA behind the C ABI of ``include/radarb200.h``
(``libradarb200.so``); there is no CPU fallback.
"""
import numpy as _np

from ._lib import RadarB200Error, load as load_library  # noqa: F401

# The library restates numpy >= 2 scalar promotion (NEP 50: `np.float32 + python float` stays float32) where the
# reference computes its grid edges (rb_arange_edges, T4:372-373). Under numpy 1.x the reference itself would produce
# different edges, and the two could disagree silently - refuse to load instead.
if int(_np.__version__.split(".")[0]) < 2:
    raise ImportError(f"radar_point_cloud_tracking_b200 needs numpy >= 2 (found {_np.__version__}): the land-grid edges "
                      "follow numpy 2's scalar promotion rules")

__all__ = ["RadarB200Error", "load_library"]
__version__ = "0.1.0"
