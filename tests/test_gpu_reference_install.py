"""The drop-in installed into a module with the reference's names: ``tracker.install`` / ``fusion.install`` applied to a
stand-in carrying the classes and configuration globals of ``4_temporal_object_tracker.py`` (T4:55-158) and
``5_gain_fusion_ply_builder.py`` (T5:52-63), whose patched names are then called on a synthetic CSV tree the way the
reference's ``run_pipeline`` calls them (T4:936-977). The clusters must equal those in ``clusters.csv`` of a real
``run_pipeline`` run of the unmodified reference on the same tree (``tests/golden/run_pipeline_csv.npz``, made by
``tests/golden/make_golden_run_pipeline.py``), and the patched ``fuse_gains_max`` the unmodified function's output
(``tests/golden/fuse_max.npz``). The reference scripts themselves are not part of this repository."""
import io
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from radar_point_cloud_tracking_b200 import synthetic as syn
from tests.common import golden, pipe_inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def csv_tree(tmp_path_factory):
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    root = tmp_path_factory.mktemp("tree") / "data"
    spec, echo = pipe_inputs()
    files = syn.write_csv_tree(spec, root, echo)
    return root, files


def _t4_stand_in():
    from radar_point_cloud_tracking_b200 import tracker as trk
    return SimpleNamespace(RadarFrame=trk.RadarFrame, Cluster=trk.Cluster,
                           **{k: getattr(trk, k) for k in trk._CFG_NAMES + ("EPS_SPACE", "EPS_TIME", "MIN_SAMPLES")})


@pytest.mark.parametrize("tag,kw", [("default", {}),
                                    ("nofilter_eps6", dict(skip_land_filter=True, eps_space=6.0, eps_time=1.0, min_samples=8))])
def test_installed_tracker_reproduces_the_reference_clusters_csv(csv_tree, tag, kw):
    from radar_point_cloud_tracking_b200 import _lib, tracker
    _, files = csv_tree
    T4 = _t4_stand_in()
    tracker.install(T4)
    p = dict(dict(skip_land_filter=False, eps_space=T4.EPS_SPACE, eps_time=T4.EPS_TIME, min_samples=T4.MIN_SAMPLES), **kw)
    launches = _lib.context(0).launch_count()
    frames = [f for f in (T4.build_frame(ff, i) for i, ff in enumerate(files)) if f is not None]        # T4:941-945
    if not p["skip_land_filter"] and len(frames) > 10:                                                 # T4:954-966
        count, isum, edges = T4.build_occupancy_grid(frames, T4.LAND_GRID_RESOLUTION)
        land = T4.identify_land_cells(count, isum, len(frames))
        frames = [T4.filter_land_from_frame(f, land, edges) for f in frames]
    clusters = T4.st_dbscan(frames, p["eps_space"], p["eps_time"], p["min_samples"])                  # T4:968-977
    assert _lib.context(0).launch_count() > launches                            # the CUDA library did the work
    got = np.array(sorted((fid, c.cluster_id, c.num_points, c.centroid[0], c.centroid[1], c.mean_intensity)
                          for fid, cl in clusters.items() for c in cl), dtype=np.float64).reshape(-1, 6)
    text = str(golden("run_pipeline_csv")[f"{tag}/clusters.csv"])
    assert text.split("\n", 1)[0] == "frame_id,cluster_id,num_points,centroid_x,centroid_y,mean_intensity"
    want = np.loadtxt(io.StringIO(text), delimiter=",", skiprows=1, ndmin=2)
    want = want[np.lexsort((want[:, 1], want[:, 0]))]
    assert len(want) > 0 and got.shape == want.shape
    assert np.array_equal(got[:, :3], want[:, :3])
    assert np.array_equal(got[:, 3:].astype(np.float32), want[:, 3:].astype(np.float32))   # the CSV holds float32 values


def test_installed_fusion_reproduces_the_reference_fuse_gains_max(csv_tree):
    """``fusion.install`` on a stand-in with T5's configuration globals: its ``fuse_gains_max`` name runs the CUDA path
    and reproduces the golden of the unmodified function (T5:222-273); the colour helpers and PLY writers it installs
    are the ones ``tests/test_plyio.py`` pins byte for byte to files the unmodified writers produced."""
    from radar_point_cloud_tracking_b200 import fusion, plyio
    _, files = csv_tree
    T5 = SimpleNamespace(NUM_ECHO_COLUMNS=1024, INTENSITY_THRESHOLD=5.0, POINT_STRIDE=8)
    fusion.install(T5)
    g = golden("fuse_max")
    for tag, res in (("r1", 1.0), ("r2p5", 2.5)):
        x, y, z = T5.fuse_gains_max(files[0], res)
        assert x.dtype == g[f"{tag}_x"].dtype
        assert np.array_equal(x, g[f"{tag}_x"]) and np.array_equal(y, g[f"{tag}_y"]) and np.array_equal(z, g[f"{tag}_i"])
    assert T5.write_ply_fast is plyio.write_ply_fast and T5.intensity_to_rgb is plyio.intensity_to_rgb
    assert T5.normalize_intensity is plyio.normalize_intensity
