"""CPU: the `key = value;` parameter files the reconstruction stage is launched with (Server/scan_processor.py:27-35) parse into
scn_tsdf_params: the reference's own files (copies in tests/golden/), and an excerpt of the same lines."""
import os

import pytest

from scannet_b200 import tsdf

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXCERPT = """\
// excerpt of Server/tools/recons/zParametersScanNet.txt (lines 20-21, 34-35, 47-58) in the reference's own syntax
s_sensorIdx = 8;	//0 kinect, 8 SensorDataReader
s_integrationWidth = 320;		//render width (decoupled from the input)
s_integrationHeight = 240;		//render height
s_sensorDepthMax = 6.0f;	//maximum sensor depth in meter
s_sensorDepthMin = 0.1f;	//minimum sensor depth in meter
s_SDFVoxelSize = 0.010f;				//voxel size in meter (IMPORTANT: reduce to improve perf.)
s_SDFTruncation = 0.06f;				//truncation in meter
s_SDFTruncationScale = 0.02f;			//truncation scale in meter per meter
s_SDFMaxIntegrationDistance = 4.0f;		//maximum integration in meter
s_SDFIntegrationWeightSample = 1;		//weight for an integrated depth value
s_SDFIntegrationWeightMax = 99999999;	//maximum integration weight for a voxel
s_hashNumBuckets = 800000;				//hash table size in buckets
s_hashNumSDFBlocks = 600000;			//smaller voxels require more space
"""


def check_scannet(p):
    assert (p.width, p.height) == (320, 240)
    assert abs(p.voxel_size - 0.010) < 1e-9 and abs(p.trunc_base - 0.06) < 1e-7 and abs(p.trunc_scale - 0.02) < 1e-7
    assert abs(p.depth_min - 0.1) < 1e-7 and abs(p.depth_max - 6.0) < 1e-7 and abs(p.max_integration_distance - 4.0) < 1e-7
    assert p.weight_sample == 1 and p.weight_max == 255          # the voxel's weight is a byte: 99999999 saturates
    assert p.max_blocks == 600000 and p.hash_slots == 4 * 800000


def test_excerpt_of_the_scannet_parameter_file(tmp_path, built):
    f = tmp_path / "zParametersScanNet.txt"; f.write_text(EXCERPT)
    check_scannet(tsdf.params_from_file(str(f)))


def test_real_reference_parameter_files(built):
    p = tsdf.params_from_file(os.path.join(G, "zParametersScanNet.txt"))
    check_scannet(p)
    # the bundling file switches the depth bilateral pre-filter on (zParametersBundlingScanNet.txt:72-74); files are applied in order
    q = tsdf.params_from_file(os.path.join(G, "zParametersBundlingScanNet.txt"), p)
    assert q.depth_filter == 1 and abs(q.depth_sigma_d - 2.0) < 1e-7 and abs(q.depth_sigma_r - 0.05) < 1e-7
    check_scannet(q)


def test_unknown_keys_comments_and_errors(tmp_path, built):
    from scannet_b200._lib import ScnError
    f = tmp_path / "p.txt"
    f.write_text("// only a comment\n\ns_unknownKey = 3;\ns_SDFVoxelSize = 0.004f; // trailing comment\n   s_depthFilter = true;\nnot a pair\n")
    p = tsdf.params_from_file(str(f))
    assert abs(p.voxel_size - 0.004) < 1e-9 and p.depth_filter == 1
    d = tsdf.default_params()
    assert (p.width, p.height, p.trunc_base) == (d.width, d.height, d.trunc_base)      # untouched fields keep their defaults
    with pytest.raises(ScnError, match="cannot open"):
        tsdf.params_from_file(str(tmp_path / "missing.txt"))
