"""CPU-side checks of the drop-in boundary: the shims register under the reference's module names,
export the reference's public names with the reference's signatures, and refuse to run without a GPU."""
import inspect
import json
import sys
from pathlib import Path

import numpy as np
import pytest

from skiing_analysis_pytorch_b200 import dropin

# public names and positional parameters of the reference modules (SURVEY.md section 8a/8b; their defaults are
# recorded in tests/golden/reference_signatures.json)
EXPECTED = {
    "triangulation.triangulate": {
        "triangulate_joints": ["keypoints1", "keypoints2", "K", "R", "T"],
        "process_triangulate": ["left_kpts", "right_kpts", "left_vframes", "right_vframes", "K", "R", "T", "output_path"],
    },
    "triangulation.reproject": {
        "reproject_points": ["X3", "K1", "dist1", "K2", "dist2", "R", "T"],
        "render_reprojection_panel": ["img1", "img2", "kptL", "kptR", "proj_L", "proj_R", "joint_names", "circle_r", "thickness",
                                      "align_height", "title_left", "title_right"],
        "reproject_and_visualize": ["img1", "img2", "X3", "kptL", "kptR", "K1", "dist1", "K2", "dist2", "R", "T", "joint_names",
                                    "circle_r", "thickness", "out_path"],
    },
    "bundle_adjustment.loss": {
        "project_points": ["X3d", "R", "t", "K"],
        "reprojection_loss": ["X3d", "R", "t", "K", "x2d", "conf2d", "w"],
        "camera_center_from_Rt": ["R", "t"],
        "camera_smooth_loss": ["R", "t", "w"],
        "baseline_reg_loss": ["R", "t", "w"],
        "bone_length_loss": ["X3d", "ref_bone_len", "w"],
        "pose_temporal_loss": ["X3d", "w"],
    },
    "vggt.triangulate": {
        "make_P": ["K", "R", "t"],
        "triangulate_point": ["P1", "P2", "x1", "x2"],
        "triangulate_one_frame": ["K", "R", "T", "kptL", "kptR", "frame_L", "frame_R", "save_dir", "dist", "visualize_3d", "frame_num"],
    },
}
EXPECTED["triangulation.postprocess"] = {
    "build_P": ["K", "R", "t"],
    "project": ["P", "X3"],
    "reproj_errors": ["P1", "P2", "X3", "x1_pix", "x2_pix"],
    "positive_depth_mask": ["R", "T", "X3"],
    "smooth_skeleton": ["X", "win", "poly"],
    "post_triage_single": ["X3_frame", "kptL_frame", "kptR_frame", "K1", "K2", "R", "T", "dist1", "dist2", "confL", "confR",
                           "conf_thr", "err_thresh_px", "return_masks"],
    "post_triage_sequence": ["X3_seq", "kptL_seq", "kptR_seq", "K1", "K2", "R", "T", "dist1", "dist2", "confL", "confR", "conf_thr",
                             "err_thresh_px", "smooth", "sg_win", "sg_poly"],
}
for _m in ("bundle_adjustment.reproject", "vggt.reproject", "front_side.side.reproject", "fuse.side.reproject"):
    EXPECTED[_m] = EXPECTED["triangulation.reproject"]


for _m in ("bundle_adjustment.fuse.fuse", "fuse.side.fuse.fuse", "front_side.side.fuse.fuse"):
    EXPECTED[_m] = {"rigid_transform_3D": ["target", "source", "tau", "allow_scale", "wL", "wR", "return_diagnostics", "verbose"]}


def test_install_registers_reference_module_names():
    saved = {k: sys.modules.get(k) for k in list(dropin.MODULE_MAP) + ["triangulation", "bundle_adjustment", "vggt", "front_side",
                                                                        "front_side.side", "fuse", "fuse.side", "bundle_adjustment.fuse", "fuse.side.fuse",
                                                                        "front_side.side.fuse"]}
    try:
        mods = dropin.install()
        assert set(mods) == set(dropin.MODULE_MAP)
        import bundle_adjustment.loss as bl
        import triangulation.reproject as tr
        from vggt.triangulate import triangulate_one_frame  # noqa: F401

        assert tr is mods["triangulation.reproject"] and bl is mods["bundle_adjustment.loss"]
        assert len(bl.BONES) == 12 and callable(sys.modules["bundle_adjustment"].run_local_ba)
        for name, funcs in EXPECTED.items():
            for fn, params in funcs.items():
                got = list(inspect.signature(getattr(mods[name], fn)).parameters)
                assert got == params, (name, fn, got)
        assert mods["triangulation.triangulate"].K_dist.shape == (14,)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_signatures_match_the_reference_checkout():
    """Parameter names and int / float / str / bool / None defaults of every shim equal the reference's, as recorded in
    tests/golden/reference_signatures.json (python -m oracle.make_golden --only-signatures); when SKA_REFERENCE_ROOT points
    at a checkout of the reference, the record is compared with it as well."""
    from oracle import ref_import

    rec = json.loads((Path(__file__).parent / "golden" / "reference_signatures.json").read_text())
    # front_side.* / fuse.*: same file content as bundle_adjustment/reproject.py and fuse.py; importing them pulls heavy packages
    assert {n: sorted(f) for n, f in rec.items()} == {n: sorted(f) for n, f in EXPECTED.items() if not n.startswith(("front_side", "fuse"))}
    for name, funcs in rec.items():
        sh = dropin.shim(name)
        for fn, params in funcs.items():
            assert ref_import.signature_record(getattr(sh, fn)) == params, (name, fn)
            assert [p["name"] for p in params] == EXPECTED[name][fn], (name, fn)
    if not ref_import.available():
        return
    try:
        for name, funcs in rec.items():
            ref = ref_import.load(name)
            for fn, params in funcs.items():
                assert ref_import.signature_record(getattr(ref, fn)) == params, (name, fn)
    finally:
        for k in list(sys.modules):
            if k.split(".")[0] in ("triangulation", "bundle_adjustment", "vggt"):
                sys.modules.pop(k, None)


def test_shims_fail_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    tri = dropin.shim("triangulation.triangulate")
    with pytest.raises(RuntimeError, match="no CPU path"):
        tri.triangulate_joints(np.zeros((17, 2), np.float32), np.zeros((17, 2), np.float32), np.eye(3), np.eye(3), np.zeros(3))
    loss = dropin.shim("bundle_adjustment.loss")
    with pytest.raises(RuntimeError, match="no CPU path"):
        loss.pose_temporal_loss(torch.zeros(4, 17, 3))
    # argument errors come first, exactly like the reference (triangulate.py:61-64)
    with pytest.raises(ValueError, match="Keypoints shape mismatch"):
        tri.triangulate_joints(np.zeros((17, 2)), np.zeros((16, 2)), np.eye(3), np.eye(3), np.zeros(3))
    rep = dropin.shim("bundle_adjustment.reproject")
    with pytest.raises(ValueError, match="Unsupported R shape"):
        rep.reproject_points(np.zeros((17, 3)), np.eye(3), None, np.eye(3), None, np.zeros(9), np.zeros(3))


def test_rotation_round_trip_is_what_cv2_applies():
    """ADVICE r1: the reference hands cv2.projectPoints a rotation VECTOR made from the float32 matrix (reproject.py:69); the
    shim's host-side restatement of that round trip (SVD projection onto SO(3), float32 vector, Rodrigues) equals cv2's."""
    import cv2
    import numpy as np

    from skiing_analysis_pytorch_b200.dropin._common import rotation_as_projectpoints_sees_it as f

    rng = np.random.default_rng(0)
    for _ in range(300):
        R = cv2.Rodrigues(rng.normal(size=3) * rng.choice([1e-4, 0.1, 1.0, 3.0]))[0]
        R = (R + rng.normal(size=(3, 3)) * rng.choice([0, 1e-6, 1e-3, 0.05])).astype(np.float32)
        rvec, _ = cv2.Rodrigues(R)
        assert np.abs(f(R) - cv2.Rodrigues(rvec.astype(np.float64))[0]).max() < 1e-9
    assert np.array_equal(f(np.eye(3)), np.eye(3))


def test_host_pipeline_chunk_schedule_partitions_the_clip():
    from skiing_analysis_pytorch_b200.api import chunk_schedule

    for T, chunk, ramp in ((1_000_000, 131072, 0), (1_000_000, 131072, 8192), (1_000_000, 65536, 4096), (5000, 1024, 8192), (100, 65536, 0),
                           (300_000, 131072, 8192), (1, 1, 0), (17, 5, 2)):
        sch = chunk_schedule(T, chunk, ramp)
        assert sch[0][0] == 0 and sch[-1][1] == T and all(a[1] == b[0] for a, b in zip(sch, sch[1:]))
        assert all(0 < b - a <= chunk for a, b in sch)
    up = [b - a for a, b in chunk_schedule(1_000_000, 131072, 8192)]
    assert up[:4] == [8192, 16384, 32768, 65536] and up[-4:] == [65536, 32768, 16384, 8192]
    assert chunk_schedule(0, 1024) == []
