"""One view loop for every kernel whose views are all valid: a candidate group of the correspondence kernel and the same views
through the triangulation entry point give the same point and the same mean reprojection error, bit for bit."""
import numpy as np
import pytest
import torch

from mocapv2_b200 import synth as S

N_SETS = 64


def dev(engine, a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(engine.device)


@pytest.mark.parametrize("fp64", [False, True])
@pytest.mark.parametrize("C", [2, 3, 4, 5, 6, 8, 16])
def test_correspondence_group_equals_triangulation(engine, C, fp64):
    """One integer centroid per camera and a cutoff no point misses: each frame-set has one root with one candidate group, whose
    point (obj[:, 0]) and mean error equal triangulate()'s for the same views exactly.  FP32 triangulates C = 2, 4, 6, 8, 16 in the
    dense kernel and C = 3, 5 in the generic one; FP64 always in the generic one."""
    rig = S.config_rig("c4")                                            # 16 cameras: the first C of them
    poses, params = rig["poses"][:C], rig["camera_params"][:C]
    rng = np.random.default_rng(100 + C)
    X = rig["centre"] + rng.uniform(-0.55, 0.55, (N_SETS, 3))
    xy = np.stack([np.floor(S.project_distorted(X, poses[c], params[c]["intrinsic_matrix"], params[c]["distortion_coef"]))
                   for c in range(C)], axis=1).astype(np.int32)         # [S, C, 2]
    cams = engine.cameras(poses, params)
    Fs = dev(engine, np.array(rig["Fs"][:C - 1], dtype=np.float64))
    r = engine.correspond(dev(engine, xy[:, :, None, :]), dev(engine, np.ones((N_SETS, C), np.int32)), Fs, cams,
                          obj_count=1, cutoff=1e9, fp64=fp64)
    assert (r.n_valid.cpu().numpy() == 1).all() and (r.n_obj.cpu().numpy() == 1).all() and (r.flags.cpu().numpy() == 0).all()
    xyz, err = engine.triangulate(dev(engine, xy).to(torch.float64 if fp64 else torch.float32), cams)
    assert np.array_equal(r.obj[:, 0].cpu().numpy(), xyz.double().cpu().numpy())
    assert np.array_equal(r.err[:, 0].cpu().numpy(), err.double().cpu().numpy())
