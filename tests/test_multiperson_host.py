"""CPU: host-side pieces of the multiperson mirror (no device work): the augmentation plan equals the reference's formulas
(multiperson_model.py:108-141, restated with ptu.linspace / ptu3d.rotation_mat), the JointInfo stand-in, the golden files."""
import os

import numpy as np
import torch

from metrabs_b200.multiperson.joint_info import JointInfo
from metrabs_b200.multiperson.multiperson_model import aug_parameters, intrinsic_matrix_from_field_of_view


def test_aug_plan_num_aug_5():
    gam, sc, fl, rf = aug_parameters(5)
    assert torch.allclose(gam, torch.tensor([0.6, 0.7, 0.8, 0.9, 1.0]))
    assert torch.allclose(sc, torch.tensor([0.8, 0.9, 1.0, 1.05, 1.1]))
    assert fl.tolist() == [False, True, False, True, False]
    assert rf.shape == (5, 3, 3)
    ang = np.deg2rad(25) * np.array([-1, -0.5, 0, 0.5, 1])
    for a in range(5):
        c, s = np.cos(-ang[a]), np.sin(-ang[a])
        r = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], dtype=np.float32)
        if fl[a]:
            r = np.diag([-1., 1, 1]).astype(np.float32) @ r
        assert np.allclose(rf[a].numpy(), r, atol=1e-6)


def test_aug_plan_degenerate_counts():
    for n in (1, 2, 3):
        gam, sc, fl, rf = aug_parameters(n)
        assert gam.shape == sc.shape == fl.shape == (n,) and rf.shape == (n, 3, 3)
    assert aug_parameters(1)[0].tolist() == [0.800000011920929]  # ptu.linspace(num=1) = midpoint


def test_fov_intrinsics():
    k = intrinsic_matrix_from_field_of_view(55, (480, 640))
    f = 640 / (np.tan(np.deg2rad(55) / 2) * 2)
    assert np.allclose(k[0].numpy(), [[f, 0, 320], [0, f, 240], [0, 0, 1]], rtol=1e-6)


def test_joint_info_mirror():
    ji = JointInfo(['pelv', 'lhip', 'rhip', 'neck', 'lsho', 'rsho', 'lone'], [(0, 1), (0, 2)])
    assert ji.mirror_mapping == [0, 2, 1, 3, 5, 4, 6]
    assert ji.n_joints == 7 and ji.stick_figure_edges == [(0, 1), (0, 2)]


def test_golden_files_present(golden_dir):
    g = np.load(os.path.join(golden_dir, 'multiperson_pipeline.npz'), allow_pickle=False)
    idx = g['crops_a5_af1_idx']  # a sample of the pixels of the 25 crops [25, 3, 64, 64], touching every crop
    assert g['crops_a5_af1'].shape == idx.shape and 0 <= idx.min() and idx.max() < 25 * 3 * 64 * 64
    assert len(np.unique(idx // (3 * 64 * 64))) == 25 and g['images'].dtype == np.uint8
    f = np.load(os.path.join(golden_dir, 'multiperson_filter.npz'), allow_pickle=False)
    assert f['keep'].sum() > 0
