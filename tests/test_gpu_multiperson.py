"""GPU: the steps either side of the crop model (SURVEY.md 8f) against goldens produced by the UNMODIFIED reference
(oracle/gen_golden_multiperson.py -> tests/golden/multiperson_*.npz):

* crop generation  - mtb_crop_setup + mtb_warp_crops vs Pose3dEstimator._get_crops (multiperson_model.py:264-355) and
                     warp_images_with_pyramid (warping.py:6-107), antialias 1 / 2, 5- and 12-coefficient distortion;
* the drop-in path - metrabs_b200's Pose3dEstimator + Metrabs vs the reference's _estimate_poses_batched (:74-185) running the
                     reference Metrabs on the same weights, frames and boxes (TTA merge, joint transform, skeletons, chunking);
* plausibility filter + pose NMS vs plausibility_check.py:8-119."""
import os

import numpy as np
import pytest
import torch

from oracle import port

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def H():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from tests import helpers
    return helpers


@pytest.fixture(scope='module')
def G(golden_dir):
    return np.load(os.path.join(golden_dir, 'multiperson_pipeline.npz'), allow_pickle=False)


def _scene(G):
    images = torch.from_numpy(G['images']).cuda()
    boxes = [torch.from_numpy(G[f'boxes_{i}']) for i in range(int(G['n_images']))]
    return images, boxes, torch.from_numpy(G['intrinsics']), torch.from_numpy(G['distortion']), \
        torch.from_numpy(G['extrinsics']), torch.from_numpy(G['world_up'])


def _per_box(G):
    images, boxes, intr, dist, ext, up = _scene(G)
    n_box = torch.tensor([len(b) for b in boxes])
    k_box = torch.repeat_interleave(intr, n_box, dim=0)
    d_box = torch.repeat_interleave(dist, n_box, dim=0)
    cam_up = torch.repeat_interleave(torch.einsum('c,bCc->bC', up, ext[..., :3, :3]), n_box, dim=0)
    ids = torch.repeat_interleave(torch.arange(len(boxes)), n_box)
    return images, torch.cat(boxes).cuda(), k_box.cuda(), d_box.cuda(), cam_up.cuda(), ids


@pytest.mark.parametrize('num_aug,af', [(5, 1), (5, 2), (2, 1), (2, 2)])
def test_crop_generation_vs_reference(H, G, num_aug, af):
    from metrabs_b200.multiperson import warping
    from metrabs_b200.multiperson.multiperson_model import aug_parameters
    images, boxes, k_box, d_box, cam_up, ids = _per_box(G)
    gam, sc, fl, rf = aug_parameters(num_aug)
    pyr = warping.build_pyramid(images)
    new_k, rot, inv, lev = warping.crop_setup(boxes, k_box, d_box, cam_up, rf, sc, 64, af)
    tag = f'crops_a{num_aug}_af{af}'
    # the per-crop matrices (multiperson_model.py:264-293, :321-355)
    assert H.rel_err(new_k, G[tag + '_newk']) < 2e-6
    assert (rot.cpu() - torch.from_numpy(G[tag + '_rot'])).abs().max() < 2e-6
    # the reference inverts new_K @ R with fp32 LU (torch.linalg.inv, :288); the device uses the fp64 adjugate: they agree to
    # the conditioning of that fp32 solve
    e_inv = max(H.rel_err(inv[i], G[tag + '_invproj'][i]) for i in range(inv.shape[0]))
    assert e_inv < 1e-4, e_inv
    # the golden holds a fixed, seeded sample of the crop pixels (flat indices into [n_crops, 3, 64, 64]) and their values
    idx = torch.from_numpy(G[tag + '_idx']).long()
    n_crops = num_aug * boxes.shape[0]

    def sample(c):
        assert c.shape == (n_crops, 3, 64, 64)
        return c.reshape(-1)[idx]
    ref = torch.from_numpy(G[tag])
    gexp = sample((gam / 2.2).repeat_interleave(boxes.shape[0])[:, None, None, None].expand(-1, 3, 64, 64))  # crop order: aug-major

    def linear(c):  # undo the final `crops **= gamma / 2.2` (multiperson_model.py:318): back to linear light
        return c.clamp_min(0) ** (1.0 / gexp)
    # (1) the warp kernel alone, on the reference's own inverse projections.  Bars: 5e-5 in LINEAR light - source coordinates
    # reach 260 px, where one fp32 ulp is 3e-5 px, and across the zero-padding border of the frame the bilinear blend has a
    # gradient of O(1) per px, so two fp32 evaluation orders of the same homography differ by ~1e-5 there (measured 1.1-1.9e-5;
    # 9.8e-6 on the 12-coefficient case without border pixels).  The gamma-encoded output x^(gamma/2.2) has slope
    # 0.27 x^-0.73 -> 40 at x = 1e-3, so dark / half-outside pixels show those differences as ~1e-4: held to 5e-4
    inv_ref = torch.from_numpy(G[tag + '_invproj']).cuda().contiguous()
    crops = sample(warping.warp_images_with_pyramid(images, pyr, k_box, inv_ref, d_box, lev, gam / 2.2, 64, ids, num_aug, af).cpu())
    err_lin = (linear(crops) - linear(ref)).abs().max().item()
    err = (crops - ref).abs().max().item()
    # (2) the whole device chain (own setup: fp64-adjugate inverse instead of the reference's fp32 LU)
    crops2 = sample(warping.warp_images_with_pyramid(images, pyr, k_box, inv, d_box, lev, gam / 2.2, 64, ids, num_aug, af).cpu())
    err2_lin = (linear(crops2) - linear(ref)).abs().max().item()
    err2 = (crops2 - ref).abs().max().item()
    print(f'{tag}: max abs crop error, linear light {err_lin:.2e} / gamma-encoded {err:.2e} on the reference matrices; {err2_lin:.2e} / '
          f'{err2:.2e} with the device setup; inverse-projection rel diff {e_inv:.1e}; levels {sorted(set(lev.cpu().tolist()))}')
    assert err_lin < 5e-5 and err < 5e-4
    assert err2_lin < 1e-4 and err2 < 5e-4
    assert len(set(lev.cpu().tolist())) >= 2  # the scene exercises more than one pyramid level


def test_twelve_coefficient_distortion(H, G):
    from metrabs_b200.multiperson import warping
    images, boxes, k_box, d_box, cam_up, ids = _per_box(G)
    d12 = torch.from_numpy(G['d12_coeffs']).cuda()
    inv = torch.from_numpy(G['d12_invproj']).cuda().contiguous()
    scales = torch.from_numpy(G['d12_scales'])
    lev = torch.clip(torch.floor(-torch.log2(scales)), 0, 2).int().cuda()
    pyr = warping.build_pyramid(images)
    crops = warping.warp_images_with_pyramid(images, pyr, k_box, inv, d12, lev, torch.tensor([1.0]), 64, ids, 1, 1)
    err = (crops.cpu() - torch.from_numpy(G['d12_crops'])).abs().max().item()
    print(f'12-coefficient distortion: max abs crop error {err:.2e}')
    assert err < 1e-5


def _device_estimator(H, G, golden_dir, precision='fp32'):
    from metrabs_b200.multiperson import Pose3dEstimator
    from metrabs_b200.multiperson.joint_info import JointInfo
    g = np.load(os.path.join(golden_dir, 'tiny_s64_j8.npz'), allow_pickle=False)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith('sd/')}
    m = H.device_model('efficientnetv2-tiny', port.PathConfig(proc_side=64), 8, sd, precision=precision)
    m.joint_names = G['joint_names']
    m.joint_edges = G['joint_edges']
    ji = JointInfo(G['joint_names'], G['joint_edges'])
    assert ji.mirror_mapping == G['mirror'].tolist()  # the 'l...' <-> 'r...' name convention
    skel = {'': dict(indices=list(range(10)), names=[f'k{i}' for i in range(10)], edges=[[0, 1]]),
            'upper': dict(indices=[5, 6, 7, 9, 0], names=list('abcde'), edges=[[0, 1]])}
    return Pose3dEstimator(m, skel, G['joint_transform'], joint_info=ji)


def test_tta_merge_vs_reference(H, G):
    """Mirror swap, poses @ R, joint transform, distorted projection, inverse extrinsics, skeleton gather and the mean over
    augmentations (multiperson_model.py:143-182, :246-259): the reference caller around a crop model that returns a fixed
    table of poses, against this package's caller around the same table."""
    from metrabs_b200.multiperson import Pose3dEstimator
    from metrabs_b200.multiperson.joint_info import JointInfo
    table = torch.from_numpy(G['merge_table']).cuda()

    class TableModel(torch.nn.Module):
        joint_names, joint_edges, input_resolution, device = G['joint_names'], G['joint_edges'], np.int32(64), 'cuda'

        def forward(self, inp):
            return table[:inp[0].shape[0]].clone()
    skel = {'': dict(indices=list(range(10)), names=[f'k{i}' for i in range(10)], edges=[[0, 1]]),
            'upper': dict(indices=[5, 6, 7, 9, 0], names=list('abcde'), edges=[[0, 1]])}
    est = Pose3dEstimator(TableModel(), skel, G['joint_transform'], joint_info=JointInfo(G['joint_names'], G['joint_edges']))
    images, boxes, intr, dist, ext, up = _scene(G)
    worst = 0.0
    for avg in (True, False):
        for sk in ('', 'upper'):
            res = est._estimate_poses_batched(images, boxes, intr, dist, ext, up, 55, 0, 1, 5, avg, sk, False)
            tag = f'merge_avg{int(avg)}_{sk or "all"}'
            for i in range(2):
                assert res['poses3d'][i].shape == G[f'{tag}_p3d_{i}'].shape
                e3 = H.rel_err(res['poses3d'][i], G[f'{tag}_p3d_{i}'])
                e2 = H.rel_err(res['poses2d'][i], G[f'{tag}_p2d_{i}'])
                worst = max(worst, e3, e2)
                assert e3 < 1e-5 and e2 < 1e-5, (tag, i, e3, e2)
    print(f'TTA merge: worst relative error vs the reference caller {worst:.2e}')


@pytest.mark.parametrize('precision', ['fp32', 'tf32x3'])
def test_pipeline_vs_reference_caller(H, G, golden_dir, precision):
    """frames + boxes -> poses3d / poses2d through THIS package's Pose3dEstimator and crop model, against the reference's
    _estimate_poses_batched driving the reference Metrabs (same committed weights).  Bars: 1e-3 on poses3d (the joint
    tolerance of BASELINE.json); poses2d is the projection x/z of those poses and the untrained tiny model emits joints with
    z near 0, so its 2D error is the 3D error amplified by the conditioning of the division - held to 2e-2 here and pinned
    to 1e-5 on well-conditioned poses by test_tta_merge_vs_reference."""
    est = _device_estimator(H, G, golden_dir, precision)
    images, boxes, intr, dist, ext, up = _scene(G)
    worst3 = worst2 = 0.0
    for avg in (True, False):
        for sk in ('', 'upper'):
            res = est._estimate_poses_batched(images, boxes, intr, dist, ext, up, 55, 64, 1, 5, avg, sk, False)
            tag = f'pipe_avg{int(avg)}_{sk or "all"}'
            for i in range(2):
                e3 = H.rel_err(res['poses3d'][i], G[f'{tag}_p3d_{i}'])
                e2 = H.rel_err(res['poses2d'][i], G[f'{tag}_p2d_{i}'])
                worst3, worst2 = max(worst3, e3), max(worst2, e2)
                assert res['poses3d'][i].shape == G[f'{tag}_p3d_{i}'].shape
                assert e3 < 1e-3 and e2 < 2e-2, (tag, i, e3, e2)
    res = est._estimate_poses_batched(images, boxes, intr, dist, ext, up, 55, 10, 1, 5, True, '', False)
    for i in range(2):
        assert H.rel_err(res['poses3d'][i], G[f'pipe_chunk2_p3d_{i}']) < 1e-3
    # the public wrappers the reference ships broken (tuple defaults, SURVEY 3.4) work here
    one = est.estimate_poses(images[0], boxes[0][:, :4], intr[0], dist[0], ext[0], up, num_aug=5)
    assert one['poses3d'].shape == (3, 10, 3) and torch.isfinite(one['poses3d']).all()
    print(f'[{precision}] worst relative error vs the reference caller: poses3d {worst3:.2e}, poses2d {worst2:.2e}')


def test_pose_filter_vs_reference(H, golden_dir):
    from metrabs_b200.multiperson import plausibility_check
    g = np.load(os.path.join(golden_dir, 'multiperson_filter.npz'), allow_pickle=False)
    p3, p2, boxes = (torch.from_numpy(g[k]).cuda() for k in ('poses3d', 'poses2d', 'boxes'))
    plausible, keep = plausibility_check.filter_poses(p3, p2, boxes, g['n_per_image'].tolist(), g['bones'], g['mean_bones'])
    want_plausible = g['plausible_bones'] & g['consistent'] & g['in_box']
    assert plausible.cpu().numpy().tolist() == want_plausible.tolist()
    assert keep.cpu().numpy().tolist() == g['keep'].tolist()
    assert 0 < int(keep.sum()) < len(keep)
