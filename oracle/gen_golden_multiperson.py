"""TEST INFRASTRUCTURE ONLY - golden fixtures for the steps either side of the crop model (SURVEY.md 8f), produced by the
UNMODIFIED reference (/root/reference/metrabs_pytorch/multiperson/{multiperson_model,warping,plausibility_check}.py)
on torch-cpu in the build container:  ``python oracle/gen_golden_multiperson.py``  ->  tests/golden/multiperson_*.npz

Stubs (the reference imports packages that are not installed and cannot be: no network): ``posepile.joint_info.JointInfo``
(names, edges, n_joints, mirror_mapping - the attributes multiperson_model.py:25,249 reads), ``get_joint2bone_mat``
(+1/-1 per stick-figure edge), ``ultralytics.YOLO`` (the detector is never called: boxes are given), ``simplepyutils``.
The crop model inside the reference ``Pose3dEstimator`` is the reference ``Metrabs`` itself (tiny EfficientNetV2 grammar,
the committed weights of tests/golden/tiny_s64_j8.npz); ``torch.autocast(device_type='cuda')`` is a no-op on a CPU-only
host, so the reference runs in fp32 here."""
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import port  # noqa: E402
from oracle import ref_import  # noqa: E402
from oracle.gen_golden import build_reference_model  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')

JOINT_NAMES = ['pelv', 'lhip', 'rhip', 'lkne', 'rkne', 'neck', 'lsho', 'rsho']
JOINT_EDGES = [(0, 1), (0, 2), (1, 3), (2, 4), (0, 5), (5, 6), (5, 7)]
MIRROR = [0, 2, 1, 4, 3, 5, 7, 6]
CROP_SAMPLE = 16  # one pixel in 16 of each crop batch is stored: the whole batches would put the fixture over 1 MB


def pixel_sample(crops, seed):
    """(sorted flat indices, values) of a fixed, seeded sample of 1/CROP_SAMPLE of the elements of ``crops``."""
    flat = crops.reshape(-1).numpy()
    idx = np.sort(np.random.default_rng(seed).choice(flat.size, flat.size // CROP_SAMPLE, replace=False)).astype(np.int32)
    return idx, flat[idx]


class StubJointInfo:
    def __init__(self, names, edges):
        self.names = list(names)
        self.stick_figure_edges = [tuple(int(i) for i in e) for e in np.asarray(edges).reshape(-1, 2)]
        self.n_joints = len(self.names)
        self.mirror_mapping = MIRROR[:self.n_joints]


def joint2bone_mat(joint_info):
    m = torch.zeros(len(joint_info.stick_figure_edges), joint_info.n_joints)
    for r, (i, j) in enumerate(joint_info.stick_figure_edges):
        m[r, i], m[r, j] = 1, -1
    return m


def import_multiperson(cfg):
    R = ref_import.import_reference(cfg.as_reference_dict())
    ji_mod = ref_import._stub('posepile.joint_info', JointInfo=StubJointInfo, get_joint2bone_mat=joint2bone_mat)
    sys.modules['posepile'].joint_info = ji_mod
    sys.modules['posepile'].datasets3d = sys.modules['posepile.datasets3d']
    ref_import._stub('ultralytics', YOLO=lambda *a, **k: None)
    import metrabs_pytorch.multiperson.multiperson_model as mm
    import metrabs_pytorch.multiperson.plausibility_check as pc
    import metrabs_pytorch.multiperson.warping as wp
    return R, mm, wp, pc


def smooth_images(n, h, w, seed):
    """uint8 frames with low-frequency content (gradients << 1 grey level / pixel): bilinear samples are then insensitive
    to the last-bit differences of two fp32 coordinate pipelines."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand(n, 3, h // 16 + 2, w // 16 + 2, generator=g)
    img = torch.nn.functional.interpolate(low, size=(h, w), mode='bicubic', align_corners=True).clamp(0, 1)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, h), torch.linspace(0, 1, w), indexing='ij')
    img = 0.7 * img + 0.3 * (0.5 + 0.5 * torch.sin(6 * xx + 4 * yy))[None, None]
    return (img * 255).round().clamp(0, 255).to(torch.uint8)


def scene():
    images = smooth_images(2, 200, 260, seed=5)
    boxes = [torch.tensor([[30., 20., 45., 80., 0.9], [100., 10., 120., 170., 0.8], [-20., 60., 150., 160., 0.7]]),
             torch.tensor([[10., 5., 240., 190., 0.95], [150., 90., 60., 60., 0.5]])]
    intr = torch.tensor([[[210., 0., 128.], [0., 205., 101.], [0., 0., 1.]],
                         [[180., 0., 131.], [0., 180., 99.], [0., 0., 1.]]])
    dist = torch.tensor([[-0.12, 0.05, 0.002, -0.003, 0.01], [0., 0., 0., 0., 0.]])
    a = 0.2
    ext = torch.eye(4).repeat(2, 1, 1)
    ext[1, :3, :3] = torch.tensor([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]], dtype=torch.float32)
    ext[1, :3, 3] = torch.tensor([100., -50., 300.])
    up = torch.tensor([0., -1., 0.])
    return images, boxes, intr, dist, ext, up


def tiny_reference_estimator(R, mm):
    g = np.load(os.path.join(OUT, 'tiny_s64_j8.npz'), allow_pickle=False)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith('sd/')}
    spec = port.effnet_spec('efficientnetv2-tiny')
    model = build_reference_model(R, spec, 8, 64)
    model.load_state_dict(sd, strict=True)
    model.joint_names = np.array(JOINT_NAMES)
    model.joint_edges = np.array(JOINT_EDGES)
    jt = torch.eye(8)
    jt = torch.cat([jt, torch.tensor([[0.5, 0.25, 0.25, 0, 0, 0, 0, 0], [0, 0, 0, 0, 0, 0.5, 0.25, 0.25]]).T], dim=1)  # [8, 10]
    skeleton_infos = {'': dict(indices=list(range(10)), names=[f'k{i}' for i in range(10)], edges=[[0, 1]]),
                      'upper': dict(indices=[5, 6, 7, 9, 0], names=['a', 'b', 'c', 'd', 'e'], edges=[[0, 1]])}
    est = mm.Pose3dEstimator(model, skeleton_infos, jt.numpy())
    # the on-disk format of scripts/demo_image.py:59-74: torch.save(model.state_dict()) of the REFERENCE model object
    torch.save(model.state_dict(), os.path.join(OUT, 'tiny_ckpt.pt'))
    return est, jt, skeleton_infos


def _torch_version_shims():
    """The reference was written against an older torch: ``torch.split(x, <int tensor>)`` (multiperson_model.py:154-155,176)
    is rejected by torch 2.11.  The shim converts the tensor to a list; the reference source stays unmodified."""
    orig = torch.split

    def split(tensor, split_size_or_sections, dim=0):
        if torch.is_tensor(split_size_or_sections):
            split_size_or_sections = [int(v) for v in split_size_or_sections]
        return orig(tensor, split_size_or_sections, dim)
    torch.split = split


def main():
    _torch_version_shims()
    cfg = port.PathConfig(proc_side=64)
    R, mm, wp, pc = import_multiperson(cfg)
    os.makedirs(OUT, exist_ok=True)
    images, boxes, intr, dist, ext, up = scene()
    est, jt, skel = tiny_reference_estimator(R, mm)
    data = dict(images=images.numpy(), intrinsics=intr.numpy(), distortion=dist.numpy(), extrinsics=ext.numpy(),
                world_up=up.numpy(), n_images=2, joint_transform=jt.numpy(), mirror=np.array(MIRROR),
                joint_names=np.array(JOINT_NAMES), joint_edges=np.array(JOINT_EDGES))
    for i, b in enumerate(boxes):
        data[f'boxes_{i}'] = b.numpy()
    n_box = torch.tensor([len(b) for b in boxes])
    # ---- crop generation goldens: _get_crops on all boxes as one batch, antialias 1 and 2 (multiperson_model.py:264-319)
    with torch.inference_mode():
        imgs_lin = (images.float() / 255) ** 2.2
        k_box = torch.repeat_interleave(intr, n_box, dim=0)
        d_box = torch.repeat_interleave(dist, n_box, dim=0)
        cam_up = torch.repeat_interleave(torch.einsum('c,bCc->bC', up, ext[..., :3, :3]), n_box, dim=0)
        image_ids = torch.repeat_interleave(torch.arange(2), n_box)
        from metrabs_b200.multiperson.multiperson_model import aug_parameters  # same formulas as :108-141 (checked below)
        for num_aug in (5, 2):
            gam, sc, fl, rf = aug_parameters(num_aug)
            for af in (1, 2):
                crops, new_k, rot = est._get_crops(imgs_lin, k_box, d_box, cam_up, torch.cat(boxes), image_ids, rf, sc, gam, af)
                tag = f'crops_a{num_aug}_af{af}'
                data[tag + '_idx'], data[tag] = pixel_sample(crops.reshape(-1, 3, 64, 64), seed=10 * num_aug + af)
                data[tag + '_newk'] = new_k.numpy()
                data[tag + '_rot'] = rot.numpy()
                invp = torch.linalg.inv(new_k @ rot)  # the reference's own fp32 inverse (multiperson_model.py:288, :292-295)
                if af > 1:
                    invp = invp @ wp.corner_aligned_scale_mat(1 / af)
                data[tag + '_invproj'] = invp.reshape(-1, 3, 3).numpy()
        # 12-coefficient distortion through warp_images_with_pyramid directly (warping.py:6-28, :80-99)
        d12 = torch.tensor([[-0.1, 0.03, 0.001, -0.002, 0.004, 0.02, -0.01, 0.003, 0.0005, -0.0004, 0.0003, 0.0002]]).repeat(5, 1)
        gam, sc, fl, rf = aug_parameters(5)
        _, _, _ = est._get_crops(imgs_lin, k_box, d_box, cam_up, torch.cat(boxes), image_ids, rf, sc, gam, 1)
        R0, box_scales = est._get_new_rotation_and_scale(k_box, d12, cam_up, torch.cat(boxes))
        new_k = torch.cat([torch.cat([k_box[:, :2, :2] * box_scales[:, None, None], torch.full((5, 2, 1), 32.)], dim=2),
                           torch.tensor([[[0., 0., 1.]]]).repeat(5, 1, 1)], dim=1)
        invp = torch.linalg.inv(new_k @ R0)
        c12 = wp.warp_images_with_pyramid(imgs_lin, k_box, invp, d12, box_scales, (64, 64), image_ids)
        data['d12_coeffs'] = d12.numpy()
        data['d12_invproj'] = invp.numpy()
        data['d12_scales'] = box_scales.numpy()
        data['d12_crops'] = c12.numpy()
        # ---- whole pipeline through the reference's own caller (_estimate_poses_batched, :74-185) with the reference crop model
        for avg in (True, False):
            for sk in ('', 'upper'):
                res = est._estimate_poses_batched(images, [b.clone() for b in boxes], intr, dist, ext, up, 55, 64, 1, 5, avg, sk, False)
                tag = f'pipe_avg{int(avg)}_{sk or "all"}'
                for i in range(2):
                    data[f'{tag}_p3d_{i}'] = res['poses3d'][i].numpy()
                    data[f'{tag}_p2d_{i}'] = res['poses2d'][i].numpy()
        # ---- the TTA merge alone: the reference caller around a STUB crop model that returns a fixed table of well-conditioned
        # poses (z = 2-4 m), so that mirror swap / poses @ R / joint transform / projection / extrinsics / mean are pinned
        # tightly (the tiny random crop model above emits poses with z near 0, whose 2D projection is ill-conditioned)
        g2 = torch.Generator().manual_seed(33)
        table = torch.cat([400 * torch.randn(25, 8, 2, generator=g2), 2000 + 2000 * torch.rand(25, 8, 1, generator=g2)], dim=-1)

        class TableModel(torch.nn.Module):
            joint_names, joint_edges, input_resolution = np.array(JOINT_NAMES), np.array(JOINT_EDGES), np.int32(64)

            def forward(self, inp):
                return table[:inp[0].shape[0]].clone()
        est2 = mm.Pose3dEstimator(TableModel(), skel, jt.numpy())
        data['merge_table'] = table.numpy()
        for avg in (True, False):
            for sk in ('', 'upper'):
                res = est2._estimate_poses_batched(images, [b.clone() for b in boxes], intr, dist, ext, up, 55, 0, 1, 5, avg, sk, False)
                tag = f'merge_avg{int(avg)}_{sk or "all"}'
                for i in range(2):
                    data[f'{tag}_p3d_{i}'] = res['poses3d'][i].numpy()
                    data[f'{tag}_p2d_{i}'] = res['poses2d'][i].numpy()
        res = est._estimate_poses_batched(images, [b.clone() for b in boxes], intr, dist, ext, up, 55, 10, 1, 5, True, '', False)
        for i in range(2):  # internal_batch_size 10 -> 2 boxes per crop-model call (batch-global RMS differs per chunking)
            data[f'pipe_chunk2_p3d_{i}'] = res['poses3d'][i].numpy()
    np.savez_compressed(os.path.join(OUT, 'multiperson_pipeline.npz'), **data)

    # ---- plausibility filter + pose NMS (plausibility_check.py:8-119)
    import simplepyutils as spu
    ji = StubJointInfo(JOINT_NAMES, JOINT_EDGES)
    mean_bones = torch.tensor([120., 120., 420., 420., 480., 180., 180.])
    spu.FLAGS.bone_length_dataset = None
    spu.FLAGS.bone_length_file = 'stub'
    spu.load_pickle = lambda f: mean_bones
    pc.FLAGS = spu.FLAGS
    g = torch.Generator().manual_seed(21)
    base = torch.tensor([[0., 0, 3000], [-120, 0, 3000], [120, 0, 3000], [-130, 420, 3010], [130, 420, 2990], [0, -480, 3000],
                         [-180, -480, 3000], [180, -480, 3000]])
    n_per_image = [6, 5]
    poses, boxes2 = [], []
    A = 5
    for img_i, n in enumerate(n_per_image):
        for b in range(n):
            shift = torch.tensor([400. * b - 800, 100. * img_i, 200. * b])
            p = (base + shift)[None].repeat(A, 1, 1) + 15 * torch.randn(A, 8, 3, generator=g)
            if (img_i, b) == (0, 1):
                p = poses[0] + 8 * torch.randn(A, 8, 3, generator=g)     # near-duplicate of box 0 -> NMS
            if (img_i, b) == (0, 2):
                p[:, 3] += torch.tensor([0., 2500., 0.])                 # absurd bone -> implausible
            if (img_i, b) == (0, 3):
                p = p + 900 * torch.randn(A, 8, 3, generator=g)          # augmentations disagree
            if (img_i, b) == (1, 2):
                p = poses[6] + 5 * torch.randn(A, 8, 3, generator=g)     # duplicate in image 1 (of its box 0)
            poses.append(p)
    poses3d = torch.stack(poses)  # [n, A, J, 3]
    k = torch.tensor([[1200., 0, 640], [0, 1200., 360], [0, 0, 1]])
    poses2d = torch.einsum('bank,jk->banj', poses3d / poses3d[..., 2:], k[:2])
    for i, p2 in enumerate(poses2d.mean(dim=1)):
        lo, hi = p2.min(dim=0).values, p2.max(dim=0).values
        box = torch.cat([lo - 10, hi - lo + 20, torch.tensor([0.5 + 0.04 * ((i * 7) % 11)])])
        if i == 4:
            box[:2] += 500.                                              # detection far away from the pose -> inconsistent
        boxes2.append(box)
    boxes2 = torch.stack(boxes2)
    boxes2[1, 4] = boxes2[0, 4]                                          # equal scores: stable order decides
    mean3, mean2 = poses3d.mean(dim=1), poses2d.mean(dim=1)
    plaus = pc.is_pose_plausible(mean3, ji)
    cons = pc.are_augmentation_results_consistent(poses3d)
    # reference defect: is_pose_consistent_with_box (plausibility_check.py:88-106) passes the (values, indices) tuple of
    # torch.min/max(dim=) on as if it were tf.reduce_min/max (metrabs_tf/multiperson/plausibility_check.py) and raises; the
    # function is unreachable in the PyTorch reference (call site commented out, multiperson_model.py:158-163).  Scoped shim:
    # reductions along a dim return the values, as the TF original does.
    tmin, tmax = torch.min, torch.max
    torch.min = lambda x, dim=None, **kw: tmin(x, dim=dim, **kw).values if dim is not None else tmin(x)
    torch.max = lambda x, dim=None, **kw: tmax(x, dim=dim, **kw).values if dim is not None else tmax(x)
    try:
        inbox = pc.is_pose_consistent_with_box(mean2, boxes2)
    finally:
        torch.min, torch.max = tmin, tmax
    # NOTE torch.min/max(dim=) return (values, indices) tuples: the reference's is_pose_consistent_with_box is written for
    # TF semantics; feed it through a thin wrapper if it raises
    mask = plaus & cons & inbox
    keep = torch.zeros(len(boxes2), dtype=torch.bool)
    s = 0
    for n in n_per_image:
        idx = pc.pose_non_max_suppression(mean3[s:s + n], boxes2[s:s + n, 4], mask[s:s + n])
        keep[s + idx] = True
        s += n
    np.savez_compressed(os.path.join(OUT, 'multiperson_filter.npz'), poses3d=poses3d.numpy(), poses2d=poses2d.numpy(),
                        boxes=boxes2.numpy(), n_per_image=np.array(n_per_image), bones=np.array(JOINT_EDGES),
                        mean_bones=mean_bones.numpy(), plausible_bones=plaus.numpy(), consistent=cons.numpy(), in_box=inbox.numpy(),
                        keep=keep.numpy())
    print('plausible', plaus.tolist(), '\nconsistent', cons.tolist(), '\nin_box', inbox.tolist(), '\nkeep', keep.tolist())


if __name__ == '__main__':
    main()
