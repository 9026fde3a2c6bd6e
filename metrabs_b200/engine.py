"""Thin object wrapper over the C handle (``mtb_handle``): owns the torch-allocated workspace and output tensors,
passes raw device pointers and the current CUDA stream to libmetrabs_b200.so."""
import ctypes as C
import sys
import weakref

import numpy as np
import torch

from metrabs_b200 import _lib
from metrabs_b200._lib import MtbConfig, check, lib

_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16,
           torch.int64: _lib.DTYPE_I64}


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def make_config(cfg, n_joints, stages=None, last_channel=0, arch=_lib.ARCH_EFFNET, feature_channels=0, device=0):
    c = MtbConfig()
    c.abi_version = _lib.MTB_ABI_VERSION
    c.arch = arch
    c.precision = {'fp32': _lib.PRECISION_FP32, 'bf16': _lib.PRECISION_BF16_TC,
                   'bf16_simt': _lib.PRECISION_BF16_SIMT, 'tf32x3': _lib.PRECISION_TF32X3}[cfg.precision]
    c.device = device
    c.proc_side = int(cfg.proc_side)
    c.stride_train = int(cfg.stride_train)
    c.stride_test = int(cfg.stride_test)
    c.centered_stride = int(bool(cfg.centered_stride))
    c.legacy_centered_stride_bug = int(bool(cfg.legacy_centered_stride_bug))
    c.depth = int(cfg.depth)
    c.n_joints = int(n_joints)
    c.feature_channels = int(feature_channels)
    c.box_size_mm = float(cfg.box_size_mm)
    c.mix_3d_inside_fov = -1.0 if cfg.mix_3d_inside_fov is None else float(cfg.mix_3d_inside_fov)
    c.weak_perspective = int(bool(cfg.weak_perspective))
    stages = stages or []
    if len(stages) > _lib.MTB_MAX_STAGES:
        raise ValueError('too many stages')
    c.n_stages = len(stages)
    c.last_channel = int(last_channel)
    for i, st in enumerate(stages):
        s = c.stages[i]
        s.block = 0 if st['block'] == 'fused' else 1
        s.expand, s.kernel, s.stride = st['expand'], st['kernel'], st['stride']
        s.cin, s.cout, s.layers = st['cin'], st['cout'], st['layers']
        s.bottomright = int(bool(st['bottomright']))
    return c


_live_engines = weakref.WeakSet()
# No atexit teardown: at interpreter exit the CUDA context may already be going away (cudaEventDestroy was observed to
# return cudaErrorContextIsDestroyed and then crash inside the driver); the process exit reclaims device memory.
# Engine.close() / __del__ release the handle during normal operation.


class Engine:
    def __init__(self, mtb_config):
        self._h = C.c_void_p()
        self.cfg = mtb_config
        self.device = torch.device('cuda', mtb_config.device)
        check(lib().mtb_create(C.byref(mtb_config), C.byref(self._h)))
        _live_engines.add(self)
        self._ws = None
        self._scratch = None
        hw, ch = C.c_int(), C.c_int()
        check(lib().mtb_feature_shape(self._h, C.byref(hw), C.byref(ch)), self._h)
        self.feature_side, self.feature_channels = hw.value, ch.value
        self.n_joints, self.depth = mtb_config.n_joints, mtb_config.depth
        self.feature_dtype = (torch.float32 if mtb_config.precision in (_lib.PRECISION_FP32, _lib.PRECISION_TF32X3)
                              else torch.bfloat16)

    def close(self):
        if getattr(self, '_h', None):
            lib().mtb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            if not sys.is_finalizing():
                self.close()
        except Exception:
            pass

    # ---- weights ------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict):
        """One mtb_load_weight per entry (reference key schema), then fold/repack/upload."""
        for name, t in state_dict.items():
            t = t.detach().to('cpu').contiguous()
            if t.dtype not in _DTYPES:
                t = t.float()
            shape = (C.c_int64 * max(t.ndim, 1))(*t.shape)
            check(lib().mtb_load_weight(self._h, name.encode(), C.c_void_p(t.data_ptr()), _DTYPES[t.dtype], shape,
                                        t.ndim), self._h)
        check(lib().mtb_finalize_weights(self._h), self._h)

    # ---- buffers --------------------------------------------------------------------------------------
    def workspace(self, batch):
        need = lib().mtb_workspace_bytes(self._h, batch)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws

    def _check_in(self, t, shape, dtype=torch.float32):
        if not t.is_cuda or t.device != self.device:
            raise _lib.MetrabsB200Error(f'expected a tensor on {self.device}, got {t.device} (no CPU fallback)')
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f'expected shape {tuple(shape)}, got {tuple(t.shape)}')
        if t.dtype != dtype:
            t = t.to(dtype)
        return t.contiguous()

    # ---- path stages ------------------------------------------------------------------------------------
    def backbone(self, crops):
        """[B,3,S,S] fp32 NCHW -> features NHWC [B,h,w,C]."""
        b, s = crops.shape[0], self.cfg.proc_side
        crops = self._check_in(crops, (b, 3, s, s))
        feats = torch.empty(b, self.feature_side, self.feature_side, self.feature_channels, dtype=self.feature_dtype,
                            device=self.device)
        ws = self.workspace(b)
        check(lib().mtb_backbone_forward(self._h, crops.data_ptr(), b, feats.data_ptr(), ws.data_ptr(), ws.numel(),
                                         _stream_ptr(self.device)), self._h)
        return feats

    def head_decode(self, features_nhwc):
        b = features_nhwc.shape[0]
        f = self._check_in(features_nhwc, (b, self.feature_side, self.feature_side, self.feature_channels),
                           self.feature_dtype)
        c2d = torch.empty(b, self.n_joints, 2, dtype=torch.float32, device=self.device)
        c3d = torch.empty(b, self.n_joints, 3, dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        check(lib().mtb_head_decode(self._h, f.data_ptr(), b, c2d.data_ptr(), c3d.data_ptr(), ws.data_ptr(),
                                    ws.numel(), _stream_ptr(self.device)), self._h)
        return c2d, c3d

    def reconstruct_absolute(self, coords2d, coords3d_rel, intrinsics):
        b = coords2d.shape[0]
        c2d = self._check_in(coords2d, (b, self.n_joints, 2))
        c3d = self._check_in(coords3d_rel, (b, self.n_joints, 3))
        k = self._check_in(intrinsics, (b, 3, 3))
        out = torch.empty(b, self.n_joints, 3, dtype=torch.float32, device=self.device)
        need = lib().mtb_reconstruct_scratch_bytes(b)
        if self._scratch is None or self._scratch.numel() < need:
            self._scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        check(lib().mtb_reconstruct_absolute(self._h, c2d.data_ptr(), c3d.data_ptr(), k.data_ptr(), b, out.data_ptr(),
                                             self._scratch.data_ptr(), _stream_ptr(self.device)), self._h)
        return out

    def forward(self, crops, intrinsics, out=None):
        b, s = crops.shape[0], self.cfg.proc_side
        crops = self._check_in(crops, (b, 3, s, s))
        k = self._check_in(intrinsics, (b, 3, 3))
        if out is None:
            out = torch.empty(b, self.n_joints, 3, dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        check(lib().mtb_forward(self._h, crops.data_ptr(), k.data_ptr(), b, out.data_ptr(), ws.data_ptr(), ws.numel(),
                                _stream_ptr(self.device)), self._h)
        return out

    def capture_forward(self, crops, intrinsics, out):
        """Captures one forward on fixed device buffers into a CUDA graph (mtb_forward never synchronises or allocates, so
        the ~465 launches of a step replay as one graph launch without the per-launch gaps of stream submission).
        Returns an object with ``replay()``; refill ``crops`` / ``intrinsics`` in place between replays and read ``out``.
        Run at least one plain ``forward`` on the same buffers first (tensor maps, kernel attributes, workspace)."""
        b, s = crops.shape[0], self.cfg.proc_side
        crops = self._check_in(crops, (b, 3, s, s))
        k = self._check_in(intrinsics, (b, 3, 3))
        ws = self.workspace(b)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.forward(crops, k, out=out)
        # the captured launches write into THIS workspace tensor: keep it alive with the graph even if a later, larger
        # batch makes workspace() replace self._ws (a freed workspace would be reused by the allocator under the graph)
        graph._mtb_keepalive = (crops, k, out, ws)
        return graph

    def forward_host(self, crops_host, intrinsics_host, out_host=None):
        """End-to-end call on HOST tensors (pinned for full-speed copies): H2D + forward + D2H + stream sync."""
        b = crops_host.shape[0]
        if crops_host.is_cuda or intrinsics_host.is_cuda:
            raise ValueError('forward_host takes host tensors')
        crops_host = crops_host.contiguous().float()
        intrinsics_host = intrinsics_host.contiguous().float()
        if out_host is None:
            out_host = torch.empty(b, self.n_joints, 3, dtype=torch.float32).pin_memory()
        check(lib().mtb_forward_host(self._h, crops_host.data_ptr(), intrinsics_host.data_ptr(), b,
                                     out_host.data_ptr(), _stream_ptr(self.device)), self._h)
        return out_host

    def forward_host_submit(self, crops_host, intrinsics_host, out_host, slot):
        """Pipelined end-to-end call (mtb_forward_host_submit): enqueues H2D (copy stream) + forward + D2H for this batch on
        slot 0/1 and returns at once.  Host tensors must be pinned fp32 contiguous and stay alive until
        ``forward_host_wait(slot)``; submit the next batch on the other slot before waiting and its copy overlaps this
        batch's forward."""
        for t in (crops_host, intrinsics_host, out_host):
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError('forward_host_submit takes contiguous fp32 host tensors')
        check(lib().mtb_forward_host_submit(self._h, crops_host.data_ptr(), intrinsics_host.data_ptr(), crops_host.shape[0],
                                            out_host.data_ptr(), int(slot), _stream_ptr(self.device)), self._h)

    def forward_host_wait(self, slot):
        check(lib().mtb_forward_host_wait(self._h, int(slot)), self._h)

    # ---- multi-GPU ------------------------------------------------------------------------------------------
    def comm_init(self, rank, world_size, broadcast_fn):
        """``broadcast_fn(bytes_or_None) -> bytes`` distributes rank 0's 128-byte NCCL unique id."""
        uid = C.create_string_buffer(128)
        if rank == 0:
            check(lib().mtb_comm_unique_id(uid))
        raw = broadcast_fn(bytes(uid.raw) if rank == 0 else None)
        buf = C.create_string_buffer(raw, 128)
        check(lib().mtb_comm_init(self._h, buf, rank, world_size), self._h)
        self.world_size = world_size

    def forward_sharded(self, crops_local, intrinsics_all, out=None):
        """mtb_forward_sharded: local crops [b,3,S,S] (the same b on every rank) + intrinsics of the FULL batch
        [world*b,3,3] -> joints of the full batch [world*b,J,3]; one all-gather of [c2d|c3d], full-batch reconstruction.
        Buffers (scratch, workspace, and `out` when given) are reused across calls."""
        b, s = crops_local.shape[0], self.cfg.proc_side
        crops_local = self._check_in(crops_local, (b, 3, s, s))
        k = self._check_in(intrinsics_all, (self.world_size * b, 3, 3))
        if out is None:
            out = torch.empty(self.world_size * b, self.n_joints, 3, dtype=torch.float32, device=self.device)
        need = lib().mtb_sharded_scratch_bytes(self._h, b)
        if getattr(self, '_sh_scratch', None) is None or self._sh_scratch.numel() < need:
            self._sh_scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        ws = self.workspace(b)
        check(lib().mtb_forward_sharded(self._h, crops_local.data_ptr(), b, k.data_ptr(), out.data_ptr(),
                                        self._sh_scratch.data_ptr(), ws.data_ptr(), ws.numel(), _stream_ptr(self.device)), self._h)
        return out

    def allgather(self, local, out=None):
        local = local.contiguous()
        if out is None:
            key = tuple(local.shape)
            cache = getattr(self, '_gather_out', None)
            if cache is None or cache[0] != key:  # one buffer per shape, reused across calls
                self._gather_out = (key, torch.empty((self.world_size,) + key, dtype=torch.float32, device=self.device))
            out = self._gather_out[1]
        check(lib().mtb_allgather_joints(self._h, local.data_ptr(), local.numel(), out.data_ptr(),
                                         _stream_ptr(self.device)), self._h)
        return out

    # ---- introspection ----------------------------------------------------------------------------------------
    def op_names(self):
        return [lib().mtb_op_name(self._h, i).decode() for i in range(lib().mtb_num_ops(self._h))]

    def debug_run_ops(self, crops, n_ops):
        b = crops.shape[0]
        crops = self._check_in(crops, (b, 3, self.cfg.proc_side, self.cfg.proc_side))
        hh, ww, cc = C.c_int(), C.c_int(), C.c_int()
        check(lib().mtb_op_output_shape(self._h, n_ops - 1, C.byref(hh), C.byref(ww), C.byref(cc)), self._h)
        out = torch.empty(b, hh.value, ww.value, cc.value, dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        check(lib().mtb_debug_run_ops(self._h, crops.data_ptr(), b, n_ops, out.data_ptr(), out.numel(), ws.data_ptr(),
                                      ws.numel(), _stream_ptr(self.device)), self._h)
        return out

    def op_io(self, op):
        """-> dict(in_shape=(H,W,C), out_shape=(H,W,C), residual=bool, scale=bool) of backbone op `op`."""
        a = [C.c_int() for _ in range(5)]
        check(lib().mtb_op_input_shape(self._h, op, *[C.byref(x) for x in a]), self._h)
        o = [C.c_int() for _ in range(3)]
        check(lib().mtb_op_output_shape(self._h, op, *[C.byref(x) for x in o]), self._h)
        return dict(in_shape=(a[0].value, a[1].value, a[2].value), out_shape=(o[0].value, o[1].value, o[2].value),
                    residual=bool(a[3].value), scale=bool(a[4].value))

    def debug_run_op(self, op, x, res=None, scale=None):
        """One op in isolation on fp32 device tensors (NHWC; the stem takes NCHW crops)."""
        io = self.op_io(op)
        b = x.shape[0]
        out = torch.empty((b,) + io['out_shape'], dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        x = x.float().contiguous()
        res = res.float().contiguous() if res is not None else None
        scale = scale.float().contiguous() if scale is not None else None
        check(lib().mtb_debug_run_op(self._h, op, x.data_ptr(), res.data_ptr() if res is not None else None,
                                     scale.data_ptr() if scale is not None else None, b, out.data_ptr(), out.numel(),
                                     ws.data_ptr(), ws.numel(), _stream_ptr(self.device)), self._h)
        return out

    def op_is_fused_block(self, op):
        """True when backbone op `op` (3x3 expand) and op + 1 (1x1 projection) run as one fused FusedMBConv kernel."""
        return bool(lib().mtb_op_is_fused_block(self._h, op))

    def debug_run_fused_block(self, op, x):
        """The fused FusedMBConv block starting at op `op` in isolation: x [B,H,W,Cin] fp32 (also the residual)."""
        io = self.op_io(op + 1)
        b = x.shape[0]
        out = torch.empty((b,) + io['out_shape'], dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        x = x.float().contiguous()
        check(lib().mtb_debug_run_fused_block(self._h, op, x.data_ptr(), b, out.data_ptr(), out.numel(), ws.data_ptr(),
                                              ws.numel(), _stream_ptr(self.device)), self._h)
        return out

    def op_is_expdw(self, op):
        """True when backbone op `op` (1x1 expand) and op + 1 (depthwise 3x3 + SE squeeze) run as one expdw_kernel launch."""
        return bool(lib().mtb_op_is_expdw(self._h, op))

    def debug_run_expdw(self, op, x, fused=True):
        """The expand + depthwise pair starting at op `op` in isolation, fused or as the two launches: x [B,H,W,Cin] fp32.
        Returns (depthwise output [B,H,W,Cexp], squeeze-excitation means [B,Cexp]), both fp32."""
        io = self.op_io(op + 1)
        b = x.shape[0]
        out = torch.empty((b,) + io['out_shape'], dtype=torch.float32, device=self.device)
        pooled = torch.empty((b, io['out_shape'][-1]), dtype=torch.float32, device=self.device)
        ws = self.workspace(b)
        x = x.float().contiguous()
        check(lib().mtb_debug_run_expdw(self._h, op, x.data_ptr(), b, out.data_ptr(), out.numel(), pooled.data_ptr(),
                                        pooled.numel(), 1 if fused else 0, ws.data_ptr(), ws.numel(),
                                        _stream_ptr(self.device)), self._h)
        return out, pooled

    def profile_begin(self, classes=None):
        """Brackets every launch of the selected kernel classes (None = all) with CUDA events on the launch stream."""
        n = lib().mtb_num_kernel_classes()
        mask = (1 << n) - 1 if classes is None else sum(1 << c for c in classes)
        check(lib().mtb_profile_begin(self._h, mask), self._h)

    def profile_end(self):
        """-> {class name: dict(ms, flops, bytes, launches)} for the classes that launched."""
        n = lib().mtb_num_kernel_classes()
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        la = (C.c_int64 * n)()
        check(lib().mtb_profile_end(self._h, ms, fl, by, la), self._h)
        return {lib().mtb_kernel_class_name(i).decode(): dict(cls=i, ms=ms[i], flops=fl[i], bytes=by[i], launches=la[i])
                for i in range(n) if la[i] > 0}

    def profile_op_times(self):
        """After profile_end(): [(op name, kernel class, ms, flops_per_crop, activation_bytes_per_crop, weight_bytes)] per op."""
        n = lib().mtb_num_ops(self._h)
        ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
        cl = (C.c_int * n)()
        check(lib().mtb_profile_op_times(self._h, ms, fl, by, cl, n), self._h)
        names = self.op_names()
        return [(names[i], lib().mtb_kernel_class_name(cl[i]).decode(), ms[i], fl[i], by[i],
                 float(lib().mtb_op_weight_bytes(self._h, i))) for i in range(n)]

    @property
    def last_launch_count(self):
        return int(lib().mtb_last_launch_count(self._h))

    @property
    def backbone_flops_per_crop(self):
        return float(lib().mtb_backbone_flops_per_crop(self._h))


def soft_argmax_device(logits, layout, n_joints, depth, height, width):
    """Standalone soft-argmax on materialised logits (mtb_softargmax).  Returns (out2d, out3d)."""
    if not logits.is_cuda:
        raise _lib.MetrabsB200Error('soft_argmax needs a CUDA tensor (no CPU fallback)')
    if logits.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        logits = logits.float()
    logits = logits.contiguous()
    dev = logits.device
    if layout == _lib.LAYOUT_BDJHW:
        b = logits.shape[0]
        out2d = out3d = None
        if depth == 0:
            out2d = torch.empty(b, n_joints, 2, dtype=torch.float32, device=dev)
        else:
            out3d = torch.empty(b, n_joints, 3, dtype=torch.float32, device=dev)
    else:
        b = logits.shape[0]
        out2d = torch.empty(b, n_joints, 2, dtype=torch.float32, device=dev)
        out3d = torch.empty(b, n_joints, 3, dtype=torch.float32, device=dev) if depth > 0 else None
    with torch.cuda.device(dev):
        check(lib().mtb_softargmax(
            logits.data_ptr(), _DTYPES[logits.dtype], layout, b, n_joints, depth, height, width,
            out2d.data_ptr() if out2d is not None else None, out3d.data_ptr() if out3d is not None else None,
            _stream_ptr(dev)))
    return out2d, out3d
