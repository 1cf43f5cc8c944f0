"""The training batch of ``MonoDataset`` built on the GPU (SURVEY.md 8f-3).

The reference's ``__getitem__`` + ``preprocess`` (/root/reference/datasets/mono_dataset.py:90-109,136-185) flips, resizes
to four scales with Pillow's LANCZOS and colour-jitters every frame of every sample on the host.  Here a dataloader worker
only decodes the frames and makes the reference's random draws (``NativeFramesMixin``); ``collate_native`` packs the
native uint8 frames, the draws and the job table into one flat buffer (one host-to-device copy per batch), and
``MonoBatch`` builds the ``inputs`` dict ``Trainer.process_batch`` consumes in 2 * num_scales + 3 launches
(``md2_batch_build_u8``), byte for byte what default collation of the reference's items gives.

    loader = DataLoader(GpuKITTIRAW(...), batch_size=12, shuffle=True, num_workers=12, pin_memory=True,
                        collate_fn=collate_native)
    build = MonoBatch(opt.height, opt.width, opt.frame_ids, len(opt.scales))
    for native in loader:
        inputs = build(native)          # ("color", f, s), ("color_aug", f, s), ("K", s), ("inv_K", s), stereo_T, ...
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import random
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _capi, jpeg, kitti_depth
from .pyramid import ColorAug

# KITTIDataset.K (kitti_dataset.py): intrinsics normalised by the image size
KITTI_K = np.array([[0.58, 0, 0.5, 0],
                    [0, 1.92, 0.5, 0],
                    [0, 0, 1, 0],
                    [0, 0, 0, 1]], dtype=np.float32)

# md2_batch_job of include/md2_loss.h
JOB_DTYPE = np.dtype([("offset", "<i8"), ("height", "<i4"), ("width", "<i4"), ("size", "<i4"), ("flip", "<i4"),
                      ("sample", "<i4"), ("reserved", "<i4")])
_PARAM_BYTES = 32           # one md2_color_jitter row
_STEREO_BYTES = 64          # one 4x4 float32 stereo_T
_DRAW_KEYS = ("frames", "do_color_aug", "do_flip", "color_aug", "side", "velodyne")


def _align(n: int, a: int = 16) -> int:
    return (n + a - 1) // a * a


@dataclasses.dataclass
class NativeBatch:
    """A batch as ``collate_native`` packs it.  ``buffer`` is one flat uint8 tensor: the jitter rows (``ColorAug.pack_params``
    layout, one per sample), the stereo_T matrices (when ``"s"`` is a frame), the job table (``JOB_DTYPE``, image
    ``fi * batch_size + b`` is frame ``frame_ids[fi]`` of sample ``b``) and the native HWC frames.  The draws stay
    readable: ``do_color_aug`` / ``do_flip`` (B,) bool, ``color_aug`` the ``ColorJitter.get_params`` tuple or None per
    sample, ``side`` per sample; ``extra`` holds the dataset's other keys (``depth_gt``), default-collated.  Items from
    ``VelodyneDepthMixin`` add the ``md2_velo_job`` table at ``velo_jobs_offset``, between the frames' job table and the
    frames (so, like every other offset but the scans', it depends only on the batch size and the frame ids), and the
    scans after the frames; ``velo_out_shape`` is the size of the depth_gt they give."""
    buffer: torch.Tensor
    batch_size: int
    frame_ids: list
    params_offset: int
    stereo_offset: int          # -1 without "s"
    jobs_offset: int
    frames_offset: int
    do_color_aug: torch.Tensor
    do_flip: torch.Tensor
    color_aug: list
    side: list
    extra: dict
    velo_jobs_offset: int = -1  # -1 without velodyne scans
    velo_out_shape: Optional[tuple] = None
    # Items from JpegFramesMixin: the md2_jpeg_job table of the JPEG frames at jpeg_jobs_offset (after the scans' job
    # table, so its place depends only on the batch size and the frame ids), their compressed streams after the
    # frames and scans.  The job table's frame offsets then index a device native-frame buffer of native_bytes, into
    # which the JPEG frames are decoded and the host-decoded frames (jpeg_copies: (offset in buffer, offset in that
    # device buffer, bytes)) are copied.
    jpeg_jobs_offset: int = -1
    jpeg_names: Optional[list] = None
    jpeg_chunks: int = 0
    jpeg_blocks: int = 0
    native_bytes: int = 0
    jpeg_copies: Optional[list] = None

    @property
    def n_images(self) -> int:
        return self.batch_size * len(self.frame_ids)

    def jobs(self) -> np.ndarray:
        """The job table as a numpy view of ``buffer`` (host buffers only)."""
        a = self.jobs_offset
        return self.buffer[a:a + self.n_images * JOB_DTYPE.itemsize].numpy().view(JOB_DTYPE)

    def pin_memory(self) -> "NativeBatch":
        """Called by ``DataLoader(pin_memory=True)``: the workers cannot pin, the loader's pinning thread can."""
        return self if self.buffer.is_pinned() else dataclasses.replace(self, buffer=self.buffer.pin_memory())


def collate_native(items: List[dict], pin_memory: Optional[bool] = None) -> NativeBatch:
    """``collate_fn`` for a dataset that returns ``NativeFramesMixin`` items.  ``pin_memory=None`` pins when called in
    the main process of a CUDA machine (inside a worker, ``DataLoader(pin_memory=True)`` pins through
    ``NativeBatch.pin_memory``)."""
    from torch.utils.data import default_collate, get_worker_info
    B = len(items)
    fids = list(items[0]["frames"].keys())
    for it in items:
        if list(it["frames"].keys()) != fids:
            raise ValueError("every item of a batch must hold the same frame ids")
    n = B * len(fids)
    frames = [items[b]["frames"][f] for f in fids for b in range(B)]
    frames = [a if isinstance(a, jpeg.JpegStream) else np.ascontiguousarray(a, dtype=np.uint8) for a in frames]
    streams = [a for a in frames if isinstance(a, jpeg.JpegStream)]
    for a in frames:
        if isinstance(a, jpeg.JpegStream):
            continue
        if a.ndim != 3 or a.shape[2] != 3:
            raise ValueError("native frames must be (h, w, 3) uint8 arrays, got %s" % (a.shape,))
    stereo = "s" in fids
    off = B * _PARAM_BYTES
    stereo_off = off if stereo else -1
    off += B * _STEREO_BYTES if stereo else 0
    jobs_off = off
    off = _align(off + n * JOB_DTYPE.itemsize)
    velo = [it["velodyne"] for it in items] if "velodyne" in items[0] else None
    velo_off = -1
    if velo is not None:        # the scans' job table ahead of the frames: its offset depends on B alone, so a graph
        if any(tuple(v.out_shape) != tuple(velo[0].out_shape) for v in velo):    # captured on one batch serves all
            raise ValueError("every velodyne scan of a batch must give the same depth_gt size")
        velo_off = off
        off = _align(off + B * kitti_depth.VELO_JOB_DTYPE.itemsize)
    jpeg_off = -1
    if streams:
        jpeg_off = off
        off = _align(off + len(streams) * jpeg.JOB_DTYPE.itemsize, 64)
    frames_off = off
    rel, total = [], 0
    for a in frames:
        rel.append(total)
        total = _align(total + a.nbytes)
    native_total = total
    copies = None
    if streams:                 # the buffer holds only the host-decoded frames; rel indexes the device frame buffer
        copies, total = [], 0
        for a, r in zip(frames, rel):
            if not isinstance(a, jpeg.JpegStream):
                copies.append((frames_off + total, r, a.nbytes))
                total = _align(total + a.nbytes)
    if velo is not None:        # the scans after the frames; their job records hold their offsets
        scans_off = frames_off + total
        total += kitti_depth.packed_bytes(velo)
    if streams:
        body_off = _align(frames_off + total, 64)
        total = body_off - frames_off + jpeg.body_bytes(streams)
    if pin_memory is None:
        pin_memory = get_worker_info() is None and torch.cuda.is_available()
    buf = torch.empty(frames_off + total, dtype=torch.uint8, pin_memory=bool(pin_memory))
    h = buf.numpy()
    draws = [it["color_aug"] for it in items]
    params = ColorAug.pack_params([d if d is not None else ((), None, None, None, None) for d in draws]).numpy()
    h[:B * _PARAM_BYTES] = params.view(np.uint8).reshape(-1)
    do_flip = [bool(it["do_flip"]) for it in items]
    sides = [it["side"] for it in items]
    if stereo:
        st = np.zeros((B, 4, 4), np.float32)
        for b in range(B):                      # as MonoDataset.__getitem__ does
            stereo_T = np.eye(4, dtype=np.float32)
            baseline_sign = -1 if do_flip[b] else 1
            side_sign = -1 if sides[b] == "l" else 1
            stereo_T[0, 3] = side_sign * baseline_sign * 0.1
            st[b] = stereo_T
        h[stereo_off:stereo_off + B * _STEREO_BYTES] = st.view(np.uint8).reshape(-1)
    jobs = h[jobs_off:jobs_off + n * JOB_DTYPE.itemsize].view(JOB_DTYPE)
    for i, a in enumerate(frames):
        jobs[i] = (rel[i], a.shape[0], a.shape[1], -1, int(do_flip[i % B]), i % B, 0)
    if copies is None:
        for a, r in zip(frames, rel):
            h[frames_off + r:frames_off + r + a.nbytes] = a.reshape(-1)
    else:
        for a, (src, _, nb) in zip([a for a in frames if not isinstance(a, jpeg.JpegStream)], copies):
            h[src:src + nb] = a.reshape(-1)
    if velo is not None:
        kitti_depth.pack_jobs(h, velo_off, scans_off, velo, do_flip, False)
    chunks = blocks = 0
    if streams:
        chunks, blocks = jpeg.pack(h, jpeg_off, body_off, streams,
                                   [r for a, r in zip(frames, rel) if isinstance(a, jpeg.JpegStream)])
    extra_keys = [k for k in items[0] if k not in _DRAW_KEYS]
    extra = default_collate([{k: it[k] for k in extra_keys} for it in items]) if extra_keys else {}
    return NativeBatch(buf, B, fids, 0, stereo_off, jobs_off, frames_off,
                       torch.tensor([bool(it["do_color_aug"]) for it in items]), torch.tensor(do_flip), draws, sides, extra,
                       velo_off, tuple(velo[0].out_shape) if velo is not None else None, jpeg_off,
                       [s.name for s in streams], chunks, blocks, native_total, copies)


class NativeFramesMixin:
    """Put in front of a reference dataset class: ``class GpuKITTIRAW(NativeFramesMixin, KITTIRAWDataset)``.

    ``__getitem__`` makes the reference's random draws in the reference's order (mono_dataset.py:136-185: do_color_aug,
    do_flip, then ``ColorJitter.get_params`` only when augmenting) and loads every frame with the dataset's own
    ``get_color(folder, index, side, False)``, unflipped and unresized: the flip, the pyramid and the jitter run in
    ``MonoBatch``.  ``depth_gt`` is the dataset's own host code (``native_depth``), unless ``VelodyneDepthMixin`` is
    put in front."""

    def __getitem__(self, index):
        from torchvision import transforms
        do_color_aug = self.is_train and random.random() > 0.5
        do_flip = self.is_train and random.random() > 0.5
        line = self.filenames[index].split()
        folder = line[0]
        frame_index = int(line[1]) if len(line) == 3 else 0
        side = line[2] if len(line) == 3 else None
        frames = {}
        for i in self.frame_idxs:
            if i == "s":
                other_side = {"r": "l", "l": "r"}[side]
                frames[i] = self.native_color(folder, frame_index, other_side)
            else:
                frames[i] = self.native_color(folder, frame_index + i, side)
        color_aug = None
        if do_color_aug:       # a tuple in the installed torchvision (SURVEY.md B.2); MonoBatch applies it
            color_aug = transforms.ColorJitter.get_params(self.brightness, self.contrast, self.saturation, self.hue)
        item = {"frames": frames, "do_color_aug": bool(do_color_aug), "do_flip": bool(do_flip), "color_aug": color_aug,
                "side": side}
        if self.load_depth:
            item.update(self.native_depth(folder, frame_index, side, do_flip))
        return item

    def native_color(self, folder, frame_index, side):
        """A native frame: the dataset's ``get_color(folder, frame_index, side, False)`` as an (h, w, 3) uint8 array
        (``JpegFramesMixin`` returns the parsed JPEG instead)."""
        return np.array(self.get_color(folder, frame_index, side, False))

    def native_depth(self, folder, frame_index, side, do_flip) -> dict:
        """The item's depth keys: ``depth_gt`` from the dataset's ``get_depth``, as MonoDataset.__getitem__ does."""
        depth_gt = self.get_depth(folder, frame_index, side, do_flip)
        return {"depth_gt": torch.from_numpy(np.expand_dims(depth_gt, 0).astype(np.float32))}


class MonoBatch:
    """``MonoBatch(height, width, frame_ids, num_scales)(native) -> inputs`` with the keys and shapes default collation of
    ``MonoDataset.__getitem__`` gives: ``("color", f, s)`` (B,3,h_s,w_s) uint8 (or float32 ``ToTensor`` values with
    ``color_dtype=torch.float32``), ``("color_aug", f, s)`` float32, ``("K", s)`` / ``("inv_K", s)`` (B,4,4) float32,
    ``"stereo_T"`` when ``"s"`` is a frame, ``"depth_gt"`` built from the scans (``md2_velo_depth``, three launches) when
    the items came from ``VelodyneDepthMixin``, and the dataset's other keys.  uint8 ``color`` is what the fused loss's uint8
    entry takes.  The K / inv_K tensors are shared between calls with the same batch size: treat them as read-only.

    The first batch that holds a new native size builds that size's tables (synchronous); after that a call only
    enqueues work, and ``build`` alone can be captured in a CUDA graph.

    Batches of ``JpegFramesMixin`` items are decoded on the device first (``md2_jpeg_decode``) into a native-frame
    buffer.  ``jpeg_capacity = (native_bytes, entropy_bytes, blocks)`` sizes that buffer and the decoder's scratch
    (``entropy_bytes`` counts each restart segment rounded up to whole 64-byte chunks, as ``collate_native`` lays them
    out); a batch over it raises before anything is enqueued.  With a capacity, a graph captured on one batch replays
    batches of other compressed lengths and native sizes that hold as many JPEG frames and no host-decoded frame;
    without, each batch is sized to itself.  ``jpeg_status`` is the device status word of every JPEG frame of the last
    build (read without synchronising); ``check_jpeg()`` synchronises and raises naming the corrupt files."""

    def __init__(self, height: int, width: int, frame_ids, num_scales: int = 4, K=None,
                 color_dtype: torch.dtype = torch.uint8, device=None, jpeg_capacity=None):
        if color_dtype not in (torch.uint8, torch.float32):
            raise ValueError("color_dtype must be torch.uint8 or torch.float32")
        self.height, self.width, self.num_scales = int(height), int(width), int(num_scales)
        self.frame_ids = list(frame_ids)
        self.color_dtype = color_dtype
        dev = torch.device(device if device is not None else "cuda")
        self.device = dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.lib = _capi.load_library()
        self._plan = C.c_void_p()
        _capi.check(self.lib, self.lib.md2_batch_plan_create(self.height, self.width, self.num_scales, C.byref(self._plan)),
                    "md2_batch_plan_create")
        self._sizes: Dict[tuple, int] = {}
        K = KITTI_K if K is None else np.asarray(K, dtype=np.float32)
        self._K = []
        for scale in range(self.num_scales):        # as MonoDataset.__getitem__ does
            Ks = K.copy()
            Ks[0, :] *= self.width // (2 ** scale)
            Ks[1, :] *= self.height // (2 ** scale)
            self._K.append((Ks, np.linalg.pinv(Ks)))
        self._k_cache: Dict[int, dict] = {}
        self.jpeg_capacity = None if jpeg_capacity is None else tuple(int(v) for v in jpeg_capacity)
        self.jpeg_status: Optional[torch.Tensor] = None
        self._jpeg_names: list = []

    def __del__(self):
        try:
            self.lib.md2_batch_plan_destroy(self._plan)
        except Exception:
            pass

    def _size_index(self, h: int, w: int) -> int:
        idx = self._sizes.get((h, w))
        if idx is None:
            i = C.c_int(-1)
            with torch.cuda.device(self.device):
                _capi.check(self.lib, self.lib.md2_batch_plan_add_native_size(self._plan, h, w, C.byref(i)),
                            "md2_batch_plan_add_native_size")
            idx = self._sizes[(h, w)] = i.value
        return idx

    def _intrinsics(self, B: int) -> dict:
        d = self._k_cache.get(B)
        if d is None:
            d = {}
            for s, (K, inv_K) in enumerate(self._K):
                d[("K", s)] = torch.from_numpy(np.stack([K] * B)).to(self.device)
                d[("inv_K", s)] = torch.from_numpy(np.stack([inv_K] * B)).to(self.device)
            self._k_cache[B] = d
        return d

    def upload(self, native: NativeBatch) -> torch.Tensor:
        """Writes the plan's size indices into the job table and copies the packed batch to the device (one copy,
        asynchronous from pinned memory)."""
        if list(native.frame_ids) != self.frame_ids:
            raise ValueError("batch holds frames %s, MonoBatch was made for %s" % (native.frame_ids, self.frame_ids))
        jobs = native.jobs()
        jobs["size"] = [self._size_index(int(h), int(w)) for h, w in zip(jobs["height"], jobs["width"])]
        return native.buffer.to(self.device, non_blocking=True)

    def build(self, native: NativeBatch, flat: torch.Tensor) -> Dict:
        """The inputs dict from ``flat``, the device copy ``upload`` made of ``native.buffer``."""
        B, F, S = native.batch_size, len(self.frame_ids), self.num_scales
        n = native.n_images
        dev = flat.device
        planes = [(self.height >> s) * (self.width >> s) for s in range(S)]
        total = 3 * n * sum(planes)
        color = torch.empty(total, dtype=self.color_dtype, device=dev)
        color_aug = torch.empty(total, dtype=torch.float32, device=dev)
        f32 = int(self.color_dtype == torch.float32)
        nb = C.c_size_t(0)
        _capi.check(self.lib, self.lib.md2_batch_scratch_bytes(self._plan, n, f32, C.byref(nb)), "md2_batch_scratch_bytes")
        scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
        base = flat.data_ptr()
        frames_ptr, frames_bytes = base + native.frames_offset, flat.numel() - native.frames_offset
        if native.jpeg_jobs_offset >= 0:
            frames = self._decode_jpeg(native, flat)
            frames_ptr, frames_bytes = frames.data_ptr(), frames.numel()
        with torch.cuda.device(dev):
            st = self.lib.md2_batch_build_u8(
                self._plan, frames_ptr, frames_bytes,
                native.buffer.data_ptr() + native.jobs_offset, base + native.jobs_offset, n,
                base + native.params_offset, B, color.data_ptr(), f32, color_aug.data_ptr(), scratch.data_ptr(),
                scratch.numel(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _capi.check(self.lib, st, "md2_batch_build_u8")
        inputs = dict(self._intrinsics(B))
        off = 0
        for s in range(S):
            h, w = self.height >> s, self.width >> s
            lv = color[off:off + 3 * n * planes[s]].view(F, B, 3, h, w)
            lva = color_aug[off:off + 3 * n * planes[s]].view(F, B, 3, h, w)
            for fi, f in enumerate(self.frame_ids):
                inputs[("color", f, s)] = lv[fi]
                inputs[("color_aug", f, s)] = lva[fi]
            off += 3 * n * planes[s]
        for k, v in native.extra.items():
            inputs[k] = v.to(dev, non_blocking=True) if torch.is_tensor(v) else v
        if native.velo_jobs_offset >= 0:
            inputs["depth_gt"] = kitti_depth.run(self.lib, flat, native.buffer.data_ptr() + native.velo_jobs_offset,
                                                 native.velo_jobs_offset, B, native.velo_out_shape)
        if native.stereo_offset >= 0:
            a = native.stereo_offset
            inputs["stereo_T"] = flat[a:a + B * _STEREO_BYTES].view(torch.float32).view(B, 4, 4)
        return inputs

    def _decode_jpeg(self, native: NativeBatch, flat: torch.Tensor) -> torch.Tensor:
        """The device native-frame buffer of a batch with JPEG frames: decoded, and the host-decoded frames copied."""
        cap = self.jpeg_capacity or (native.native_bytes, native.jpeg_chunks * jpeg.CHUNK_BYTES, native.jpeg_blocks)
        need = (native.native_bytes, native.jpeg_chunks * jpeg.CHUNK_BYTES, native.jpeg_blocks)
        if any(n > c for n, c in zip(need, cap)):
            raise ValueError("batch needs (native bytes, entropy bytes, blocks) = %s, over MonoBatch's jpeg_capacity %s"
                             % (need, cap))
        n = len(native.jpeg_names)
        frames = torch.empty(cap[0], dtype=torch.uint8, device=flat.device)
        for src, dst, nbytes in native.jpeg_copies:        # host-decoded frames: one cudaMemcpyAsync each
            frames[dst:dst + nbytes].copy_(flat[src:src + nbytes], non_blocking=True)
        status = torch.empty(n, dtype=torch.int32, device=flat.device)
        jpeg.run(self.lib, flat, native.buffer.data_ptr() + native.jpeg_jobs_offset, native.jpeg_jobs_offset, n, frames,
                 status, max(1, cap[1] // jpeg.CHUNK_BYTES), max(1, cap[2]))
        self.jpeg_status, self._jpeg_names = status, list(native.jpeg_names)
        return frames

    def check_jpeg(self) -> None:
        """Synchronises and raises ValueError naming every JPEG file of the last build whose data was corrupt."""
        if self.jpeg_status is None:
            return
        err = jpeg.status_error(self.jpeg_status.cpu().tolist(), self._jpeg_names)
        if err:
            raise ValueError(err)

    def __call__(self, native: NativeBatch) -> Dict:
        return self.build(native, self.upload(native))
