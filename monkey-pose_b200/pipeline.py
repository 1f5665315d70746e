"""Camera frames -> joints on the device: the inference loop of the reference (`test_model` / `eval_model_on_real_data`,
train_cnn_networks_hgru.py:264-419 -- attention CNN, `prepare_data_test`, pose network, x cube[2]/2,
`getAbsoluteCoordinates`, one frame at a time through two `sess.run` calls and a host crop) for a whole batch with no
host round trip between the stages, and with the upload of the frames overlapped with the attention CNN:

    frames (pinned host, [N,H,W] float32 in [0,1] -- or raw 16-bit millimetres, converted on the device)
      --H2D in `chunks` pieces on a copy stream-->  attention CNN per piece as it lands  -->  centres of mass (device)
      --> window arithmetic + crop (device) --> pose network (fused tensor-core forward) --> absolute joints (device)
      --D2H--> xyz, uvd [N,23,3]

Without an attention network (`attn=None`) the centres come from the detector itself, as `cropArea3D` does when
none is given (tf_monkeydetector.py:303-308: `calculateCoM` of each frame, optionally refined on the first crop,
`docom`, :316-333) -- also on the device.

Everything numerical runs in libhgru_b200.so; this module only orders the calls on two CUDA streams.  No CPU fallback.
"""
import torch

from .tf_monkeydetector import prepare_data_test, preprocess_real_depth


class FramesToJoints(object):
    """attn: `attn_model_struct` (or None: centres of mass estimated from the frames by the detector, refined on the
    first crop when `docom`); its `compute_mode` ('bf16x3' or 'fp16') sets the attention CNN's arithmetic.
    pose: `model` (parameters loaded), md: `tfMonkeyDetector`, config: an object with `image_orig_size`,
    `image_target_size`, `image_max_depth` (the reference's `monkeyConfig`), cube_z: seqconfig ['cube'][2]
    (mm).  `chunks`: pieces the upload is cut into (the attention CNN starts on piece c while piece c+1 is
    on the bus); 1 = plain stream order."""

    def __init__(self, attn, pose, md, config, cube_z=1200.0, num_joints=23, chunks=4, near=1000, far=3000,
                 docom=False):
        self.attn, self.pose, self.md, self.config = attn, pose, md, config
        self.docom = bool(docom)
        self.scale = float(cube_z) / 2.0
        self.out_dims = 3 * int(num_joints)
        self.chunks = int(chunks)
        self.near, self.far = int(near), int(far)      # raw 16-bit input: train_cnn_networks_hgru.py:383-384
        self._raw_dev = None
        self._copy_stream = None
        self._frames_dev = None
        self._events = None

    def _buffers(self, shape, device):
        if self._frames_dev is None or tuple(self._frames_dev.shape) != tuple(shape):
            self._frames_dev = torch.empty(shape, device=device, dtype=torch.float32)
            self._tr = torch.empty((shape[0], 3), device=device, dtype=torch.float32)
            self._copy_stream = torch.cuda.Stream(device=device)
            self._events = [torch.cuda.Event() for _ in range(max(1, self.chunks))]
        return self._frames_dev

    def __call__(self, frames, centres=None):
        """frames: [N,H,W] float32 in [0,1], pinned host memory (or a CUDA tensor: then nothing is uploaded) -- or raw
        16-bit depth in millimetres (uint16 / int16, pinned host): half the upload, thresholded and normalised on the
        device as eval_model_on_real_data does on the host (:381-386).
        centres: optional CUDA float32 [N,3] replacing the attention CNN's output (it still runs).
        Returns (xyz, uvd): [N,J,3] float32 on the host (pinned), camera-space mm and image-space (u, v, d)."""
        if frames.dim() == 4:
            frames = frames[..., 0]
        N = int(frames.shape[0])
        main = torch.cuda.current_stream()
        raw16 = (not frames.is_floating_point()) and frames.element_size() == 2
        if frames.is_cuda:
            dev_frames = preprocess_real_depth(frames, self.near, self.far, max_depth=self.config.image_max_depth) \
                if raw16 else frames.to(torch.float32).contiguous()
            pieces = [(0, N)]
            self._buffers(frames.shape, frames.device)
        else:
            dev_frames = self._buffers(frames.shape, torch.device("cuda", torch.cuda.current_device()))
            # equal pieces only (one attention plan serves them all); small or indivisible batches go up in one piece
            nch = self.chunks if (self.chunks > 1 and N >= 4 * self.chunks and N % self.chunks == 0) else 1
            per = (N + nch - 1) // nch
            pieces = [(lo, min(lo + per, N)) for lo in range(0, N, per)]
            if raw16 and (self._raw_dev is None or tuple(self._raw_dev.shape) != tuple(frames.shape)
                          or self._raw_dev.dtype != frames.dtype):
                self._raw_dev = torch.empty(frames.shape, device=dev_frames.device, dtype=frames.dtype)
            target = self._raw_dev if raw16 else dev_frames
            self._copy_stream.wait_stream(main)                 # the previous call's readers are done with the buffer
            with torch.cuda.stream(self._copy_stream):
                for i, (lo, hi) in enumerate(pieces):
                    target[lo:hi].copy_(frames[lo:hi], non_blocking=True)
                    self._events[i].record(self._copy_stream)
        for i, (lo, hi) in enumerate(pieces):
            if not frames.is_cuda:
                main.wait_event(self._events[i])
                if raw16:
                    preprocess_real_depth(self._raw_dev[lo:hi], self.near, self.far,
                                          max_depth=self.config.image_max_depth, out=dev_frames[lo:hi])
            if self.attn is not None:
                self._tr[lo:hi] = self.attn.build(dev_frames[lo:hi], 3)              # train_cnn_networks_hgru.py:281-283
        if self.attn is None and centres is None:
            # no attention output: the detector's own estimate (tf_monkeydetector.py:303-308, 316-333)
            ts, md_ = self.config.image_target_size, self.config.image_max_depth
            patches, _, coms = self.md.cropArea3D_batch_device(dev_frames, dsize=(ts[1], ts[0]), frame_scale=md_,
                                                               out_divisor=md_, docom=self.docom)
            patches = patches[..., None]
        else:
            tr = self._tr if centres is None else centres
            patches, coms, _ = prepare_data_test(dev_frames, tr, self.md, self.config)   # :284 (windows on the device)
        out = self.pose.build(patches, self.out_dims)                                # :291-294
        xyz, uvd = self.md.getAbsoluteCoordinates_batch(out, coms, self.scale)       # :295-298
        xyz_h = torch.empty(xyz.shape, dtype=torch.float32, pin_memory=True)
        uvd_h = torch.empty(uvd.shape, dtype=torch.float32, pin_memory=True)
        xyz_h.copy_(xyz, non_blocking=True)
        uvd_h.copy_(uvd, non_blocking=True)
        main.synchronize()
        return xyz_h, uvd_h


class StreamedForward(object):
    """A stream of host batches through `model.build`, double-buffered: while batch i runs, batch i+1 is copied to the
    device on a second stream and the predictions of batch i-1 travel back -- the role the reference gives its input
    queues (`tf.train.shuffle_batch(..., num_threads=2, capacity=...)`, data_loader.py:38, started by
    `tf.train.start_queue_runners`, train_cnn_networks_hgru.py:200-201,309-310: the next batch is staged while
    `sess.run` computes).  Per-batch results are bitwise those of `model.build(batch, output_shape)`; only the order
    of the copies changes.  Everything numerical runs in libhgru_b200.so; no CPU fallback.

        for out in StreamedForward(m, 69)(batches):      # batches: iterable of pinned [N,128,128,1] float32 tensors
            ...                                          # out: [N,69] float32 on the host, in batch order
    """

    def __init__(self, pose, output_shape):
        self.pose, self.output_shape = pose, int(output_shape)
        self._shape = None

    def _buffers(self, shape, device):
        if self._shape != tuple(shape):
            if self._shape is not None:          # (the caller has drained the stream: see __call__)
                self._copy.synchronize()
                torch.cuda.current_stream().synchronize()
            self._shape = tuple(shape)
            self._dev = [torch.empty(shape, device=device, dtype=torch.float32) for _ in range(2)]
            self._host = [torch.empty((shape[0], self.output_shape), dtype=torch.float32, pin_memory=True)
                          for _ in range(2)]
            self._copy = torch.cuda.Stream(device=device)
            self._landed = [torch.cuda.Event() for _ in range(2)]
            self._consumed = [torch.cuda.Event() for _ in range(2)]
            self._done = [torch.cuda.Event() for _ in range(2)]

    def __call__(self, batches):
        device = torch.device("cuda", torch.cuda.current_device())
        main = torch.cuda.current_stream()
        pending = None                       # slot whose predictions are on their way back
        i = 0                                # batches since the buffers were (re)made
        for b in batches:
            if b.is_cuda:
                raise ValueError("StreamedForward takes host batches (use model.build for device tensors)")
            if b.dim() == 3:
                b = b[..., None]
            if self._shape is not None and self._shape != tuple(b.shape):
                # a new batch shape mid-stream: hand out what is in flight, then start over with new buffers
                if pending is not None:
                    self._done[pending].synchronize()
                    yield self._host[pending].clone()
                    pending = None
                i = 0
            self._buffers(b.shape, device)
            s = i & 1
            if i >= 2:
                self._copy.wait_event(self._consumed[s])         # batch i-2 has been read out of this buffer
            else:
                self._copy.wait_stream(main)
            with torch.cuda.stream(self._copy):
                self._dev[s].copy_(b, non_blocking=True)
                self._landed[s].record(self._copy)
            main.wait_event(self._landed[s])
            out = self.pose.build(self._dev[s], self.output_shape)
            self._consumed[s].record(main)
            if pending is not None:                              # hand batch i-1 out while batch i runs
                self._done[pending].synchronize()
                yield self._host[pending].clone()
            self._host[s].copy_(out, non_blocking=True)
            self._done[s].record(main)
            pending = s
            i += 1
        if pending is not None:
            self._done[pending].synchronize()
            yield self._host[pending].clone()
