"""`attn_model_struct` -- mirror of the reference's attention (centre-of-mass) CNN class
(train_cnn_networks_hgru.py:422-525), the network that runs right before the crop stage: same constructor, same
`build(depth, output_shape, batch_norm=None, train_mode=None)`, same attribute names (`pool1` .. `pool5`, `fc1`,
`relu1`, `fcout`, `out_put`), same `data_dict[name][idx]` weight injection and `var_dict[(name, idx)]` registry
(:615-633).  `depth` is a torch CUDA tensor [N,H,W,1] (or [N,H,W]) instead of a tf.Tensor; the forward runs in
libhgru_b200.so (`attn_*` entry points of include/hgru_b200.h) -- there is no CPU fallback.

`train_mode` in (None, False): the fused tensor-core pipeline, inference-mode batch norm (moving statistics), with the
GEMM layers (aconv_2 .. aconv_5, afc_1) in `compute_mode`: 'bf16x3' (default: bf16 hi/lo operand splits, three
products per k-step, fp32-class accuracy, <= 1e-4 relative) or 'fp16' (fp16 operands, one product per k-step at the
bf16 rate, fp32 accumulation: <= 2.5e-3 relative on every activation).  aconv_1 and afc_out are fp32 in both.
`train_mode=True` -- what the reference passes both in training (:117) and, as committed, in
`eval_model_on_real_data` (:360) -- composes the graph layer by layer from the class's own layer methods
(`monkey_pose_b200.layers.LayerOps`): batch statistics in the six batch norms, dropout keep 0.7 after relu(afc_1)
with the documented counter-based mask, moving-statistics updates in `updated_moving_stats`.  Forward only.  It
keeps its exact fp32 layer path whatever `compute_mode` says.
Non-reference knobs: `widths`, `fc_hidden` (defaults = the reference's 64..1024 / 1024), `compute_mode`, `seed`,
`dropout_seed`.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import initialization as init
from .hgru_module import _as_dev, _stream
from .layers import LayerOps

_BN_FIELDS = ("gamma", "beta", "moving_mean", "moving_variance")
_MODES = ("bf16x3", "fp16")        # compute_mode -> HGRU_MODE_* through _lib.MODES


class attn_model_struct(LayerOps):
    _bn_scopes = init.ATTN_BN_SCOPES

    def __init__(self, trainable=True):
        self.trainable = trainable
        self.data_dict = None
        self.var_dict = {}
        self._BATCH_NORM_DECAY = 0.997
        self._BATCH_NORM_EPSILON = 1e-5
        # ---- non-reference knobs (defaults reproduce the reference's shapes) ----
        self.widths = (64, 128, 256, 512, 1024)     # :443, :456, :469, :482, :495
        self.fc_hidden = 1024                        # :501 (and hard-coded again at :522)
        self.compute_mode = 'bf16x3'
        self.seed = 42
        self.dropout_seed = 1234
        self._plan = None
        self._plan_key = None
        self._plan_capacity = 0                      # frames the plan was created for: it runs every batch up to that
        self._dev_params = None

    @property
    def compute_mode(self):
        """Arithmetic of the GEMM layers of the inference build: 'bf16x3' (default) or 'fp16'."""
        return self._compute_mode

    @compute_mode.setter
    def compute_mode(self, mode):
        if mode not in _MODES:
            raise ValueError("attn_model_struct.compute_mode must be one of %s, not %r" % (list(_MODES), mode))
        self._compute_mode = mode

    def __getitem__(self, name):
        return getattr(self, name)

    def __contains__(self, name):
        return hasattr(self, name)

    def __del__(self):
        try:
            if self._plan is not None:
                _lib.load().attn_plan_destroy(self._plan)
        except Exception:
            pass

    # -- parameters --------------------------------------------------------------------------
    def load_params(self, flat):
        """Inject variables from a flat {reference variable name: array} dict, e.g. 'aconv_1/aconv_1_filters',
        'afc_out/afc_out_biases', 'batch_normalization_5/moving_mean'."""
        dd = {}
        for name, _ in init.ATTN_CONV:
            dd[name] = [flat["%s/%s_filters" % (name, name)], flat["%s/%s_biases" % (name, name)]]
        for name in ("afc_1", "afc_out"):
            dd[name] = [flat["%s/%s_weights" % (name, name)], flat["%s/%s_biases" % (name, name)]]
        for s in init.ATTN_BN_SCOPES:
            dd[s] = [flat["%s/%s" % (s, f)] for f in _BN_FIELDS]
        self.data_dict = dd
        self._dev_params = None

    def load_checkpoint(self, prefix, scope="cnn"):
        """Variables of a `tf.train.Saver` checkpoint (see monkey_pose_b200.model.load_checkpoint)."""
        from . import tf_checkpoint
        import os
        if os.path.isdir(prefix):
            prefix = tf_checkpoint.latest_checkpoint(prefix) or prefix
        lead = scope + "/" if scope else ""
        names = [n for n, _, _ in tf_checkpoint.list_variables(prefix)
                 if n.startswith(lead) and not n.rsplit("/", 1)[-1].startswith("Adam")]
        flat = {n[len(lead):]: v for n, v in tf_checkpoint.read_checkpoint(prefix, names=names).items()}
        self.load_params(flat)
        return sorted(flat)

    def _materialise(self, output_shape):
        fresh = init.attn_params(self.widths, self.fc_hidden, output_shape, self.seed)
        P = {}
        for name, _ in init.ATTN_CONV:
            P[name + "_filters"] = self.get_var(fresh["%s/%s_filters" % (name, name)], name, 0, name + "_filters")
            P[name + "_biases"] = self.get_var(fresh["%s/%s_biases" % (name, name)], name, 1, name + "_biases")
        for name in ("afc_1", "afc_out"):
            P[name + "_weights"] = self.get_var(fresh["%s/%s_weights" % (name, name)], name, 0, name + "_weights")
            P[name + "_biases"] = self.get_var(fresh["%s/%s_biases" % (name, name)], name, 1, name + "_biases")
        for s in init.ATTN_BN_SCOPES:
            for i, f in enumerate(_BN_FIELDS):
                P["%s/%s" % (s, f)] = self.get_var(fresh["%s/%s" % (s, f)], s, i, f)
        # the widths actually in use come from the variables (get_conv_var ignores its channel arguments when the
        # name is in data_dict, :571-581)
        widths = tuple(int(P[n + "_filters"].shape[3]) for n, _ in init.ATTN_CONV)
        return P, widths, int(P["afc_1_weights"].shape[1])

    # -- forward -----------------------------------------------------------------------------
    def build(self, depth, output_shape, batch_norm=None, train_mode=None):
        """:440-525.  depth [N,H,W,1] / [N,H,W] torch CUDA float32 (already divided by image_max_depth, as every
        caller does, e.g. train_cnn_networks.py:115-116); sets and returns `out_put` [N, output_shape]."""
        if not (torch.is_tensor(depth) and depth.is_cuda):
            raise RuntimeError("attn_model_struct.build needs a torch CUDA tensor (there is no CPU fallback)")
        if depth.dim() == 4:
            if depth.shape[3] != 1:
                raise ValueError("depth must have one channel")
            depth = depth[..., 0]
        if depth.dim() != 3:
            raise ValueError("depth must be [N,H,W,1] or [N,H,W]")
        depth = depth.to(torch.float32).contiguous()
        N, H, W = [int(v) for v in depth.shape]
        if train_mode:
            return self._build_layerwise(depth, int(output_shape), train_mode)
        for nme in ("pool1", "pool2", "pool3", "pool4", "pool5", "fc1", "relu1", "conv1", "conv2", "conv3", "conv4",
                    "conv5"):
            self.__dict__.pop(nme, None)           # tensors of an earlier training-mode build
        lib = _lib.load()
        if self._dev_params is None:
            self._dev_params = self._materialise(int(output_shape))
        P, widths, F = self._dev_params
        # a plan runs any batch up to its capacity (attn_forward_batch); a larger batch re-creates it at that size
        key = (H, W, widths, F, int(output_shape), self.compute_mode, depth.device.index)
        if self._plan_key != key or N > self._plan_capacity:
            if self._plan is not None:
                lib.attn_plan_destroy(self._plan)
                self._plan = None
            plan = ctypes.c_void_p()
            wa = (ctypes.c_int * 5)(*widths)
            if self.compute_mode == 'bf16x3':       # attn_plan_create's plan, the entry point callers count on
                _lib.check(lib.attn_plan_create(N, H, W, wa, F, int(output_shape), ctypes.byref(plan)),
                           "attn_plan_create")
            else:
                _lib.check(lib.attn_plan_create_mode(N, H, W, wa, F, int(output_shape),
                                                     _lib.MODES[self.compute_mode], ctypes.byref(plan)),
                           "attn_plan_create_mode")
            self._plan, self._plan_key, self._plan_capacity = plan, key, N
            q = _lib.AttnParams()
            for i, (name, _) in enumerate(init.ATTN_CONV):
                q.conv_filters[i] = P[name + "_filters"].data_ptr()
                q.conv_biases[i] = P[name + "_biases"].data_ptr()
            q.fc_1_weights, q.fc_1_biases = P["afc_1_weights"].data_ptr(), P["afc_1_biases"].data_ptr()
            q.fc_out_weights, q.fc_out_biases = P["afc_out_weights"].data_ptr(), P["afc_out_biases"].data_ptr()
            for i, s in enumerate(init.ATTN_BN_SCOPES):
                for j, f in enumerate(_BN_FIELDS):
                    q.bn[i][j] = P["%s/%s" % (s, f)].data_ptr()
            _lib.check(lib.attn_set_params(plan, ctypes.byref(q), float(self._BATCH_NORM_EPSILON), _stream()),
                       "attn_set_params")
        out = torch.empty((N, int(output_shape)), device=depth.device, dtype=torch.float32)
        _lib.check(lib.attn_forward_batch(self._plan, N, depth.data_ptr(), out.data_ptr(), _stream()),
                   "attn_forward_batch")
        self.gpu_launches = int(lib.attn_plan_launch_count(self._plan))
        self._shapes = {"resized": (N, 128, 128, 1), "fc1": (N, F)}
        for i, c in enumerate(widths):
            self._shapes["pool%d" % (i + 1)] = (N, 64 >> i, 64 >> i, c)
        self.fcout = out
        self.out_put = out
        return out

    def _build_layerwise(self, depth, output_shape, train_mode):
        """:440-525 statement by statement on the layer methods (batch norm over the last axis of the fc tensor, R-D5)."""
        self.updated_moving_stats = {}
        complete = self.data_dict is not None and all(
            n in self.data_dict for n in [c for c, _ in init.ATTN_CONV] + ["afc_1", "afc_out"] + list(init.ATTN_BN_SCOPES))
        if not complete:
            self._defaults = init.attn_params(self.widths, self.fc_hidden, output_shape, self.seed)
        else:
            self._defaults = None
        x = self.resize_images(depth, [128, 128])                                                   # :442
        cin = 1
        for i, ((name, fs), co) in enumerate(zip(init.ATTN_CONV, self.widths)):
            if self.data_dict is not None and name in self.data_dict:
                co = int(np.asarray(self.data_dict[name][0]).shape[3])
            conv = self.conv_layer(x, cin, co, name, filter_size=fs)                                 # :443 ...
            setattr(self, "conv%d" % (i + 1), conv)
            x = self.batch_normalization(self.max_pool(conv, "apool_%d" % (i + 1)), i, train_mode)   # :444-454 ...
            setattr(self, "pool%d" % (i + 1), x)
            cin = co
        in_size = int(np.prod([int(v) for v in x.shape[1:]]))
        fch = self.fc_hidden
        if self.data_dict is not None and "afc_1" in self.data_dict:
            fch = int(np.asarray(self.data_dict["afc_1"][0]).shape[1])
        self.fc1 = self.fc_layer(x, in_size, fch, "afc_1")                                           # :501
        self.relu1 = self.batch_normalization(self.fc1, 5, train_mode, relu_first=True,              # :502-513
                                              dropout_keep=0.7 if train_mode is True else 1.0)
        self.fcout = self.fc_layer(self.relu1, fch, output_shape, "afc_out")                         # :524
        self.out_put = self.fcout
        self.gpu_launches = 1 + 5 * 4 + 2 + 2
        return self.out_put

    def activation(self, name):
        """Intermediate tensors of the last build(): 'resized', 'pool1'..'pool5' (after batch-norm, :444-499),
        'fc1' (:501, before relu)."""
        if self._plan is None or name not in self._shapes:
            raise KeyError(name)
        dst = torch.empty(self._shapes[name], device=self.out_put.device, dtype=torch.float32)
        _lib.check(_lib.load().attn_get_activation(self._plan, name.encode(), dst.data_ptr(), _stream()),
                   "attn_get_activation")
        return dst

    def __getattr__(self, name):
        # pool1..pool5 / fc1 are materialised on demand (a TF graph only computes what is fetched)
        if name in ("pool1", "pool2", "pool3", "pool4", "pool5", "fc1") and self.__dict__.get("_plan") is not None:
            return self.activation(name)
        raise AttributeError(name)
