"""B200-native drop-in for the reference's `hgru_pose.model` (hgru_pose.py:6-216).

`model(trainable=True)`, `.build(depth, output_shape, batch_norm=None, train_mode=None)` and the
attributes it sets (`conv1, pool1, conv2, conv3, hgru, fc1, relu1, fc4, out_put`), the
`data_dict[name][idx]` weight injection and the `var_dict[(name, idx)]` registry are the
reference's.  `depth` is a torch tensor [N,128,128,1] float32: a CUDA tensor runs device to device,
a (pinned) CPU tensor goes through the host entry point (H2D copy, forward, D2H copy) and
`out_put` comes back on the host.

The reference graph cannot run as committed (SURVEY.md section 8c, defects D4-D6); this module
implements the documented resolutions: hgru = build()[0] (R-D4), batch-norm over the last axis of
the fc tensor (R-D5), fc_out consumes relu1 (R-D6).

Two execution paths behind `build()`:
  * train_mode in (None, False): the fused tensor-core pipeline (`pose_forward`), inference-mode batch norm
    (moving statistics) -- the hot path, the benchmark and the parity mode, the one that shards over GPUs;
  * train_mode=True (what the reference's only live caller passes, train_cnn_networks_hgru.py:142): the graph
    composed layer by layer from the model's own layer methods the way the reference composes it
    (`conv_layer`, `max_pool`, `hgru_layer`, `fc_layer`, tf.layers.batch_normalization(training=True) with
    batch statistics, dropout keep 0.7) -- forward only, single GPU (batch statistics couple the batch).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import initialization as init
from .hgru_module import _as_dev, _stream
from .layers import LayerOps

BN_SCOPES = init.BN_SCOPES
_BN_FIELDS = ("gamma", "beta", "moving_mean", "moving_variance")


class _Lazy(object):
    """Intermediate activation fetched from the plan on first access."""

    def __init__(self, owner, name, shape):
        self.owner, self.name, self.shape = owner, name, shape

    def get(self):
        out = torch.empty(self.shape, device='cuda', dtype=torch.float32)
        _lib.check(_lib.load().pose_get_activation(self.owner._plan, self.name.encode(), out.data_ptr(),
                                                   _stream()), "pose_get_activation")
        return out


_LAZY_NAMES = ("conv1", "pool1", "conv2", "conv3", "hgru", "fc1", "relu1")


class model(LayerOps):
    _bn_scopes = BN_SCOPES

    def __init__(self, trainable=True):
        self.trainable = trainable
        self.data_dict = None
        self.var_dict = {}
        self.SRF = 1
        self.SSN = 15
        self.SSF = 15
        self.strides = [1, 1, 1, 1]
        self._BATCH_NORM_DECAY = 0.997
        self._BATCH_NORM_EPSILON = 1e-5
        self.padding = 'SAME'
        self.timesteps = 8
        self.aux = {
            'recurrent_nl': 'tanh',
            'rectify_weights': None,
            'pre_batchnorm': False,
            'gate_filter': 1,
            'xi': False,
            'post_batchnorm': False,
            'dense_connections': False,
            'symmetric_weights': True,
            'symmetric_gate_weights': False,
            'batch_norm': False,
            'atrous_convolutions': False,
            'output_gru_gates': False,
            'association_field': True,
            'multiplicative_excitation': True,
            'gru_gates': True,
            'gamma': True,
            'adapation': True,
            'trainable': True,
        }
        # ---- non-reference knobs (defaults reproduce the reference's shapes) ----
        self.channels = 64            # stem width = hGRU hidden channels k (hgru_pose.py:50,61,71)
        self.fc_hidden = 1024         # hgru_pose.py:91
        self.compute_mode = 'bf16'    # 'fp32' (SIMT, <=1e-4) | 'bf16' (tcgen05, <=1e-2) | 'fp16' (tcgen05 fp16
        #                               operands, bf16 speed, <=2.5e-3, 15x15 kernels) | 'bf16x3' (tcgen05 hi/lo
        #                               splits, <=1e-4, 15x15 kernels); see ContextualCircuit
        self.hidden_state = None      # O_0 [N,64,64,k]; None -> seeded xavier-uniform draw
        self.seed = 42
        self.dropout_seed = 1234      # train_mode=True: seed of the counter-based dropout mask
        self._plan = None
        self._plan_key = None
        self._plan_capacity = 0       # frames the plan was created for: it runs every batch up to that size
        self._dev_params = None
        self._h0_cache = None         # (key, device tensor) of the seeded O_0 draw, at the plan's capacity
        self._lazy = {}

    def __getattr__(self, name):
        """The tensors the reference's build() leaves as attributes (hgru_pose.py:50-105: conv1, pool1, conv2,
        conv3, hgru, fc1, relu1 -- batch-normalised where the reference re-assigns them).  The fused pipeline keeps
        only what later kernels read, so these are materialised on first access after a build()."""
        if name in _LAZY_NAMES:
            lazy = self.__dict__.get("_lazy") or {}
            if name in lazy:
                val = lazy[name].get() if hasattr(lazy[name], "get") else lazy[name]()
                self.__dict__[name] = val
                return val
        raise AttributeError(name)

    def __getitem__(self, name):
        return getattr(self, name)

    def __contains__(self, name):
        return hasattr(self, name)

    # -- parameters --------------------------------------------------------------------------
    def load_params(self, flat):
        """Inject variables from a flat {reference variable name: array} dict, e.g.
        'conv_1/conv_1_filters', 'batch_normalization_3/moving_mean', 'contextual_circuit/p_r'."""
        dd = {}
        for name in ("conv_1", "conv_2", "conv_3"):
            dd[name] = [flat["%s/%s_filters" % (name, name)], flat["%s/%s_biases" % (name, name)]]
        for name in ("fc_1", "fc_out"):
            dd[name] = [flat["%s/%s_weights" % (name, name)], flat["%s/%s_biases" % (name, name)]]
        for s in BN_SCOPES:
            dd[s] = [flat["%s/%s" % (s, f)] for f in _BN_FIELDS]
        dd["contextual_circuit"] = {n: flat["contextual_circuit/" + n] for n in _lib.HGRU_PARAM_ORDER}
        self.data_dict = dd
        self._dev_params = None

    def load_checkpoint(self, prefix, scope="cnn", bn_offset=None):
        """Inject the variables of a TensorFlow V2 checkpoint written by the reference's
        `tf.train.Saver` (train_cnn_networks_hgru.py:188, 248-250; restored at :312-313).  `prefix` is what
        `tf.train.latest_checkpoint(config.model_output)` returns; a directory is resolved the same way.
        The reference builds the model under `tf.variable_scope("cnn")` (:96), so names carry that
        prefix; optimizer slots (`.../Adam`, `beta1_power`, ...) and `global_step` are ignored.
        Read without TensorFlow by `monkey_pose_b200.tf_checkpoint`."""
        from . import tf_checkpoint
        import os
        if os.path.isdir(prefix):
            found = tf_checkpoint.latest_checkpoint(prefix)
            if found is None:
                raise FileNotFoundError("no `checkpoint` state file in %s" % prefix)
            prefix = found
        lead = scope + "/" if scope else ""
        wanted = {}
        for name, _, _ in tf_checkpoint.list_variables(prefix):
            if not name.startswith(lead):
                continue
            short = name[len(lead):]
            tail = short.rsplit("/", 1)[-1]
            if tail.startswith("Adam") or tail in ("beta1_power", "beta2_power", "global_step"):
                continue
            wanted[name] = short
        flat = {wanted[n]: v for n, v in tf_checkpoint.read_checkpoint(prefix, names=list(wanted)).items()}
        # The reference builds the attention CNN first in the same variable scope (:115-117), so its six
        # tf.layers.batch_normalization calls take the names batch_normalization .. _5 and this model's five
        # layers are batch_normalization_6 .. _10 in such checkpoints.
        if bn_offset is None:
            bn_offset = 6 if any(n.startswith("aconv_1/") for n in flat) else 0
        if bn_offset:
            for i, s in enumerate(BN_SCOPES):
                src = "batch_normalization_%d" % (i + bn_offset)
                for f in _BN_FIELDS:
                    flat["%s/%s" % (s, f)] = flat["%s/%s" % (src, f)]
        try:
            self.load_params(flat)
        except KeyError as e:
            raise KeyError("checkpoint %s lacks variable %s (scope %r)" % (prefix, e, scope))
        return sorted(flat)

    def _materialise(self, in_ch, hw, output_shape):
        """Create every variable of the graph (hgru_pose.py:165-194 + hgru_module.py:262-503)."""
        k, T, S = self.channels, self.timesteps, 2 * (self.SSF // 2) + 1
        fresh = self.__dict__.get("_defaults")      # None when data_dict supplies every variable

        def default(key):
            return fresh[key] if fresh is not None else None

        P = {}
        for name in ("conv_1", "conv_2", "conv_3"):
            P[name + "_filters"] = self.get_var(default("%s/%s_filters" % (name, name)), name, 0, name + "_filters")
            P[name + "_biases"] = self.get_var(default("%s/%s_biases" % (name, name)), name, 1, name + "_biases")
        for name in ("fc_1", "fc_out"):
            P[name + "_weights"] = self.get_var(default("%s/%s_weights" % (name, name)), name, 0, name + "_weights")
            P[name + "_biases"] = self.get_var(default("%s/%s_biases" % (name, name)), name, 1, name + "_biases")
        P["bn"] = []
        for s in BN_SCOPES:
            P["bn"].append([self.get_var(default("%s/%s" % (s, f)), s, i, f) for i, f in enumerate(_BN_FIELDS)])
        cc = self.data_dict.get("contextual_circuit") if self.data_dict else None
        P["hgru"] = {}
        for n in _lib.HGRU_PARAM_ORDER:
            v = cc[n] if cc is not None else fresh["contextual_circuit/" + n]
            P["hgru"][n] = _as_dev(v)
            self.var_dict[("contextual_circuit", n)] = P["hgru"][n]
        # shape checks (TF would raise at graph construction)
        exp = {"conv_1_filters": (3, 3, in_ch, k), "conv_2_filters": (3, 3, k, k), "conv_3_filters": (3, 3, k, k),
               "fc_1_weights": (hw * hw * k, self.fc_hidden), "fc_out_weights": (self.fc_hidden, output_shape)}
        for n, shp in exp.items():
            if tuple(P[n].shape) != shp:
                raise ValueError("%s has shape %s, expected %s" % (n, tuple(P[n].shape), shp))
        return P

    # -- layer methods: conv_layer / max_pool / fc_layer / get_*_var / batch_normalization come from LayerOps
    def hgru_layer(self, bottom):
        """hgru_pose.py:107-118: ContextualCircuit(X=bottom, timesteps, SRF, SSN, SSF, strides, padding, aux).build().
        As in the reference this is what build() of the circuit returns -- the tuple (O, weights, activities) under
        the default return_weights=True (reference defect D4; callers take element 0)."""
        from .hgru_module import ContextualCircuit
        x = self._need_cuda(bottom, "hgru_layer")
        cc = self.data_dict.get("contextual_circuit") if self.data_dict else None
        d = self.__dict__.get("_defaults")
        if cc is None and d is not None and "contextual_circuit/p_r" in d:
            cc = {n: d["contextual_circuit/" + n] for n in _lib.HGRU_PARAM_ORDER}
        layer = ContextualCircuit(X=x, timesteps=self.timesteps, SRF=self.SRF, SSN=self.SSN, SSF=self.SSF,
                                  strides=self.strides, padding=self.padding, aux=self.aux, params=cc,
                                  hidden_state=self.hidden_state, compute_mode=self.compute_mode, seed=self.seed)
        return layer.build()

    # -- forward -----------------------------------------------------------------------------
    def _build_layerwise(self, depth, output_shape, train_mode):
        """hgru_pose.py:47-105 statement by statement on the layer methods (R-D4, R-D5, R-D6 applied)."""
        C = self.channels
        self.updated_moving_stats = {}
        x = self._need_cuda(depth, "build(train_mode=True)")
        self.conv1 = self.conv_layer(x, int(x.shape[-1]), C, "conv_1", filter_size=3)                # :50
        self.pool1 = self.max_pool(self.conv1, 'pool_1')                                             # :51
        self.pool1 = self.batch_normalization(self.pool1, 0, train_mode)                             # :52-60
        self.conv2 = self.conv_layer(self.pool1, C, C, "conv_2", filter_size=3)                      # :61
        self.conv2 = self.batch_normalization(self.conv2, 1, train_mode)                             # :62-70
        self.conv3 = self.conv_layer(self.conv2, C, C, "conv_3", filter_size=3)                      # :71
        self.conv3 = self.batch_normalization(self.conv3, 2, train_mode)                             # :72-80
        hg = self.hgru_layer(self.conv3)                                                             # :81
        self.hgru = hg[0] if isinstance(hg, tuple) else hg                                           # R-D4
        self.hgru = self.batch_normalization(self.hgru, 3, train_mode)                               # :82-90
        in_size = int(np.prod([int(v) for v in self.hgru.shape[1:]]))
        self.fc1 = self.fc_layer(self.hgru, in_size, self.fc_hidden, "fc_1")                         # :91
        # relu (:92), dropout keep 0.7 when train_mode == True (:93-94), batch norm over the last axis (:95-103, R-D5)
        self.relu1 = self.batch_normalization(self.fc1, 4, train_mode, relu_first=True,
                                              dropout_keep=0.7 if train_mode is True else 1.0)
        self.fc4 = self.fc_layer(self.relu1, self.fc_hidden, int(output_shape), "fc_out")            # :104 (R-D6)
        self.out_put = self.fc4                                                                      # :105
        self.gpu_launches = 6 + 2 * 5 + 2 + 22      # (not counted by a plan: layer kernels + the circuit's own)
        self._lazy = {}
        return self.out_put

    def build(self, depth, output_shape, batch_norm=None, train_mode=None):
        """hgru_pose.py:47-105.  `batch_norm` is accepted and ignored exactly as in the reference."""
        if not torch.is_tensor(depth):
            depth = torch.as_tensor(np.asarray(depth, dtype=np.float32))
        if depth.dim() != 4 or depth.shape[-1] != 1 or depth.shape[1] != depth.shape[2] or depth.shape[1] % 2:
            raise ValueError("depth must be [N, 2*HW, 2*HW, 1]")
        depth = depth.to(torch.float32).contiguous()
        for n in _LAZY_NAMES:
            self.__dict__.pop(n, None)
        if train_mode:
            self._need_cuda(depth, "build(train_mode=True)")
        N, hw = int(depth.shape[0]), int(depth.shape[1]) // 2
        S = 2 * (self.SSF // 2) + 1
        complete = self.data_dict is not None and all(
            n in self.data_dict for n in ("conv_1", "conv_2", "conv_3", "fc_1", "fc_out", "contextual_circuit") + BN_SCOPES)
        dkey = (self.channels, S, self.timesteps, hw, self.fc_hidden, int(output_shape), self.seed)
        if complete:
            self._defaults, self._defaults_key = None, None
        elif self.__dict__.get("_defaults_key") != dkey:
            # one seeded draw of the whole graph's variables, shared by the fused and the layer-wise path
            self._defaults = init.pose_params(channels=self.channels, S=S, T=self.timesteps, hw=hw,
                                              fc_hidden=self.fc_hidden, out=int(output_shape), seed=self.seed)
            self._defaults_key = dkey
        if train_mode:
            return self._build_layerwise(depth, output_shape, train_mode)
        lib = _lib.load()
        mode = _lib.MODES[self.compute_mode]
        # The plan key leaves out the batch: a plan runs any batch up to its capacity (pose_forward_batch) with no
        # re-allocation and no re-packing of the weights.  A larger batch re-creates it at that size; capacity never
        # shrinks.
        key = (torch.cuda.current_device(), hw, self.channels, S, self.timesteps, self.fc_hidden, int(output_shape),
               mode)
        if self._plan is None or key != self._plan_key or N > self._plan_capacity:
            if self._plan is not None:
                lib.pose_plan_destroy(self._plan)
            h = ctypes.c_void_p()
            _lib.check(lib.pose_plan_create(N, hw, self.channels, S, self.timesteps, self.fc_hidden,
                                            int(output_shape), mode, ctypes.byref(h)), "pose_plan_create")
            self._plan, self._plan_key, self._plan_capacity, self._dev_params = h, key, N, None
        st = _stream()
        if self._dev_params is None:
            P = self._materialise(int(depth.shape[-1]), hw, int(output_shape))
            q = _lib.PoseParams()
            for f in ("conv_1_filters", "conv_1_biases", "conv_2_filters", "conv_2_biases", "conv_3_filters",
                      "conv_3_biases", "fc_1_weights", "fc_1_biases", "fc_out_weights", "fc_out_biases"):
                setattr(q, f, P[f].data_ptr())
            for i in range(5):
                for j in range(4):
                    q.bn[i][j] = P["bn"][i][j].data_ptr()
            for n in _lib.HGRU_PARAM_ORDER:
                setattr(q, n, P["hgru"][n].data_ptr())
            _lib.check(lib.pose_set_params(self._plan, ctypes.byref(q), float(self._BATCH_NORM_EPSILON), st),
                       "pose_set_params")
            self._dev_params = P
        h0 = None
        if self.hidden_state is not None:
            h0 = _as_dev(self.hidden_state)
            if tuple(h0.shape) != (N, hw, hw, self.channels):
                raise ValueError("hidden_state must be [N,%d,%d,%d]" % (hw, hw, self.channels))
        elif self.aux.get('hidden_init', 'random') == 'random':
            # the seeded O_0 draw is made once per shape at the plan's capacity and kept on the device (268 MB at
            # N = 256, 64 channels).  The generator fills in C order, so its first N frames are the draw of N frames.
            cap = self._plan_capacity
            hkey = (torch.cuda.current_device(), cap, hw, self.channels, self.seed)
            if self._h0_cache is None or self._h0_cache[0] != hkey:
                self._h0_cache = (hkey, _as_dev(init.hidden_init((cap, hw, hw, self.channels), seed=self.seed + 7)))
            h0 = self._h0_cache[1] if N == cap else self._h0_cache[1][:N]
        elif self.aux.get('hidden_init') not in ('zeros', 'identity'):
            raise RuntimeError("hidden_init must be 'random', 'zeros' or 'identity'")      # hgru_module.py:891-892
        # 'identity': O_0 = X = conv3 of this forward (hgru_module.py:876-878), taken inside the library
        identity = self.hidden_state is None and self.aux.get('hidden_init') == 'identity'
        _lib.check(lib.pose_set_hidden_init(self._plan, 1 if identity else 0), "pose_set_hidden_init")
        self._h0 = h0
        h0_ptr = h0.data_ptr() if h0 is not None else None
        if depth.is_cuda:
            out = torch.empty((N, int(output_shape)), device=depth.device, dtype=torch.float32)
            _lib.check(lib.pose_forward_batch(self._plan, N, depth.data_ptr(), h0_ptr, out.data_ptr(), st),
                       "pose_forward_batch")
        else:
            out = torch.empty((N, int(output_shape)), dtype=torch.float32, pin_memory=True)
            _lib.check(lib.pose_forward_host_batch(self._plan, N, depth.data_ptr(), h0_ptr, out.data_ptr(), st),
                       "pose_forward_host_batch")
        self.gpu_launches = lib.pose_plan_launch_count(self._plan)
        act = (N, hw, hw, self.channels)
        self._act = {"pool1": _Lazy(self, "pool1", act), "conv2": _Lazy(self, "conv2", act),
                     "conv3": _Lazy(self, "conv3", act), "hgru": _Lazy(self, "hgru", act),
                     "fc1": _Lazy(self, "fc1", (N, self.fc_hidden))}
        # attribute surface of the reference (hgru_pose.py:50-105), materialised on first access (__getattr__)
        C = self.channels
        dev_depth = depth

        def conv1():
            d = dev_depth if dev_depth.is_cuda else dev_depth.cuda()
            return self.conv_layer(d, int(d.shape[-1]), C, "conv_1", filter_size=3)

        self._lazy = {"conv1": conv1, "pool1": self._act["pool1"], "conv2": self._act["conv2"],
                      "conv3": self._act["conv3"], "fc1": self._act["fc1"],
                      # the reference re-assigns self.hgru / self.relu1 to their batch-normalised tensors (:82, :95)
                      "hgru": lambda: self.batch_normalization(self._act["hgru"].get(), 3, False),
                      "relu1": lambda: self.batch_normalization(self._act["fc1"].get(), 4, False, relu_first=True)}
        self.fc4 = out
        self.out_put = out
        return out

    def activation(self, name):
        """Intermediate tensor of the last build() straight from the plan (`pool1`, `conv2`, `conv3` [post
        batch-norm, as in the reference], `hgru` [PRE batch-norm: the circuit's output], `fc1`)."""
        return self._act[name].get()

    def __del__(self):
        try:
            if self._plan is not None:
                _lib.load().pose_plan_destroy(self._plan)
                self._plan = None
        except Exception:
            pass
