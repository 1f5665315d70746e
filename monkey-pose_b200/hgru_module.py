"""B200-native drop-in for the reference's `hgru_module.ContextualCircuit` (hgru_module.py:54-959).

Same constructor keywords, same `build()` return convention, same variable names; tensors are
torch CUDA tensors (NHWC float32) instead of tf.Tensors and the arithmetic runs in the sm_100a
kernels of libhgru_b200.so.  Only the path hgru_pose.py configures is implemented; every other
option the reference declares is accepted as a key and raises NotImplementedError when selected
(SURVEY.md section 8a, row a19).
"""
import math

import numpy as np
import torch

from . import _lib
from . import initialization as init


def auxilliary_variables():
    """Defaults of the reference's auxilliary_variables() (hgru_module.py:9-51).  TensorFlow
    callables are named by strings here ('tanh', 'sigmoid')."""
    return {
        'lesions': [None],
        'lesion_beta': False,
        'lesion_nu': False,
        'lesion_omega': False,
        'lesion_kappa': False,
        'dtype': 'float32',
        'return_weights': True,
        'hidden_init': 'random',
        'gate_bias_init': 'chronos',
        'association_field': True,
        'tuning_nl': 'tanh',
        'store_states': False,
        'train': True,
        'dropout': None,
        'recurrent_nl': 'tanh',
        'gate_nl': 'sigmoid',
        'ecrf_nl': 'tanh',
        'normal_initializer': True,
        'symmetric_weights': True,
        'symmetric_gate_weights': False,
        'gru_gates': False,
        'output_gru_gates': False,
        'post_tuning_nl': 'tanh',
        'gate_filter': 1,
        'zeta': False,
        'gamma': True,
        'xi': False,
        'beta': True,
        'nu': True,
        'batch_norm': False,
        'adapation': False,
        'integration_type': 'alternate',
        'dense_connections': False,
        'atrous_convolutions': False,
        'multiplicative_excitation': True,
        'rectify_weights': None,
    }


# Plans own their workspace (gigabytes at batch 256), so only the most recently used few shapes stay alive.  A plan
# serves every batch up to its capacity (hgru_forward_batch), so the batch size is not part of the key.
_PLAN_CACHE = {}          # key -> (plan handle, capacity), in least-recently-used order (dicts keep insertion order)
PLAN_CACHE_SIZE = 4


def clear_plan_cache():
    """Destroy every cached layer plan and free its device workspace."""
    lib = _lib.load()
    torch.cuda.synchronize()
    for plan, _ in _PLAN_CACHE.values():
        lib.hgru_plan_destroy(plan)
    _PLAN_CACHE.clear()


def _get_plan(N, H, W, k, S, T, mode):
    """A plan of this shape that runs N frames: the cached one when its capacity is at least N, else a new plan for
    N frames, which replaces a smaller cached one."""
    key = (torch.cuda.current_device(), H, W, k, S, T, mode)
    entry = _PLAN_CACHE.pop(key, None)
    lib = _lib.load()
    if entry is not None and entry[1] < N:
        torch.cuda.synchronize()                            # (its last forward may still be running)
        lib.hgru_plan_destroy(entry[0])
        entry = None
    if entry is None:
        import ctypes
        while len(_PLAN_CACHE) >= PLAN_CACHE_SIZE:          # evict the least recently used plan
            old = next(iter(_PLAN_CACHE))
            torch.cuda.synchronize()                        # (its last forward may still be running)
            lib.hgru_plan_destroy(_PLAN_CACHE.pop(old)[0])
        h = ctypes.c_void_p()
        _lib.check(lib.hgru_plan_create(N, H, W, k, S, T, mode, ctypes.byref(h)), "hgru_plan_create")
        entry = (h, N)
    _PLAN_CACHE[key] = entry          # (re)insert as most recently used
    return entry[0]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _as_dev(x, shape=None):
    t = torch.as_tensor(x, dtype=torch.float32)
    if not t.is_cuda:
        t = t.cuda()
    t = t.contiguous()
    if shape is not None:
        t = t.reshape(shape)
    return t


class ContextualCircuit(object):
    def __getitem__(self, name):
        return getattr(self, name)

    def __contains__(self, name):
        return hasattr(self, name)

    def __init__(
            self,
            X,
            timesteps=1,
            SRF=1,
            SSN=9,
            SSF=29,
            strides=[1, 1, 1, 1],
            padding='SAME',
            aux=None,
            train=True,
            params=None,
            hidden_state=None,
            compute_mode='bf16',
            seed=42):
        """Global initializations and settings (hgru_module.py:61-128).

        X: torch CUDA tensor [n,h,w,k] float32 (static batch, hgru_module.py:74).
        Non-reference keywords: `params` (dict of the `contextual_circuit/*` variables, by their
        reference names), `hidden_state` (O_0, [n,h,w,k]), `compute_mode`, `seed`.
        compute_mode (arithmetic of the 15x15 and 1x1 convolutions; state and integration math are fp32 in all):
          'fp32'   SIMT, exact fp32;
          'bf16'   tcgen05 tensor cores, bf16 operands (8 significand bits), fp32 accumulation;
          'fp16'   the 'bf16' mode with fp16 operands (11 significand bits) at the same speed; S = 15, k <= 64 (else
                   NotImplementedError); operands saturate at +-65504, so an initial state beyond that is clamped in
                   the first timestep's gated operand;
          'bf16x3' tcgen05 on bf16 hi/lo splits (three products), fp32-class accuracy; S = 15.
        """
        if not (torch.is_tensor(X) and X.dim() == 4):
            raise ValueError("X must be a 4-D torch tensor [n,h,w,k] (CUDA for build())")
        self.X = X.to(torch.float32).contiguous()
        self.n, self.h, self.w, self.k = [int(x) for x in X.shape]
        self.timesteps = timesteps
        self.strides = strides
        self.padding = padding
        self.train = train

        aux_vars = auxilliary_variables()
        if aux is not None and isinstance(aux, dict):
            for k, v in aux.items():
                aux_vars[k] = v
        self.update_params(aux_vars)

        self.SRF, self.SSN, self.SSF = SRF, SSN, SSF
        if isinstance(SSF, list):
            raise NotImplementedError('hierarchical_convolutions (list-valued SSF) are not on the hot path')
        self.SSF_ext = 2 * int(math.floor(SSF / 2.0)) + 1            # hgru_module.py:94-97
        if self.SSN is None:
            self.SSN = self.SRF * 3
        if self.SSF is None:
            self.SSF = self.SRF * 5

        self.q_shape = [self.SRF, self.SRF, self.k, self.k]
        self.u_shape = [self.SRF, self.SRF, self.k, 1]
        self.p_shape = [self.SSF_ext, self.SSF_ext, self.k, self.k]
        self.i_shape = [self.gate_filter, self.gate_filter, self.k, self.k]
        self.o_shape = [self.gate_filter, self.gate_filter, self.k, self.k]
        self.bias_shape = [1, 1, 1, self.k]
        self.tuning_params = ['Q', 'P']
        self.tuning_shape = [1, 1, self.k, self.k]

        if isinstance(self.recurrent_nl, str):
            self.recurrent_nl = self.interpret_nl(self.recurrent_nl)
        self.ii, self.oi = self.interpret_integration(self.integration_type)

        if compute_mode not in _lib.MODES:
            raise ValueError("compute_mode must be one of %s" % sorted(_lib.MODES))
        self.compute_mode = compute_mode
        self._injected = params
        self._hidden_state = hidden_state
        self._seed = seed
        self._check_supported()

    # -- option handling ---------------------------------------------------------------------
    def interpret_nl(self, nl_type):
        """hgru_module.py:130-143 -- only tanh runs in the kernels."""
        if nl_type == 'tanh':
            return 'tanh'
        elif nl_type in ('relu', 'selu', 'leaky_relu', 'hard_tanh'):
            raise NotImplementedError('recurrent_nl=%s: only tanh is on the hot path' % nl_type)
        else:
            raise NotImplementedError(nl_type)

    def interpret_integration(self, integration_type):
        """hgru_module.py:145-157."""
        if integration_type == 'alternate':
            return 'input_integration', 'output_integration'
        elif integration_type in ('mely', 'control'):
            raise NotImplementedError(
                'Requested integration %s is declared by the reference but not on the hot path'
                % integration_type)
        else:
            raise NotImplementedError('Requested integration %s' % integration_type)

    def update_params(self, kwargs):
        if kwargs is not None:
            for k, v in kwargs.items():
                setattr(self, k, v)

    def _check_supported(self):
        def need(cond, what):
            if not cond:
                raise NotImplementedError(what + ' (not on the path hgru_pose.py configures)')
        need(list(self.strides) == [1, 1, 1, 1], 'strides != [1,1,1,1]')
        need(self.padding == 'SAME', "padding != 'SAME'")
        need(self.gate_filter == 1, 'gate_filter != 1')
        need(self.gru_gates is True, 'gru_gates=False')
        need(not self.output_gru_gates, 'output_gru_gates=True')
        need(self.multiplicative_excitation is True, 'multiplicative_excitation=False')
        need(self.association_field is True, 'association_field=False')
        need(self.rectify_weights is None, 'rectify_weights')
        need(not self.atrous_convolutions, 'atrous_convolutions')
        need(not self.batch_norm, 'batch_norm inside the circuit')
        need(self.gamma is True or torch.is_tensor(self.gamma), 'gamma=False')
        need(self.beta is True or torch.is_tensor(self.beta), 'beta=False')
        need(self.nu is True or torch.is_tensor(self.nu), 'nu=False')
        need(not self.zeta or torch.is_tensor(self.zeta), 'zeta=True')
        need(not self.xi or torch.is_tensor(self.xi), 'xi=True')
        need(self.lesions in ([None], None, []), 'lesions')
        need(not (self.lesion_beta or self.lesion_nu or self.lesion_omega or self.lesion_kappa), 'lesion_*')
        need(not self.store_states, 'store_states (use build(trace=True))')
        need(self.gate_nl in ('sigmoid',), 'gate_nl != sigmoid')
        if self.train and self.dropout is not None:
            raise NotImplementedError                                   # hgru_module.py:702-703
        need(self.dtype in ('float32', torch.float32), 'dtype != float32')

    # -- parameters --------------------------------------------------------------------------
    def prepare_tensors(self):
        """Variables of scope `contextual_circuit` (hgru_module.py:172-503) as torch CUDA tensors,
        registered as attributes under the reference's names."""
        self.weight_dict = {
            'P': {'r': {'weight': 'p_r', 'activity': 'P_r', 'tuning': 'p_t'}},
            'I': {'r': {'weight': 'i_r', 'bias': 'i_b', 'activity': 'I_r'}},
            'O': {'r': {'weight': 'o_r', 'bias': 'o_b', 'activity': 'O_r'}},
            'xi': {'r': {'weight': 'xi'}}, 'beta': {'r': {'weight': 'beta'}},
            'nu': {'r': {'weight': 'nu'}}, 'zeta': {'r': {'weight': 'zeta'}},
            'gamma': {'r': {'weight': 'gamma'}}, 'phi': {'r': {'weight': 'phi'}},
            'kappa': {'r': {'weight': 'kappa'}}, 'rho': {'r': {'weight': 'rho'}},
        }
        k, S, T = self.k, self.SSF_ext, self.timesteps
        shapes = {'p_r': (S, S, k, k), 'i_r': (1, 1, k, k), 'o_r': (1, 1, k, k), 'rho': (T,)}
        for n in ('i_b', 'o_b', 'beta', 'nu', 'gamma', 'kappa', 'omega', 'lateral_bias'):
            shapes[n] = (1, 1, 1, k)
        # `rho` exists only with adapation=True (hgru_module.py:490-493); without it the state is not rescaled
        # (:847-849) -- the kernels then multiply by a vector of ones that is not a variable of the layer.
        adapt = bool(self.adapation)
        if self._injected is not None:
            src = {}
            for n in _lib.HGRU_PARAM_ORDER:
                if n == 'rho' and not adapt:
                    continue
                v = self._injected.get(n, self._injected.get('contextual_circuit/' + n))
                if v is None:
                    raise KeyError('params is missing %r' % n)
                src[n] = v
        else:
            if self.gate_bias_init != 'chronos':
                raise NotImplementedError("gate_bias_init != 'chronos'")
            src = init.hgru_params(k, S, T, seed=self._seed)
        self._rho_ones = None
        for n in _lib.HGRU_PARAM_ORDER:
            if n == 'rho' and not adapt:
                self._rho_ones = torch.ones(T, device=self.X.device, dtype=torch.float32)
                if hasattr(self, 'rho'):
                    delattr(self, 'rho')
                continue
            t = _as_dev(src[n])
            if tuple(t.shape) != shapes[n]:
                if t.numel() != int(np.prod(shapes[n])):
                    raise RuntimeError('%s has shape %s, expected %s' % (n, tuple(t.shape), shapes[n]))
                t = t.reshape(shapes[n])
            setattr(self, n, t)
        dev = self.X.device
        self.zeta = torch.ones((), device=dev)          # tf.constant(1.) hgru_module.py:437-438
        self.xi = torch.ones((), device=dev)            # hgru_module.py:463-464

    def gather_tensors(self, wak='weight'):
        weights = {}
        for k, v in self.weight_dict.items():
            for wk, wv in v.items():
                if wak in wv.keys() and hasattr(self, wv[wak]):
                    weights['%s_%s' % (k, wk)] = self[wv[wak]]
        return weights

    # -- the per-timestep methods (hgru_module.py:505-861) -----------------------------------------------------------
    # Stand-alone, exact fp32, unfused: what a caller stepping the circuit by hand gets (call prepare_tensors() first,
    # as the reference's build() does).  build() itself runs the fused tensor-core pipeline, never these.
    def _rows(self, t):
        if not (torch.is_tensor(t) and t.is_cuda and t.dim() == 4 and int(t.shape[3]) == self.k):
            raise RuntimeError("expected a [n,h,w,%d] torch CUDA tensor (no CPU fallback)" % self.k)
        t = t.to(torch.float32).contiguous()
        return t, int(t.shape[0]) * int(t.shape[1]) * int(t.shape[2])

    def _conv2d(self, data, weights, bias):
        """Stride-1 SAME cross-correlation + bias (None: zeros) through the stand-alone exact conv kernel."""
        w_shape = [int(w) for w in weights.shape]
        data = data.to(torch.float32).contiguous()
        weights = _as_dev(weights).contiguous()
        n, h, w = [int(v) for v in data.shape[:3]]
        out = torch.empty((n, h, w, w_shape[3]), device=data.device, dtype=torch.float32)
        if bias is None:
            bias = torch.zeros(w_shape[3], device=data.device, dtype=torch.float32)
        _lib.check(_lib.load().layer_conv2d_forward(
            data.data_ptr(), n, h, w, w_shape[2], weights.data_ptr(), w_shape[0], w_shape[3],
            bias.contiguous().data_ptr(), 0, out.data_ptr(), _stream()), "layer_conv2d_forward")
        return out

    def conv_2d_op(self, data, weight_key, out_key=None, weights=None, symmetric_weights=False, rectify=None):
        """2D convolutions, return or assign activity as attribute (hgru_module.py:505-581).  `symmetric_weights` only
        changes the gradient in the reference (:521-535); the forward is a plain stride-1 SAME cross-correlation."""
        if weights is None:
            weights = self[weight_key]
        if rectify is not None:
            weights = rectify(weights, 0)
        w_shape = [int(w) for w in weights.shape]
        if len(w_shape) > 1 and int(w_shape[-2]) > 1:
            if self.atrous_convolutions:
                raise NotImplementedError('atrous_convolutions (not on the path hgru_pose.py configures)')
            if len(w_shape) != 4 or w_shape[0] != w_shape[1] or w_shape[0] % 2 == 0:
                raise NotImplementedError('conv_2d_op: square odd HWIO filters only')
            if not (torch.is_tensor(data) and data.is_cuda and data.dim() == 4 and int(data.shape[3]) == w_shape[2]):
                raise RuntimeError("data must be a [n,h,w,%d] torch CUDA tensor (no CPU fallback)" % w_shape[2])
            activities = self._conv2d(data, weights, None)
        elif len(w_shape) > 1 and int(w_shape[-2]) == 1:
            raise NotImplementedError('separable spatial convolutions (hgru_module.py:549-570) are not on the hot path')
        else:
            raise RuntimeError                                          # hgru_module.py:571-572
        if out_key is None:
            return activities
        setattr(self, out_key, activities)

    def p_convolution(self, data, key, rectification):
        """Apply the eCRF association field convolution (hgru_module.py:615-624)."""
        p_weights = self[key]
        if self.rectify_weights == True:  # noqa: E712 (the reference's own test)
            p_weights = rectification(p_weights, 0)
        return self.conv_2d_op(data=data, weight_key=key, weights=p_weights, symmetric_weights=self.symmetric_weights)

    def process_p(self, data, key, rectification, full=True):
        """Wrapper for eCRF operations: the association-field convolution + lateral_bias (hgru_module.py:626-658)."""
        if not full:
            raise NotImplementedError('1x1 tuning convolutions (association_field=False) are not on the hot path')
        if isinstance(self.p_shape[0], list):
            raise NotImplementedError('hierarchical_convolutions are not on the hot path')
        if self.rectify_weights == True:  # noqa: E712
            return self.p_convolution(data=data, key=key, rectification=rectification) + self.lateral_bias
        # p_convolution (:615-624) with `+ lateral_bias` (:657) as the convolution kernel's bias: same rounding, one pass
        if not (torch.is_tensor(data) and data.is_cuda and data.dim() == 4 and int(data.shape[3]) == self.k):
            raise RuntimeError("data must be a [n,h,w,%d] torch CUDA tensor (no CPU fallback)" % self.k)
        return self._conv2d(data, self[key], self.lateral_bias.reshape(-1))

    def _gate(self, x, wkey, bkey, gated):
        x, rows = self._rows(x)
        g = torch.empty_like(x)
        xg = torch.empty_like(x) if gated else None
        _lib.check(_lib.load().circuit_gate_forward(
            x.data_ptr(), rows, self.k, self[wkey].data_ptr(), self[bkey].data_ptr(), g.data_ptr(),
            xg.data_ptr() if gated else None, _stream()), "circuit_gate_forward")
        return g, xg

    def circuit_input(self, O):
        """Circuit input operates on recurrent output (O): (P, I_update) (hgru_module.py:692-724).  The gate is
        applied to a copy, as in the reference's graph (the caller's O is unchanged)."""
        if self.train and self.dropout is not None:
            raise NotImplementedError
        I_update, gated = self._gate(O, self.weight_dict['I']['r']['weight'], self.weight_dict['I']['r']['bias'],
                                     bool(self.gru_gates))
        P = self.process_p(data=gated if self.gru_gates else O, key=self.weight_dict['P']['r']['weight'],
                           rectification=None, full=self.association_field)
        if self.rectify_weights == False:  # noqa: E712
            P = torch.clamp(P, max=0)
        return P, I_update

    def circuit_output(self, I):
        """Circuit output operates on recurrent input (I): (P, O_update) (hgru_module.py:726-756)."""
        if self.train and self.dropout is not None:
            raise NotImplementedError
        O_update, gated = self._gate(I, self.weight_dict['O']['r']['weight'], self.weight_dict['O']['r']['bias'],
                                     bool(self.output_gru_gates))
        P = self.process_p(data=gated if self.output_gru_gates else I, key=self.weight_dict['P']['r']['weight'],
                           rectification=None, full=self.association_field)
        if self.rectify_weights == False:  # noqa: E712
            P = torch.clamp(P, min=0)
        return P, O_update

    def input_integration(self, P, I, O, I_update):
        """Integration on the input: tanh(xi X - (beta O + nu) P) (hgru_module.py:795-804)."""
        if not self.gru_gates:
            raise NotImplementedError('gru_gates=False (not on the path hgru_pose.py configures)')
        P, rows = self._rows(P)
        O, _ = self._rows(O)
        out = torch.empty_like(P)
        _lib.check(_lib.load().circuit_input_integration_forward(
            self.X.data_ptr(), O.data_ptr(), P.data_ptr(), self.beta.data_ptr(), self.nu.data_ptr(), float(self.xi),
            rows, self.k, out.data_ptr(), _stream()), "circuit_input_integration_forward")
        return out

    def output_integration(self, P, I, O, O_update, _rho=None):
        """Integration on the output (hgru_module.py:806-823): multiplicative excitation, mixed with the old O by the
        output gate."""
        if not self.multiplicative_excitation or self.output_gru_gates:
            raise NotImplementedError('additive gating / output_gru_gates (not on the path hgru_pose.py configures)')
        P, rows = self._rows(P)
        I, _ = self._rows(I)
        O, _ = self._rows(O)
        G, _ = self._rows(O_update)
        out = torch.empty_like(P)
        _lib.check(_lib.load().circuit_output_integration_forward(
            I.data_ptr(), P.data_ptr(), O.data_ptr(), G.data_ptr(), self.gamma.data_ptr(), self.kappa.data_ptr(),
            self.omega.data_ptr(), float(self.zeta), _rho.data_ptr() if _rho is not None else None, rows, self.k,
            out.data_ptr(), _stream()), "circuit_output_integration_forward")
        return out

    def full(self, i0, O, I, store_O=None, store_I=None):
        """Contextual circuit body: one timestep (hgru_module.py:825-857).  Returns (i0 + 1, O, I, store_I, store_O)."""
        P, I_update = self.circuit_input(O)
        I = getattr(self, self.ii)(P=P, I=I, O=O, I_update=I_update)
        P, O_update = self.circuit_output(I)
        if self.adapation:
            rho_i = self.rho.reshape(-1)[int(i0):int(i0) + 1]          # tf.gather(self.rho, i0): O * rho[i0] (:847-849)
            O = getattr(self, self.oi)(P=P, I=I, O=O, O_update=O_update, _rho=rho_i)
        else:
            O = getattr(self, self.oi)(P=P, I=I, O=O, O_update=O_update)
        if self.store_states:
            raise NotImplementedError('store_states (use build(trace=True))')
        i0 += 1
        return i0, O, I, store_I, store_O

    def condition(self, i0, O, I, store_I, store_O):
        """While loop halting condition (hgru_module.py:859-861)."""
        return i0 < self.timesteps

    # -- declared by the reference, not on the path hgru_pose.py configures (SURVEY.md 8 a19): same names, and the
    #    reference's own error type for an unimplemented option
    def _off_path(self, what, lines):
        raise NotImplementedError('%s (hgru_module.py:%s) is declared by the reference but not on the path '
                                  'hgru_pose.py configures' % (what, lines))

    def symmetric_weights(self, w, name):
        """hgru_module.py:165-170 (shadowed in the reference by the boolean option of the same name, :163)."""
        self._off_path('symmetric_weights()', '165-170')

    def apply_tuning(self, data, wm, nl=False, rectify=None):
        self._off_path('apply_tuning', '583-603')

    def zoneout(self, dropout):
        self._off_path('zoneout', '605-613')

    def hierarchical_convolutions(self, data, key, rectification):
        self._off_path('hierarchical_convolutions', '660-690')

    def mely_input_integration(self, P, I, O, I_update):
        self._off_path('mely_input_integration', '758-767')

    def mely_output_integration(self, P, I, O, O_update):
        self._off_path('mely_output_integration', '769-773')

    def input_integration_control(self, P, I, O, I_update):
        self._off_path('input_integration_control', '775-780')

    def output_integration_control(self, P, I, O, O_update):
        self._off_path('output_integration_control', '782-793')

    # -- forward -----------------------------------------------------------------------------
    def _initial_state(self):
        if self._hidden_state is not None:
            O = _as_dev(self._hidden_state)
            if tuple(O.shape) != tuple(self.X.shape):
                raise RuntimeError('hidden_state shape %s != X shape %s' % (tuple(O.shape), tuple(self.X.shape)))
            return O
        if self.hidden_init == 'identity':
            return self.X.clone()
        elif self.hidden_init == 'random':
            # xavier-uniform over the activation shape (hgru_module.py:879-887), seeded
            g = torch.Generator(device='cpu').manual_seed(self._seed + 1)
            rf = self.n * self.h
            lim = math.sqrt(6.0 / (self.w * rf + self.k * rf))
            O = (torch.rand(tuple(self.X.shape), generator=g) * 2.0 - 1.0) * lim
            return O.to(self.X.device)
        elif self.hidden_init == 'zeros':
            return torch.zeros_like(self.X)
        else:
            raise RuntimeError                                          # hgru_module.py:891-892

    def build(self, trace=False):
        """Run the circuit (hgru_module.py:872-959): `timesteps` iterations of `full` (:825-857).

        Returns O, or (O, weights, activities) when return_weights (the reference default).
        trace=True (non-reference) additionally stores per-timestep `self.I_steps`/`self.O_steps`
        [T,n,h,w,k]."""
        if not self.X.is_cuda:
            raise RuntimeError("ContextualCircuit.build() needs X on a CUDA device (no CPU fallback)")
        lib = _lib.load()
        self.prepare_tensors()
        plan = _get_plan(self.n, self.h, self.w, self.k, self.SSF_ext, self.timesteps,
                         _lib.MODES[self.compute_mode])
        self._plan = plan
        st = _stream()
        ptrs = [(self._rho_ones if (n == 'rho' and self._rho_ones is not None) else getattr(self, n)).data_ptr()
                for n in _lib.HGRU_PARAM_ORDER]
        _lib.check(lib.hgru_set_params(plan, *ptrs, st), "hgru_set_params")
        O0 = self._initial_state()
        O = torch.empty_like(self.X)
        I_tr = O_tr = None
        if trace:
            I_tr = torch.empty((self.timesteps,) + tuple(self.X.shape), device=self.X.device)
            O_tr = torch.empty_like(I_tr)
        _lib.check(lib.hgru_forward_batch(plan, self.n, self.X.data_ptr(), O0.data_ptr(), O.data_ptr(),
                                          I_tr.data_ptr() if trace else None,
                                          O_tr.data_ptr() if trace else None, st), "hgru_forward_batch")
        self.I_steps, self.O_steps = I_tr, O_tr
        self.gpu_launches = lib.hgru_plan_launch_count(plan)
        if self.return_weights:
            weights = self.gather_tensors(wak='weight')
            tuning = self.gather_tensors(wak='tuning')
            weights = dict(weights, **{})
            del tuning
            activities = self.gather_tensors(wak='activity')
            if self.association_field:
                weights['p_t'] = self.p_r
            return O, weights, activities
        return O
