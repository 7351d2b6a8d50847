"""Host-side mirror of models/network_utils.py for the render path: encodings and MLP
factories with the reference's names, config keys, parameter names and init rules, so that
models/geometry.py / models/texture.py can be pointed at this module unchanged.

    VanillaFrequency ........ models/network_utils.py:14-40
    ProgressiveBandHashGrid . models/network_utils.py:43-68
    CompositeEncoding ....... models/network_utils.py:71-90
    get_encoding ............ models/network_utils.py:93-106
    VanillaMLP .............. models/network_utils.py:109-157
    get_mlp ................. models/network_utils.py:194-204
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import relu_mlp, sdf_field, tc_autograd as tca
from . import tinycudann as tcnn
from .fused_mlp import PackedMLP


class Config(dict):
    """Minimal stand-in for the OmegaConf nodes the reference passes around
    (attribute access + .get + nested dicts)."""

    def __getattr__(self, k):
        try:
            v = self[k]
        except KeyError as e:
            raise AttributeError(k) from e
        return Config(v) if isinstance(v, dict) and not isinstance(v, Config) else v

    def __setattr__(self, k, v):
        self[k] = v


def config_to_primitive(config):
    return dict(config)


def update_module_step(m, epoch, global_step):
    """systems/utils.py: call update_step if the module has one."""
    if hasattr(m, "update_step"):
        m.update_step(epoch, global_step)


_FOLD_SCOPE = [0]          # 0: no sharing; otherwise the id of the running training step (see VanillaMLP.effective_weights)


class fold_once:
    """Context manager: within it every VanillaMLP folds its weight-norm parametrisation once."""
    _next = 0

    def __enter__(self):
        fold_once._next += 1
        self._prev, _FOLD_SCOPE[0] = _FOLD_SCOPE[0], fold_once._next
        return self

    def __exit__(self, *exc):
        _FOLD_SCOPE[0] = self._prev
        return False


class VanillaFrequency(nn.Module):
    def __init__(self, in_channels, config):
        super().__init__()
        self.N_freqs = config["n_frequencies"]
        self.n_input_dims = in_channels
        self.x_scale = config.get("x_scale", 1.0)
        self.x_offset = config.get("x_offset", 0.0)
        self.freq_bands = 2 ** torch.linspace(0, self.N_freqs - 1, self.N_freqs)
        self.n_output_dims = in_channels * 2 * self.N_freqs
        self.n_masking_step = config.get("n_masking_step", 0)
        self.update_step(None, None)

    def forward(self, x):
        """[..., C] -> [..., 2*F*C] in the reference's order (sin f0 | cos f0 | sin f1 | ...), models/network_utils.py:
        27-33.  All bands in one multiply / sin / cos instead of a Python loop of 4 launches per band: the products
        `freq * x` are the same fp32 multiplies (the bands are powers of two), so the values are bit-identical."""
        if x.is_cuda and self.N_freqs <= 16 and x.numel() > 0:
            # one kernel (csrc/glue.cu) instead of multiply / sin / cos / stack / mask / reshape
            from .glue import freq_encode
            mask = None if bool((self.mask == 1).all()) else self.mask
            return freq_encode(x, self.N_freqs, self.x_scale, self.x_offset, mask)
        x = x * self.x_scale + self.x_offset
        if self._bands is None or self._bands.device != x.device:
            self._bands = self.freq_bands.to(device=x.device, dtype=x.dtype)
            self._mask_dev = None if bool((self.mask == 1).all()) else self.mask.to(device=x.device, dtype=x.dtype)
        fx = x[..., None, :] * self._bands[:, None]                       # [..., F, C]
        out = torch.stack((torch.sin(fx), torch.cos(fx)), dim=-2)          # [..., F, 2, C]
        if self._mask_dev is not None:
            out = out * self._mask_dev[:, None, None]
        return out.reshape(*x.shape[:-1], self.n_output_dims)

    _bands = None
    _mask_dev = None

    def update_step(self, epoch, global_step):
        if self.n_masking_step <= 0 or global_step is None:
            self.mask = torch.ones(self.N_freqs, dtype=torch.float32)
        else:
            k = torch.arange(0, self.N_freqs)
            self.mask = (1.0 - torch.cos(math.pi * (global_step / self.n_masking_step * self.N_freqs - k).clamp(0, 1))) / 2.0
        self._bands = None                       # re-derive the device copies of bands / mask on the next call


class ProgressiveBandHashGrid(nn.Module):
    def __init__(self, in_channels, config):
        super().__init__()
        self.n_input_dims = in_channels
        encoding_config = dict(config)
        encoding_config["otype"] = "HashGrid"
        self.encoding = tcnn.Encoding(in_channels, encoding_config)
        self.n_output_dims = self.encoding.n_output_dims
        self.n_level = config["n_levels"]
        self.n_features_per_level = config["n_features_per_level"]
        self.start_level, self.start_step, self.update_steps = \
            config["start_level"], config["start_step"], config["update_steps"]
        self.current_level = self.start_level
        self.register_buffer("mask", torch.zeros(self.n_level * self.n_features_per_level), persistent=False)

    all_levels_on = False       # host-side: mask == 1 everywhere (set by update_step, the only writer of the mask)

    def forward(self, x):
        y = self.encoding(x)
        return y if self.all_levels_on else y * self.mask

    def update_step(self, epoch, global_step):
        current_level = min(self.start_level + max(global_step - self.start_step, 0) // self.update_steps,
                            self.n_level)
        self.current_level = current_level
        self.mask[: self.current_level * self.n_features_per_level] = 1.0
        self.all_levels_on = current_level >= self.n_level


class CompositeEncoding(nn.Module):
    def __init__(self, encoding, include_xyz=False, xyz_scale=1.0, xyz_offset=0.0):
        super().__init__()
        self.encoding = encoding
        self.include_xyz, self.xyz_scale, self.xyz_offset = include_xyz, xyz_scale, xyz_offset
        self.n_output_dims = int(self.include_xyz) * self.encoding.n_input_dims + self.encoding.n_output_dims

    def forward(self, x, *args):
        if not self.include_xyz:
            return self.encoding(x, *args)
        return torch.cat([x * self.xyz_scale + self.xyz_offset, self.encoding(x, *args)], dim=-1)

    def update_step(self, epoch, global_step):
        update_module_step(self.encoding, epoch, global_step)


def get_encoding(n_input_dims, config):
    config = Config(config)
    if config.otype == "VanillaFrequency":
        encoding = VanillaFrequency(n_input_dims, config_to_primitive(config))
    elif config.otype == "ProgressiveBandHashGrid":
        encoding = ProgressiveBandHashGrid(n_input_dims, config_to_primitive(config))
    else:
        encoding = tcnn.Encoding(n_input_dims, config_to_primitive(config))
    return CompositeEncoding(encoding, include_xyz=config.get("include_xyz", False),
                             xyz_scale=config.get("xyz_scale", 2.0), xyz_offset=config.get("xyz_offset", -1.0))


def get_activation(name):
    """models/utils.py:72-99 (subset reachable from the two configs)."""
    if name is None or str(name).lower() == "none":
        return lambda x: x
    name = name.lower()
    if name == "sigmoid":
        return torch.sigmoid
    if name == "tanh":
        return torch.tanh
    return getattr(F, name)


class VanillaMLP(nn.Module):
    """Same parameters as the reference (layers.N.weight | weight_g + weight_v, layers.N.bias,
    N = 0, 2, 4, ...).  forward() runs the fused sm_100a MLP kernels when they are built for the
    layer shape, through torch autograd otherwise."""

    def __init__(self, dim_in, dim_out, config):
        super().__init__()
        self.dim_in, self.dim_out = dim_in, dim_out
        self.n_neurons, self.n_hidden_layers = config["n_neurons"], config["n_hidden_layers"]
        self.sphere_init, self.weight_norm = config.get("sphere_init", False), config.get("weight_norm", False)
        self.sphere_init_radius = config.get("sphere_init_radius", 0.5)
        self.inside_outside = config.get("inside_outside", False)
        layers = [self.make_linear(dim_in, self.n_neurons, True, False), self.make_activation()]
        for _ in range(self.n_hidden_layers - 1):
            layers += [self.make_linear(self.n_neurons, self.n_neurons, False, False), self.make_activation()]
        layers += [self.make_linear(self.n_neurons, dim_out, False, True)]
        self.layers = nn.Sequential(*layers)
        self.output_activation = get_activation(config.get("output_activation", None))
        oa = config.get("output_activation", None)
        self.config_output_activation_is_identity = oa is None or str(oa).lower() == "none"

    @property
    def activation_name(self):
        return "softplus100" if self.sphere_init else "relu"

    def linears(self):
        return [m for m in self.layers if not isinstance(m, (nn.Softplus, nn.ReLU))]

    def effective_weights(self):
        """[(W [out,in], b [out])] with weight-norm folded (differentiable torch ops on the
        tiny parameter tensors; the big per-sample work happens in the kernels).

        Inside a `fold_once()` scope (one training step: train._Trainer) the folded tensors are computed once and
        shared by every call -- the split-sum step evaluates the SDF field with autograd four times, each of which used
        to fold the weights again, forward and backward (~90 tiny launches per step).  Autograd accumulates the calls'
        weight gradients on the shared tensor and runs the weight-norm backward once: the same sum, one rounding
        order.  Outside a scope nothing is cached (a graph kept past its backward could not be reused)."""
        key = (_FOLD_SCOPE[0], torch.is_grad_enabled())
        if _FOLD_SCOPE[0] and self._folded is not None and self._folded[0] == key:
            return self._folded[1]
        out = []
        for lin in self.linears():
            if hasattr(lin, "weight_g"):
                v, g = lin.weight_v, lin.weight_g
                W = v * (g / v.norm(dim=1, keepdim=True))
            else:
                W = lin.weight
            out.append((W, lin.bias))
        if _FOLD_SCOPE[0]:
            self._folded = (key, out)
        return out

    _folded = None

    def forward(self, x):
        return self._forward([x])

    def forward_segments(self, segs):
        """forward(cat(segs, -1)) without materialising the concatenation when a fused kernel takes the
        segments directly (models/texture.py builds its network inputs with torch.cat)."""
        return self._forward([s.reshape(-1, s.shape[-1]) for s in segs])

    def _forward(self, segs):
        """output_activation(network(cat(segs, -1))); the kernels follow from the inputs and the net's shape:
          CPU or non-2-D input: the nn.Linear stack;
          no grad: one fused tcgen05 inference launch -- SDF-shaped nets on the features-on-lanes kernels of
                   sdf_field (~2x the rows/s of the generic chain kernel), every other net on csrc/mlp_fwd.cu;
          grad:    SDF-shaped nets as one fused forward node / one fused backward kernel (sdf_field), ReLU nets of
                   width 128 as one tcgen05 launch per layer (relu_mlp), every other shape through the tcgen05 GEMM
                   primitives of tc_autograd (closed under differentiation; activations stay in torch).
        mlp_precision picks the operand precision of the sdf_field and relu_mlp kernels.  Only the kernels of ReLU
        nets read up to 3 input segments; everything else gets their concatenation."""
        if len(segs) > 1 and (len(segs) > 3 or self.sphere_init or not segs[0].is_cuda):
            segs = [torch.cat(segs, dim=-1)]
        x = segs[0]
        sdf_net = sdf_field.supports(self)
        if not (x.is_cuda and x.dim() == 2):
            h = self.layers(x.float())
        elif not torch.is_grad_enabled():
            h = self.packed()(x if sdf_net else segs)
        elif sdf_net:
            h, _ = sdf_field.fused_sdf(self, x, want_g0=False)
        elif relu_mlp.supports(self):
            h = relu_mlp.relu_mlp(self, segs)
        else:
            h = (x if len(segs) == 1 else torch.cat(segs, dim=-1)).float()
            ws = self.effective_weights()
            for i, (W, b) in enumerate(ws):
                h = tca.linear(h, W, b)
                if i + 1 < len(ws):
                    h = F.softplus(h, beta=100) if self.sphere_init else F.relu(h)
        return self.output_activation(h)

    def packed(self):
        """The inference launcher with this net's packed weights (PackedSDF for an SDF-shaped net, PackedMLP
        otherwise), made once; it re-packs when a parameter changes."""
        if self._packed is None:
            self._packed = sdf_field.PackedSDF(self) if sdf_field.supports(self) else PackedMLP(self)
        return self._packed

    _packed = None
    # "fp32": every GEMM as three fp16 products of hi|lo operands with fp32 accumulation -- fp32-class, the parity path.
    # "fp16": the reduced-precision VARIANT named by the north star -- single fp16 plane, one product per GEMM, half
    #         the activation-stream bytes (fused SDF field fwd/bwd and the ReLU training nets).  Stated tolerance:
    #         tests/test_gpu_mlp_fp16.py (outputs 2e-3 of their scale; end to end: images 5e-3, gradients 3e-2 rel-L2).
    mlp_precision = "fp32"

    def make_linear(self, dim_in, dim_out, is_first, is_last):
        layer = nn.Linear(dim_in, dim_out, bias=True)
        if self.sphere_init:
            if is_last:
                sign = -1.0 if self.inside_outside else 1.0
                nn.init.constant_(layer.bias, -sign * self.sphere_init_radius)
                nn.init.normal_(layer.weight, mean=sign * math.sqrt(math.pi) / math.sqrt(dim_in), std=0.0001)
            elif is_first:
                nn.init.constant_(layer.bias, 0.0)
                nn.init.constant_(layer.weight[:, 3:], 0.0)
                nn.init.normal_(layer.weight[:, :3], 0.0, math.sqrt(2) / math.sqrt(dim_out))
            else:
                nn.init.constant_(layer.bias, 0.0)
                nn.init.normal_(layer.weight, 0.0, math.sqrt(2) / math.sqrt(dim_out))
        else:
            nn.init.constant_(layer.bias, 0.0)
            nn.init.kaiming_uniform_(layer.weight, nonlinearity="relu")
        if self.weight_norm:
            layer = nn.utils.weight_norm(layer)
        return layer

    def make_activation(self):
        return nn.Softplus(beta=100) if self.sphere_init else nn.ReLU(inplace=True)


def get_mlp(n_input_dims, n_output_dims, config):
    config = Config(config)
    if config.otype == "VanillaMLP":
        return VanillaMLP(n_input_dims, n_output_dims, config_to_primitive(config))
    if config.otype == "Identity":
        return nn.Identity()
    raise NotImplementedError("tcnn networks are not built by the reference (README.md:56 --no-networks)")
