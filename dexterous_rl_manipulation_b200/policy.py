"""A trained MLP policy evaluated inside the fused rollout (``dexsim_rollout_mlp``).

``MlpPolicy.from_torch(net)`` packs the parameters of an ``nn.Sequential`` of the form
``Linear(45, h1), ReLU|Tanh, [Linear(h1, h2), same activation,] Linear(h_last, 15)`` once, on the device;
``env.rollout(k, policy=mlp)`` then acts with it on the observation of every env at every step, and ``mlp.mean(obs)``
returns the network's output for given observations with the rollout's arithmetic (include/dexsim.h).
"""
import ctypes as C
import hashlib

import torch

from . import _lib


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class MlpPolicy:
    """Gaussian MLP policy: action = clip(mean(obs) + action_std * N(0, 1), -1, 1), the normals drawn in the kernel
    from Philox stream 4 (``action_std=None``: the deterministic policy clip(mean(obs), -1, 1))."""

    def __init__(self, params, hidden, activation, action_std=None, device="cuda"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("MlpPolicy needs a CUDA device; there is no CPU path")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        hidden = tuple(int(h) for h in hidden)
        if len(hidden) not in (1, 2) or not all(1 <= h <= _lib.MLP_MAX_WIDTH for h in hidden):
            raise ValueError(f"one or two hidden layers of 1..{_lib.MLP_MAX_WIDTH} units, got {hidden}")
        if activation not in ("relu", "tanh"):
            raise ValueError("activation must be 'relu' or 'tanh'")
        sizes = (45,) + hidden + (15,)
        expect = sum(o * i + o for i, o in zip(sizes[:-1], sizes[1:]))
        params = torch.as_tensor(params, dtype=torch.float32).reshape(-1)
        if params.numel() != expect:
            raise ValueError(f"{expect} packed parameters expected for {sizes}, got {params.numel()}")
        self.hidden, self.activation = hidden, activation
        self.params = params.to(self.device).contiguous().clone()       # a fresh allocation: 16-byte aligned
        self.action_std = None
        # whether the policy has a Gaussian density (the log_prob of a policy record): action_std given, every entry
        # finite and > 0 -- decided here, on the host, once
        self.std_has_density = False
        if action_std is not None:
            std = torch.as_tensor(action_std, dtype=torch.float32).reshape(-1)
            if std.numel() == 1:
                std = std.expand(15)
            if std.numel() != 15:
                raise ValueError("action_std must be a scalar or hold 15 entries")
            self.std_has_density = bool(torch.isfinite(std.cpu()).all()) and bool((std.cpu() > 0).all())
            self.action_std = torch.zeros(16, dtype=torch.float32, device=self.device)
            self.action_std[:15] = std.to(self.device)
        self._struct = _lib.DexsimMlpPolicy(
            self.params.data_ptr(), len(hidden), (C.c_int32 * 2)(hidden[0], hidden[1] if len(hidden) == 2 else 0),
            _lib.ACT_RELU if activation == "relu" else _lib.ACT_TANH,
            None if self.action_std is None else self.action_std.data_ptr())

    @classmethod
    def from_torch(cls, module, action_std=None, device="cuda"):
        """Pack ``nn.Sequential(Linear(45, h1), ReLU|Tanh, [Linear(h1, h2), same activation,] Linear(h_last, 15))``.
        Any other module, a Linear without bias or a width outside 1..64 raises ValueError."""
        return cls(*cls.pack(module), action_std=action_std, device=device)

    @staticmethod
    def pack(module):
        """(params, hidden, activation) of ``from_torch`` on the host: the float32 parameters in the packed layout of
        include/dexsim.h (W1, b1, [W2, b2,] W3, b3, each in torch's [out, in] order), the hidden widths and
        'relu' / 'tanh'."""
        nn = torch.nn
        if not isinstance(module, nn.Sequential):
            raise ValueError("expected an nn.Sequential")
        layers = list(module)
        if len(layers) not in (3, 5):
            raise ValueError("expected Linear, activation, [Linear, activation,] Linear")
        linears, acts = layers[0::2], layers[1::2]
        if not all(type(m) is nn.Linear and m.bias is not None for m in linears):
            raise ValueError("every other layer must be an nn.Linear with bias")
        kinds = {type(a) for a in acts}
        if kinds not in ({nn.ReLU}, {nn.Tanh}):
            raise ValueError("the hidden layers must all use nn.ReLU or all use nn.Tanh")
        if linears[0].in_features != 45 or linears[-1].out_features != 15:
            raise ValueError("the network must map 45 observation entries to 15 actions")
        for a, b in zip(linears[:-1], linears[1:]):
            if a.out_features != b.in_features:
                raise ValueError("consecutive Linear layers do not fit together")
        hidden = [m.out_features for m in linears[:-1]]
        if not all(1 <= h <= _lib.MLP_MAX_WIDTH for h in hidden):
            raise ValueError(f"hidden widths must be 1..{_lib.MLP_MAX_WIDTH}, got {hidden}")
        with torch.no_grad():
            params = torch.cat([t.detach().to(torch.float32).reshape(-1).cpu()
                                for m in linears for t in (m.weight, m.bias)])
        return params, hidden, "relu" if kinds == {nn.ReLU} else "tanh"

    def sha256(self):
        """Hex SHA-256 of what fixes the policy's actions: the hidden widths, the activation, the packed parameters and
        ``action_std`` (or its absence).  Evaluation results carry it so that a saved result can be tied to its
        network, and replays refuse a different one."""
        h = hashlib.sha256(repr((self.hidden, self.activation)).encode())
        h.update(self.params.cpu().numpy().tobytes())
        h.update(b"std:" + self.action_std[:15].cpu().numpy().tobytes() if self.action_std is not None else b"no std")
        return h.hexdigest()

    def mean(self, obs):
        """The network's output for ``obs`` [n, 45] (any device, cast to float32): [n, 15] on the policy's device,
        bit for bit what the fused rollout computes for the same observations (``dexsim_mlp_policy_mean``)."""
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device).reshape(-1, 45)
        n = obs.shape[0]
        ld = max(32, (n + 31) // 32 * 32)
        soa = torch.zeros(45, ld, dtype=torch.float32, device=self.device)
        soa[:, :n] = obs.t()
        out = torch.empty(15, ld, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().dexsim_mlp_policy_mean(C.byref(self._struct), soa.data_ptr(), n, ld, out.data_ptr(),
                                                         _stream(self.device)), "dexsim_mlp_policy_mean")
        return out[:, :n].t()
