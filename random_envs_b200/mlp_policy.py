"""A trained MLP policy for the fused cart-pole kernels (include/renv.h ``renv_mlp_policy``).

    policy = MLPPolicy.from_module(net, device)      # net: Linear(4,h1) -> Tanh|ReLU -> Linear(h1,h2) -> act -> Linear(h2,o)
    actions = venv.policy_actions(policy)            # then venv.step(actions), or
    venv.rollout(policy, num_steps=500)              # K fused env-steps with the policy evaluated in the kernel

One architecture is supported, padded on the host to 64 units: ``h1, h2 <= 64``, the same ``Tanh`` or ``ReLU`` in both
places, ``o`` = 1 or 2 outputs.  The action is ``argmax(l0, l1)`` with ties going to 0 (``torch.argmax``); a 1-output
head is taken as ``l0 = 0, l1 = l``, i.e. ``a = [l > 0]``.  The padding is exact: the added units have zero weights and
biases and ``tanh(0) = relu(0) = 0``.  The kernels evaluate the net with fp32-class accuracy (the 64 x 64 layer on the
tensor cores as 3xTF32): ``max |logit - float64 logit| <= 1e-5 * max(1, max |float64 logit|)``.

A 1-output net packed the same way is a critic: ``V(s) = l1`` (``outputs == 1``), which
``RandomCartPoleVecEnv.gae(traj, critic)`` evaluates on a collected trajectory.

``MLPPopulation`` stacks P such policies (one activation) for ``RandomCartPoleVecEnv.evaluate_population``, which
evaluates them all on common tasks in one kernel.
"""
import numpy as np

from . import _device, _lib

HIDDEN = 64
PARAM_FLOATS = 4612             # RENV_MLP_PARAM_FLOATS
_OFF = dict(w1=0, b1=256, w2=320, b2=4416, w3=4480, b3=4608)
TANH, RELU = 0, 1               # RENV_MLP_TANH / RENV_MLP_RELU


def _layers(module):
    t = _device.torch()
    nn = t.nn
    mods = list(module) if isinstance(module, nn.Sequential) else None
    if mods is None or len(mods) != 5:
        raise ValueError("the policy must be nn.Sequential(Linear(4, h1), act, Linear(h1, h2), act, Linear(h2, o))")
    l1, a1, l2, a2, l3 = mods
    if not all(type(m) is nn.Linear for m in (l1, l2, l3)):
        raise ValueError("layers 0, 2 and 4 of the policy must be nn.Linear")
    if type(a1) is not type(a2) or type(a1) not in (nn.Tanh, nn.ReLU):
        raise ValueError("the activations must both be nn.Tanh or both nn.ReLU, got %s and %s"
                         % (type(a1).__name__, type(a2).__name__))
    if l1.in_features != 4:
        raise ValueError("the policy takes the 4-dim cart-pole observation, not %d inputs" % l1.in_features)
    if l1.out_features > HIDDEN or l2.out_features > HIDDEN:
        raise ValueError("hidden widths above %d are not supported (%d, %d)" % (HIDDEN, l1.out_features, l2.out_features))
    if l2.in_features != l1.out_features or l3.in_features != l2.out_features:
        raise ValueError("consecutive Linear layers do not chain")
    if l3.out_features not in (1, 2):
        raise ValueError("the head must have 1 or 2 outputs (Discrete(2)), not %d" % l3.out_features)
    return (l1, l2, l3), (TANH if type(a1) is nn.Tanh else RELU)


def pack(module):
    """Validate ``module`` and return (float32 numpy array of PARAM_FLOATS in the include/renv.h layout, activation id)."""
    (l1, l2, l3), act = _layers(module)
    out = np.zeros(PARAM_FLOATS, dtype=np.float32)

    def put(name, shape, lin, weight):
        block = np.zeros(shape, dtype=np.float32)
        v = (lin.weight if weight else lin.bias)
        if v is not None:
            v = v.detach().to("cpu").float().numpy()
            block[tuple(slice(0, s) for s in v.shape)] = v
        out[_OFF[name]:_OFF[name] + block.size] = block.ravel()
        return block

    put("w1", (HIDDEN, 4), l1, True); put("b1", (HIDDEN,), l1, False)
    put("w2", (HIDDEN, HIDDEN), l2, True); put("b2", (HIDDEN,), l2, False)
    w3 = np.zeros((2, HIDDEN), dtype=np.float32)
    b3 = np.zeros(2, dtype=np.float32)
    w = l3.weight.detach().to("cpu").float().numpy()
    b = l3.bias.detach().to("cpu").float().numpy() if l3.bias is not None else np.zeros(w.shape[0], np.float32)
    if w.shape[0] == 2:
        w3[:, :w.shape[1]], b3[:] = w, b
    else:                                   # 1 output l: l0 = 0, l1 = l
        w3[1, :w.shape[1]], b3[1] = w[0], b[0]
    out[_OFF["w3"]:_OFF["w3"] + 2 * HIDDEN] = w3.ravel()
    out[_OFF["b3"]:_OFF["b3"] + 2] = b3
    return out, act


def reference_logits(params, activation, obs):
    """float64 evaluation of packed parameters on (N, 4) float64 observations -> (N, 2) logits (torch, any device)."""
    t = _device.torch()
    p = t.as_tensor(np.asarray(params, dtype=np.float64) if not isinstance(params, t.Tensor) else params.double().cpu(),
                    dtype=t.float64).to(obs.device)
    act = t.tanh if activation == TANH else t.relu
    g = lambda k, shape: p[_OFF[k]:_OFF[k] + int(np.prod(shape))].reshape(shape)
    h = act(obs @ g("w1", (HIDDEN, 4)).t() + g("b1", (HIDDEN,)))
    h = act(h @ g("w2", (HIDDEN, HIDDEN)).t() + g("b2", (HIDDEN,)))
    return h @ g("w3", (2, HIDDEN)).t() + g("b3", (2,))


class MLPPolicy:
    """Packed device parameters of a supported ``nn.Sequential`` policy (see the module docstring).  ``outputs`` is
    the width of the net's head, 1 or 2 (``from_module`` reads it from the net)."""

    def __init__(self, params, activation, device, outputs=2):
        t = _device.torch()
        if outputs not in (1, 2):
            raise ValueError("outputs must be 1 or 2, got %r" % (outputs,))
        self.activation = int(activation)
        self.outputs = int(outputs)     # width of the head: 1 for a critic V(s) = l1 (``RandomCartPoleVecEnv.gae``)
        self.device = t.device(device)
        self.params = t.as_tensor(params, dtype=t.float32).to(self.device).contiguous()    # 16-byte aligned allocation
        s = _lib.MlpPolicy()
        s.params, s.activation = self.params.data_ptr(), self.activation
        self.struct = s

    @classmethod
    def from_module(cls, module, device=None):
        """Validate and pack ``module``.  Raises ValueError for anything but the supported architecture."""
        params, act = pack(module)
        return cls(params, act, _device.require_cuda(device), outputs=list(module)[4].out_features)

    def reference_logits(self, obs):
        """float64 logits of the packed (padded) net for (N, 4) observations."""
        return reference_logits(self.params, self.activation, obs.double())


class MLPPopulation:
    """P packed MLP policies with one activation, for ``RandomCartPoleVecEnv.evaluate_population``.  ``params`` is a
    (P, PARAM_FLOATS) float32 device tensor whose row p is laid out as ``MLPPolicy.params``.  It may be edited in place
    between evaluations, e.g. for ES perturbations of the weights; the padded entries of a net narrower than 64 units
    must stay zero, otherwise the padded units stop being inert and the population is no longer the nets it was made
    from."""

    def __init__(self, params, activation, device=None):
        t = _device.torch()
        params = t.as_tensor(params, dtype=t.float32)
        if params.dim() != 2 or params.shape[0] < 1 or params.shape[1] != PARAM_FLOATS:
            raise ValueError("a population is a (P >= 1, %d) array of packed policies, got %s"
                             % (PARAM_FLOATS, tuple(params.shape)))
        if int(activation) not in (TANH, RELU):
            raise ValueError("activation must be TANH (%d) or RELU (%d), got %r" % (TANH, RELU, activation))
        self.activation = int(activation)
        # rows of 18,448 bytes: each 16-byte aligned
        self.params = params.to(device if device is not None else params.device).contiguous()
        self.device = self.params.device        # with its index: "cuda" is the current device, as for the env's buffers

    @classmethod
    def from_modules(cls, modules, device=None):
        """Validate and pack every module of ``modules``; they must share one activation (ValueError otherwise)."""
        packed = [pack(m) for m in modules]
        if not packed:
            raise ValueError("a population needs at least one module")
        acts = sorted({act for _, act in packed})
        if len(acts) != 1:
            raise ValueError("the modules of a population must share one activation (Tanh or ReLU), got both")
        return cls(np.stack([p for p, _ in packed]), acts[0], _device.require_cuda(device))

    @classmethod
    def from_policies(cls, policies):
        """Stack ``MLPPolicy`` objects of one activation and one device (copies their parameters)."""
        policies = list(policies)
        if not policies:
            raise ValueError("a population needs at least one policy")
        if len({p.activation for p in policies}) != 1 or len({p.device for p in policies}) != 1:
            raise ValueError("the policies of a population must share one activation and one device")
        t = _device.torch()
        return cls(t.stack([p.params for p in policies]), policies[0].activation, policies[0].device)

    def __len__(self):
        return int(self.params.shape[0])

    def member(self, p):
        """An ``MLPPolicy`` viewing row ``p`` of ``params`` (no copy: in-place edits show through both ways)."""
        return MLPPolicy(self.params[p], self.activation, self.device)
