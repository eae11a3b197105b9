"""Policy-side consumer of the observation tensor (SURVEY.md 8f-4): the network of the reference's
models/conv_to_fcnet_v2.py (ConvToFCNetv2) evaluated on uint8 observations that never leave the GPU.

    trunk   Conv2D(6, 3x3, stride 1, 'valid') -> ReLU -> flatten -> Dense(32) -> ReLU -> Dense(32) -> ReLU
            (conv_to_fcnet_v2.py:36-66, filters as train_baseline.py:104 configures them) -- ONE fused tcgen05 kernel
            behind the C ABI (`ssd_policy_features`, csrc/ssd_policy.cu) that reads the uint8 [B, N, 15, 15, 3] tensor
            `BatchedSSDEnv.step` wrote and folds the (x - 128) / 255 of map_env.py:199 into the first layer;
    head    LSTM(cell_size) -> logits / value (conv_to_fcnet_v2.py:68-92).  For the reference's cell_size 128 this is a second
            fused tcgen05 kernel (`ssd_policy_lstm_heads`: gate GEMM in tensor memory, cell update, head GEMM and -- in
            `act` -- Gumbel-max sampling of the action, one pass over the recurrent state).  Other cell sizes take the
            unfused route: library GEMMs (torch / cuBLAS, bf16 operands) around the one-pass cell update
            `ssd_policy_lstm_cell`.

The recurrent state (h, c) of the fused route lives in HBM in the kernel's tiled layout, shape [ceil(M/128), 8, 128, 16]
(group of 128 agents, block of 16 units, agent, unit): a warp of the cell update then moves 2 KB contiguous per access.  Treat
it as opaque between steps (as RLlib does with state_out -> state_in); `state_rows` / `state_from_rows` convert to and from
[M, cell_size].

One network per agent id -- the reference's training scripts (run_scripts/train_baseline.py, train_moa.py) build a policy per
'agent-i' and map agent i to it -- is `ConvToFCNet([weights_0, ..., weights_{P-1}])`: agent (b, p) of a [B, P, 15, 15, 3]
observation tensor is evaluated with weights_p by the same two kernels (one CTA serves one policy), outputs stay agent-major,
and the tiled state is grouped per policy, [P * ceil(B/128), 8, 128, 16].

A policy pool -- K <= 255 weight sets loaded once, and a uint8 policy id per agent with every call, as RLlib's
policy_mapping_fn may assign them per agent and per episode -- is `PolicyPool([weights_0, ..., weights_{K-1}])`: several runs
or seeds on one GPU, cross-play teams, population play.  The kernels group the agents by id on the device; an id >= K leaves
the agent to the caller's own code (scripted agents).  Its state is the shared network's agent-major tiled layout, so the ids
may change while a state is alive.

Weights are numpy fp32 arrays in the Keras layouts (conv kernel [kh, kw, in, out], dense kernels [in, out], LSTM kernel
[in, 4u] / recurrent kernel [u, 4u] / bias [4u] with gates ordered i, f, c, o), so a checkpoint of the reference model
loads without transposition.  There is no CPU path: the trunk raises without the CUDA library.

`policy_step` returns what a sampler records per step -- the action, its log-probability, the entropy, the logits, the value and
the next state (a `PolicyStep`) -- for a sampled, a greedy or a caller-given action, from the same fused head kernel
(`ssd_policy_lstm_heads_dist`).

`MOANet` is the model of other agents of the causal-influence models (train_moa.py): from the trunk features, the joint action
and the policy's logits it predicts the others' next actions, for the actual and for every counterfactual own action, and
returns the social-influence reward (`MOAStep`), all in one kernel (`ssd_moa_step`).  `MOAPool` is its policy pool: K <= 255
MOA weight sets and a policy id per agent with every step (`ssd_moa_pool_step`), typically the ids of the PolicyPool call of
the same step.  `policy_step(..., features=x)` takes the features already computed for the MOA, so the trunk runs once per step.
"""
import collections
import ctypes as C

import numpy as np
import torch

from . import _lib

VIEW_RADIUS = 7
OBS_SIDE = 2 * VIEW_RADIUS + 1
CONV_FILTERS = 6
FEATURES = 32
FLAT = (OBS_SIDE - 2) * (OBS_SIDE - 2) * CONV_FILTERS   # 1014


PolicyStep = collections.namedtuple("PolicyStep", "actions logp entropy logits value h c")
PolicyStep.__doc__ = """One step of the policy for M agents: actions int8 [M], logp float32 [M] (log softmax(logits) at the action), entropy
float32 [M] (of softmax(logits)), logits float32 [M, A], value float32 [M], and the next recurrent state (h, c)."""

_MODES = {"sample": _lib.ACT_SAMPLE, "greedy": _lib.ACT_GREEDY, "given": _lib.ACT_GIVEN}


def random_weights(num_outputs, cell_size=128, seed=0):
    """Random-init weights of the right shapes (normc for the dense layers as conv_to_fcnet_v2.py:63, glorot elsewhere)."""
    rng = np.random.RandomState(seed)

    def normc(shape, std=1.0):
        w = rng.randn(*shape).astype(np.float32)
        return (w * std / np.sqrt(np.square(w).sum(axis=0, keepdims=True))).astype(np.float32)

    def glorot(shape, fan_in, fan_out):
        lim = np.sqrt(6.0 / (fan_in + fan_out))
        return rng.uniform(-lim, lim, size=shape).astype(np.float32)

    u = cell_size
    return {
        "conv_w": glorot((3, 3, 3, CONV_FILTERS), 27, 9 * CONV_FILTERS), "conv_b": (0.1 * rng.randn(CONV_FILTERS)).astype(np.float32),
        "fc1_w": normc((FLAT, FEATURES)), "fc1_b": (0.1 * rng.randn(FEATURES)).astype(np.float32),
        "fc2_w": normc((FEATURES, FEATURES)), "fc2_b": (0.1 * rng.randn(FEATURES)).astype(np.float32),
        "lstm_w": glorot((FEATURES, 4 * u), FEATURES, 4 * u), "lstm_u": glorot((u, 4 * u), u, 4 * u),
        "lstm_b": np.concatenate([np.zeros(u), np.ones(u), np.zeros(2 * u)]).astype(np.float32),   # unit forget bias
        "logits_w": glorot((u, num_outputs), u, num_outputs), "logits_b": np.zeros(num_outputs, np.float32),
        "value_w": glorot((u, 1), u, 1), "value_b": np.zeros(1, np.float32),
    }


def _cuda_device(device):
    device = torch.device(device)
    if device.type != "cuda":
        raise _lib.SsdError("the policy trunk runs on a CUDA device only")
    if device.index is None:  # 'cuda' means the current device, not device 0
        device = torch.device("cuda", torch.cuda.current_device())
    return device


def _aligned(t):
    """`t` contiguous and starting on a 16-byte boundary, as the C ABI requires: a view such as obs[1:] is contiguous but starts
    inside its allocation (675 bytes in), so it is copied."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _weight_sets(weights):
    """One dict or a list of dicts -> the list of weight sets as contiguous fp32 arrays, checked to share names and shapes."""
    sets = list(weights) if isinstance(weights, (list, tuple)) else [weights]
    if not sets:
        raise ValueError("no weight sets")
    sets = [{k: np.ascontiguousarray(v, dtype=np.float32) for k, v in ws.items()} for ws in sets]
    w = sets[0]
    for name, shape in (("conv_w", (3, 3, 3, CONV_FILTERS)), ("conv_b", (CONV_FILTERS,)), ("fc1_w", (FLAT, FEATURES)),
                        ("fc1_b", (FEATURES,)), ("fc2_w", (FEATURES, FEATURES)), ("fc2_b", (FEATURES,))):
        if w[name].shape != shape:
            raise ValueError("%s has shape %s, expected %s" % (name, w[name].shape, shape))
    for p, ws in enumerate(sets[1:], 1):
        if sorted(ws) != sorted(w) or any(ws[k].shape != w[k].shape for k in w):
            raise ValueError("weights[%d] does not have the names and shapes of weights[0]" % p)
    return sets


def _step_mode(mode, actions, m, num_outputs, device):
    """-> (SSD_ACT_* code, the given actions as a contiguous int8 [m] tensor or None).  Integer actions outside 0..A-1 become
    -1 or A before the narrowing to int8, so every one of them gets logp NaN (none wraps onto a valid action).  They are
    widened to int64 first: clamped in an unsigned dtype, the bound -1 would itself wrap to the dtype's maximum."""
    if mode not in _MODES:
        raise ValueError("mode must be 'sample', 'greedy' or 'given', not %r" % (mode,))
    if mode != "given":
        if actions is not None:
            raise ValueError("actions are an input of mode 'given' only")
        return _MODES[mode], None
    if not isinstance(actions, torch.Tensor) or actions.device != device or actions.numel() != m \
            or actions.dtype.is_floating_point or actions.dtype.is_complex or actions.dtype == torch.bool:
        raise ValueError("mode 'given' takes actions, an integer tensor of %d elements on %s" % (m, device))
    a = actions.reshape(-1)
    if a.dtype != torch.int8:
        a = a.long().clamp(-1, num_outputs).to(torch.int8)
    return _MODES[mode], a.contiguous()


def _torch_step(logits, value, h, c, code, given, generator):
    """PolicyStep of the unfused route: log_softmax, argmax and torch.multinomial over the logits `forward` returned."""
    logp_all = torch.log_softmax(logits, dim=1)
    if code == _lib.ACT_SAMPLE:
        a = torch.multinomial(torch.softmax(logits, dim=1), 1, generator=generator).squeeze(1)
    elif code == _lib.ACT_GREEDY:
        a = logits.argmax(dim=1)   # the first maximum
    else:
        a = given.long()
    valid = (a >= 0) & (a < logits.shape[1])
    logp = logp_all.gather(1, torch.where(valid, a, 0)[:, None]).squeeze(1).masked_fill(~valid, float("nan"))
    entropy = -(logp_all.exp() * logp_all).sum(dim=1)
    return PolicyStep(given if given is not None else a.to(torch.int8), logp, entropy, logits, value, h, c)


def _state_rows(state, m, P):
    """Tiled state [G, 8, 128, 16] (grouped per policy for P > 1) -> agent-major [m, cell_size] (a copy)."""
    g, b, r, e = state.shape
    rows = state.permute(0, 2, 1, 3).reshape(g * r, b * e)
    if P == 1:
        return rows[:m].contiguous()
    return rows.reshape(P, g // P * r, b * e)[:, :m // P].transpose(0, 1).reshape(m, b * e)   # (p, b) -> agent b * P + p


def _state_from_rows(rows, P):
    """Agent-major [m, cell_size] -> tiled state [P * ceil(m / P / 128), cell_size/16, 128, 16], zero padded."""
    m, u = rows.shape
    g = (m // P + 127) // 128
    full = torch.zeros((P, g * 128, u), dtype=rows.dtype, device=rows.device)
    full[:, :m // P] = rows.reshape(m // P, P, u).transpose(0, 1)
    return full.reshape(P * g, 128, u // 16, 16).permute(0, 2, 1, 3).contiguous()


class _Handle(object):
    """A library handle on self.device: its lifetime and the stream its calls are ordered on."""
    _destroy = "ssd_policy_destroy"

    def close(self):
        if self._h:
            getattr(_lib.lib, self._destroy)(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)


class _Policy(_Handle):
    """What ConvToFCNet and PolicyPool share: the Philox key of the fused sampler and the calls of the fused head."""
    _sample_seed, _sample_counter = 0, 0

    def seed_sampling(self, seed):
        """Key of the Philox streams `act` samples from (counter = number of `act` and sampling `policy_step` calls since)."""
        self._sample_seed, self._sample_counter = int(seed) & (2 ** 64 - 1), 0

    def _heads(self, obs, ids, h, c, code=None, given=None, dist=False, features=None):
        """-> PolicyStep of the fused head on the features of obs, or on `features` (checked by `_given_features`) without running
        the trunk (ids: the pool's policy ids as `_ids` returns them, None for a network).  dist False:
        ssd_policy_[pool_]lstm_heads, which samples the actions when code is ACT_SAMPLE and takes none otherwise (logp and entropy
        None); dist True: ssd_policy_[pool_]lstm_heads_dist in mode `code`, on the `given` actions for ACT_GIVEN.  A sampling call
        advances the Philox counter."""
        if features is not None:
            x = features
        else:
            x = self.features(obs) if ids is None else self.features(obs, ids)
        m = x.shape[0]
        self._check_state(h, c, m)
        h, c = _aligned(h), _aligned(c)
        h_new, c_new = torch.empty_like(h), torch.empty_like(c)
        logits = torch.empty((m, self.num_outputs), dtype=torch.float32, device=self.device)
        value = torch.empty((m,), dtype=torch.float32, device=self.device)
        a = logp = entropy = None
        if given is not None:
            a = given
        elif dist or code == _lib.ACT_SAMPLE:   # a pool's skipped agents keep -1
            a = torch.empty((m,), dtype=torch.int8, device=self.device) if ids is None else torch.full((m,), -1, dtype=torch.int8, device=self.device)
        p = lambda t: C.c_void_p(t.data_ptr() if t is not None else None)
        lead = (self._h, p(x)) if ids is None else (self._h, p(x), p(ids))
        state = (p(h), p(c), p(h_new), p(c_new), p(logits), p(value))
        key = (m, self._sample_seed, self._sample_counter & 0xFFFFFFFF, self._stream())
        if dist:
            logp, entropy = torch.empty_like(value), torch.empty_like(value)
            fn = _lib.lib.ssd_policy_lstm_heads_dist if ids is None else _lib.lib.ssd_policy_pool_lstm_heads_dist
            _lib.check(fn(*lead, *state, code, p(a), p(logp), p(entropy), *key))
        else:
            fn = _lib.lib.ssd_policy_lstm_heads if ids is None else _lib.lib.ssd_policy_pool_lstm_heads
            _lib.check(fn(*lead, *state, p(a), *key))
        if code == _lib.ACT_SAMPLE:
            self._sample_counter += 1
        return PolicyStep(a, logp, entropy, logits, value, h_new, c_new)

    def _given_features(self, features, m):
        """`features` of a policy_step call: None, or float32 [m, 32] on the device (what `features` returns), made aligned."""
        if features is None:
            return None
        if not isinstance(features, torch.Tensor) or features.dtype != torch.float32 or features.device != self.device \
                or tuple(features.shape) != (m, FEATURES):
            raise ValueError("features must be a float32 [%d, %d] tensor on %s" % (m, FEATURES, self.device))
        return _aligned(features)


class ConvToFCNet(_Policy):
    """Forward pass of ConvToFCNetv2 for a batch of agents; `obs` is the uint8 tensor of the step path.

    `weights` is one dict (one network shared by all agents) or a list of P dicts, weights[p] being the policy of 'agent-p':
    agent m = b * P + p of the flattened [B, P, ...] batch is then evaluated with weights[p].  P > 1 needs the fused head
    (cell_size 128, 1..15 outputs)."""

    def __init__(self, weights, device="cuda:0"):
        self.device = _cuda_device(device)
        sets = _weight_sets(weights)
        w = sets[0]
        self.num_policies = P = len(sets)
        self.weights = w if P == 1 and not isinstance(weights, (list, tuple)) else sets
        self.cell_size = w["lstm_u"].shape[0] if "lstm_u" in w else 0
        self.num_outputs = w["logits_w"].shape[1] if "logits_w" in w else 0
        fused = self.cell_size == 128 and 1 <= self.num_outputs <= 15
        if P > 1 and not fused:
            raise ValueError("a network per agent needs the fused head: cell_size 128 and 1..15 outputs (got %d, %d)"
                             % (self.cell_size, self.num_outputs))
        if P > 1:   # P consecutive arrays behind every weight pointer
            w = {k: np.ascontiguousarray(np.stack([ws[k] for ws in sets])) for k in w}
        self._h = C.c_void_p()
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        _lib.check(_lib.lib.ssd_policy_create_n(VIEW_RADIUS, self.device.index, P, ptr(w["conv_w"]), ptr(w["conv_b"]), ptr(w["fc1_w"]),
                                                ptr(w["fc1_b"]), ptr(w["fc2_w"]), ptr(w["fc2_b"]), C.byref(self._h)))
        self._head = {}
        self._fused_head = False
        if fused:
            _lib.check(_lib.lib.ssd_policy_set_head_n(self._h, P, self.cell_size, self.num_outputs, ptr(w["lstm_w"]), ptr(w["lstm_u"]),
                                                      ptr(w["lstm_b"]), ptr(w["logits_w"]), ptr(w["logits_b"]), ptr(w["value_w"]),
                                                      ptr(w["value_b"])))
            self._fused_head = True
        if self.cell_size and P == 1:
            if self.cell_size % 8:
                raise ValueError("cell_size must be a multiple of 8")
            dev = lambda k, dt: torch.from_numpy(w[k]).to(self.device, dtype=dt).contiguous()
            self._head = {"lstm_w": dev("lstm_w", torch.bfloat16), "lstm_u": dev("lstm_u", torch.bfloat16), "lstm_b": dev("lstm_b", torch.float32),
                          "logits_w": dev("logits_w", torch.bfloat16), "logits_b": dev("logits_b", torch.float32),
                          "value_w": dev("value_w", torch.bfloat16), "value_b": dev("value_b", torch.float32)}

    def _groups(self, m):
        """Number of 128-agent state groups of m agents: P * ceil(m / P / 128)."""
        P = self.num_policies
        if m % P:
            raise ValueError("%d agents do not split into %d per-agent policies" % (m, P))
        return P * ((m // P + 127) // 128)

    def features(self, obs, out=None):
        """uint8 [..., 15, 15, 3] on the device -> float32 [M, 32] (M = product of the leading dims).  A network per agent
        takes [B, P, 15, 15, 3] or [B * P, 15, 15, 3]; rows stay agent-major."""
        if obs.dtype != torch.uint8 or obs.device != self.device or tuple(obs.shape[-3:]) != (OBS_SIDE, OBS_SIDE, 3):
            raise ValueError("obs must be a uint8 [..., %d, %d, 3] tensor on %s" % (OBS_SIDE, OBS_SIDE, self.device))
        P = self.num_policies
        if P > 1 and not (obs.dim() == 4 and obs.shape[0] % P == 0 or obs.dim() == 5 and obs.shape[1] == P):
            raise ValueError("a network of %d per-agent policies takes obs [B, %d, %d, %d, 3] or [B * %d, %d, %d, 3], not %s"
                             % (P, P, OBS_SIDE, OBS_SIDE, P, OBS_SIDE, OBS_SIDE, tuple(obs.shape)))
        obs = _aligned(obs)
        m = obs.numel() // (OBS_SIDE * OBS_SIDE * 3)
        if out is None:
            out = torch.empty((m, FEATURES), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib.ssd_policy_features(self._h, C.c_void_p(obs.data_ptr()), m, C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def initial_state(self, m):
        """Zero (h, c) for m agents, in the layout `forward` / `act` carry (tiled for the fused route, [m, cell_size] otherwise)."""
        shape = (self._groups(m), self.cell_size // 16, 128, 16) if self._fused_head else (m, self.cell_size)
        z = torch.zeros(shape, dtype=torch.float32, device=self.device)
        return z, z.clone()

    def state_rows(self, state, m):
        """Tiled state [G, 8, 128, 16] -> agent-major [m, cell_size] (a copy)."""
        if state.dim() == 2:
            return state[:m]
        self._groups(m)
        return _state_rows(state, m, self.num_policies)

    def state_from_rows(self, rows):
        """Agent-major [m, cell_size] -> tiled state [G, cell_size/16, 128, 16] (G = ceil(m/128), per policy for P > 1), zero padded."""
        self._groups(rows.shape[0])
        return _state_from_rows(rows, self.num_policies)

    def _check_state(self, h, c, m):
        if h.dim() != 4 or (h.shape[0] * 128 < m if self.num_policies == 1 else h.shape[0] != self._groups(m)):
            raise ValueError("the fused route carries (h, c) in the tiled layout of initial_state / state_from_rows")

    def _fused(self, obs, h, c, sample):
        """-> (logits, value, h', c', actions) of ssd_policy_lstm_heads; actions None unless `sample`."""
        s = self._heads(obs, None, h, c, _lib.ACT_SAMPLE if sample else None)
        return s.logits, s.value, s.h, s.c, s.actions

    def forward(self, obs, h, c):
        """-> (logits [M, A], value [M], h', c'), all float32; (h, c) in the layout of `initial_state`."""
        if not self._fused_head:
            return self.forward_unfused(obs, h, c)
        return self._fused(obs, h, c, sample=False)[:4]

    def forward_unfused(self, obs, h, c):
        """The same forward pass with library GEMMs: the trunk kernel, the gate GEMMs (cuBLAS, bf16 x bf16 -> fp32 accumulate), the
        one-pass cell update, the head GEMMs.  Any cell size that is a multiple of 8; (h, c) are [M, cell_size] here.  Shared
        weights only."""
        if self.num_policies > 1:
            raise ValueError("forward_unfused runs one shared network; a network per agent runs on the fused route (forward / act)")
        hd = self._head
        x16 = self.features(obs).to(torch.bfloat16)
        gates = torch.mm(x16, hd["lstm_w"]).addmm_(h.to(torch.bfloat16), hd["lstm_u"])   # bf16 [M, 4u], bias added in the cell kernel
        m, u = h.shape
        c_new, h_new = torch.empty_like(c), torch.empty_like(h)
        h16 = torch.empty((m, u), dtype=torch.bfloat16, device=self.device)
        p = lambda t: C.c_void_p(t.data_ptr())
        _lib.check(_lib.lib.ssd_policy_lstm_cell(p(gates), p(hd["lstm_b"]), p(_aligned(c)), p(c_new), p(h_new), p(h16), m, u, self._stream()))
        logits = torch.mm(h16, hd["logits_w"]).float() + hd["logits_b"]
        value = (torch.mm(h16, hd["value_w"]).float() + hd["value_b"]).squeeze(1)
        return logits, value, h_new, c_new

    def act(self, obs, h, c, generator=None):
        """Sample int8 actions [M] on the device for the next `BatchedSSDEnv.step`: inside the fused kernel (Philox streams,
        see `seed_sampling`), or with torch.multinomial (`generator`) on the unfused route."""
        if self._fused_head and generator is None:
            logits, value, h, c, a = self._fused(obs, h, c, sample=True)
            return a, value, h, c
        logits, value, h, c = self.forward(obs, h, c)
        a = torch.multinomial(torch.softmax(logits, dim=1), 1, generator=generator).squeeze(1).to(torch.int8)
        return a, value, h, c

    def policy_step(self, obs, h, c, mode="sample", actions=None, generator=None, features=None):
        """-> PolicyStep(actions, logp, entropy, logits, value, h', c') for the M agents of obs; (h, c) as for `forward`.

        mode 'sample': the action `act` draws -- the same Philox stream, and the call advances its counter, so `act` and
        `policy_step` calls may be interleaved; with `generator` (or on the unfused route) torch.multinomial as in `act`.
        mode 'greedy': the first argmax of the logits (np.argmax of them where they are finite).  mode 'given': `actions` (integers, M of them) are the caller's, e.g. a
        recorded trajectory or another policy's choice, and are returned as int8; logp is NaN where one is outside 0..A-1.
        logp and entropy are those of softmax(logits), computed from the float32 logits returned: on the fused route in the head
        kernel itself (ssd_policy_lstm_heads_dist), on the unfused route with torch.log_softmax.

        features: float32 [M, 32] on the device, what `features(obs)` returned for these observations (e.g. computed once
        for an MOANet / MOAPool of the same step).  The trunk is then not run and the head reads them; the result is bitwise that
        of the call without them.  obs may then be None (M is features.shape[0]); obs that is given is not read.  Fused route
        only (no `generator`)."""
        if features is not None:
            if not isinstance(features, torch.Tensor) or features.dim() != 2:
                raise ValueError("features must be a float32 [M, %d] tensor on %s" % (FEATURES, self.device))
            m = features.shape[0]
            if obs is not None and obs.numel() // (OBS_SIDE * OBS_SIDE * 3) != m:
                raise ValueError("features has %d rows, obs %d agents" % (m, obs.numel() // (OBS_SIDE * OBS_SIDE * 3)))
            if not self._fused_head or generator is not None:
                raise ValueError("features= runs the fused head kernel: cell_size 128, 1..15 outputs and no generator")
        else:
            m = obs.numel() // (OBS_SIDE * OBS_SIDE * 3)
        x = self._given_features(features, m)
        code, given = _step_mode(mode, actions, m, self.num_outputs, self.device)
        if not self._fused_head or (code == _lib.ACT_SAMPLE and generator is not None):
            return _torch_step(*self.forward(obs, h, c), code, given, generator)
        return self._heads(obs, None, h, c, code, given, dist=True, features=x)


class PolicyPool(_Policy):
    """K weight sets (1 <= K <= 255, each a dict as for ConvToFCNet) loaded once; every call takes `policy_ids`, a uint8 tensor
    on the device of shape obs.shape[:-3]: agent m is evaluated with weight_sets[policy_ids[m]], and the ids may differ from
    call to call.  An id >= K means "no pool policy": nothing is written for that agent (its rows of features, logits, value,
    h' and c' are left as they were in the output buffers, which `forward` allocates uninitialised) and `act` returns -1
    for it, so the caller drives it with its own code.  The recurrent state is the shared network's tiled layout
    [ceil(M/128), 8, 128, 16], independent of the ids; an agent that was skipped wants a fresh state row (state_from_rows)
    before it returns to a pool policy.  Needs the fused head (cell_size 128, 1..15 outputs).  The id values are checked on
    the device only (a host check would synchronise).  Calls on one pool must be ordered on one stream: the grouping of the
    agents by id uses scratch that belongs to the pool."""

    def __init__(self, weight_sets, device="cuda:0"):
        self.device = _cuda_device(device)
        sets = _weight_sets(weight_sets if isinstance(weight_sets, (list, tuple)) else [weight_sets])
        w = sets[0]
        self.num_policies = len(sets)
        self.cell_size = w["lstm_u"].shape[0] if "lstm_u" in w else 0
        self.num_outputs = w["logits_w"].shape[1] if "logits_w" in w else 0
        if self.cell_size != 128 or not 1 <= self.num_outputs <= 15:
            raise ValueError("a policy pool needs the fused head: cell_size 128 and 1..15 outputs (got %d, %d)" % (self.cell_size, self.num_outputs))
        w = {k: np.ascontiguousarray(np.stack([ws[k] for ws in sets])) for k in w}   # K consecutive arrays behind every pointer
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        names = ("conv_w", "conv_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "lstm_w", "lstm_u", "lstm_b", "logits_w", "logits_b", "value_w", "value_b")
        self._h = C.c_void_p()
        _lib.check(_lib.lib.ssd_policy_create_pool(VIEW_RADIUS, self.device.index, self.num_policies, self.cell_size, self.num_outputs,
                                                   *[ptr(w[k]) for k in names], C.byref(self._h)))

    def _ids(self, obs, policy_ids):
        if obs.dtype != torch.uint8 or obs.device != self.device or obs.dim() < 4 or tuple(obs.shape[-3:]) != (OBS_SIDE, OBS_SIDE, 3):
            raise ValueError("obs must be a uint8 [..., %d, %d, 3] tensor on %s" % (OBS_SIDE, OBS_SIDE, self.device))
        if not isinstance(policy_ids, torch.Tensor) or policy_ids.dtype != torch.uint8 or policy_ids.device != self.device \
                or tuple(policy_ids.shape) != tuple(obs.shape[:-3]):
            raise ValueError("policy_ids must be a uint8 tensor of shape %s on %s" % (tuple(obs.shape[:-3]), self.device))
        return _aligned(obs), policy_ids.contiguous()

    def features(self, obs, policy_ids, out=None):
        """uint8 [..., 15, 15, 3] + uint8 ids [...] on the device -> float32 [M, 32], agent-major."""
        obs, ids = self._ids(obs, policy_ids)
        m = ids.numel()
        if out is None:
            out = torch.empty((m, FEATURES), dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib.ssd_policy_pool_features(self._h, C.c_void_p(obs.data_ptr()), C.c_void_p(ids.data_ptr()), m,
                                                     C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def initial_state(self, m):
        """Zero (h, c) for m agents in the tiled layout [ceil(m/128), 8, 128, 16]."""
        z = torch.zeros(((m + 127) // 128, self.cell_size // 16, 128, 16), dtype=torch.float32, device=self.device)
        return z, z.clone()

    def state_rows(self, state, m):
        """Tiled state -> agent-major [m, 128] (a copy)."""
        return _state_rows(state, m, 1)

    def state_from_rows(self, rows):
        """Agent-major [m, 128] -> tiled state [ceil(m/128), 8, 128, 16], zero padded."""
        return _state_from_rows(rows, 1)

    def _check_state(self, h, c, m):
        if h.dim() != 4 or h.shape[0] * 128 < m or h.shape != c.shape:
            raise ValueError("(h, c) must be in the tiled layout of initial_state / state_from_rows")

    def _run(self, obs, policy_ids, h, c, sample):
        """-> (logits, value, h', c', actions) of ssd_policy_pool_lstm_heads; actions None unless `sample`."""
        s = self._heads(*self._ids(obs, policy_ids), h, c, _lib.ACT_SAMPLE if sample else None)
        return s.logits, s.value, s.h, s.c, s.actions

    def forward(self, obs, policy_ids, h, c):
        """-> (logits [M, A], value [M], h', c'), all float32; rows of skipped agents are not written."""
        return self._run(obs, policy_ids, h, c, sample=False)[:4]

    def act(self, obs, policy_ids, h, c):
        """Sample int8 actions [M] on the device (Philox streams, see `seed_sampling`); -1 for skipped agents."""
        logits, value, h, c, a = self._run(obs, policy_ids, h, c, sample=True)
        return a, value, h, c

    def policy_step(self, obs, policy_ids, h, c, mode="sample", actions=None, features=None):
        """-> PolicyStep(actions, logp, entropy, logits, value, h', c'), as ConvToFCNet.policy_step on the pool's kernels:
        'sample' draws what `act` draws and advances the same counter, 'greedy' takes the first argmax of the logits, 'given'
        scores the caller's `actions` (returned as int8).  Skipped agents (id >= K) get action -1 in 'sample' and 'greedy'; their
        rows of logp and entropy, like those of logits, value, h' and c', are not written.

        features: float32 [M, 32] on the device, what `features(obs, policy_ids)` returned (e.g. computed once for an MOAPool
        of the same step).  The trunk is then not run; the head still groups the agents by `policy_ids` itself, and the result is
        bitwise that of the call without features.  obs may then be None (policy_ids is a uint8 tensor of M elements on the
        device); obs that is given is checked against policy_ids but not read."""
        if features is None or obs is not None:
            obs, ids = self._ids(obs, policy_ids)
        else:
            if not isinstance(policy_ids, torch.Tensor) or policy_ids.dtype != torch.uint8 or policy_ids.device != self.device:
                raise ValueError("policy_ids must be a uint8 tensor on %s" % (self.device,))
            ids = policy_ids.contiguous()
        x = self._given_features(features, ids.numel())
        code, given = _step_mode(mode, actions, ids.numel(), self.num_outputs, self.device)
        return self._heads(obs, ids, h, c, code, given, dist=True, features=x)


MOAStep = collections.namedtuple("MOAStep", "pred influence influence_per_agent h c counterfactual")
MOAStep.__doc__ = """One step of the model of other agents for M agents: pred float32 [M, N-1, A] (logits of the others' actions at the
actual joint action), influence float32 [M], influence_per_agent float32 [M, N-1], the next state (h, c), and counterfactual
float32 [M, A, N-1, A] (the logits with the own action replaced by each a') or None."""

_DIVERGENCES = {"kl": _lib.DIV_KL, "jsd": _lib.DIV_JSD}


def random_moa_weights(num_agents, num_actions, seed=0, cell_size=128):
    """Random-init MOA weights (glorot, unit forget bias) in the Keras layouts `MOANet` takes."""
    rng = np.random.RandomState(seed)
    glorot = lambda shape: rng.uniform(-1, 1, size=shape).astype(np.float32) * np.float32(np.sqrt(6.0 / sum(shape)))
    u, k_in, n_out = cell_size, FEATURES + num_agents * num_actions, (num_agents - 1) * num_actions
    return {"moa_lstm_w": glorot((k_in, 4 * u)), "moa_lstm_u": glorot((u, 4 * u)),
            "moa_lstm_b": np.concatenate([np.zeros(u), np.ones(u), np.zeros(2 * u)]).astype(np.float32),
            "moa_logits_w": glorot((u, n_out)), "moa_logits_b": (0.1 * rng.randn(n_out)).astype(np.float32)}


class MOANet(_Handle):
    """Model of other agents of the causal-influence models (models/moa_model.py MOA_LSTM) and the social-influence reward
    (common_funcs.py compute_influence_reward), forward only, in one fused kernel (`ssd_moa_step`).

    For agent m = b * N + i the input is [x | onehot(a_{b,i}) | onehot(a_{b,j}) for j != i in increasing j], x the 32 trunk
    features (ConvToFCNet.features); LSTM(128) then Dense((N-1) * A).  `weights` is one dict (shared by all agents) or a list of
    N dicts (agent i uses weights[i], as ConvToFCNet([w_0, ..., w_{N-1}])), with keys moa_lstm_w [32 + N A, 512], moa_lstm_u
    [128, 512], moa_lstm_b [512], moa_logits_w [128, (N-1) A], moa_logits_b [(N-1) A].  The recurrent state has the tiled layout
    of ConvToFCNet (grouped per weight set for a list of N)."""
    _destroy = "ssd_moa_destroy"

    def __init__(self, weights, num_agents, device="cuda:0"):
        sets = list(weights) if isinstance(weights, (list, tuple)) else [weights]
        n = int(num_agents)
        if len(sets) not in (1, n):
            raise ValueError("weights is one dict or a list of num_agents = %d dicts, not %d" % (n, len(sets)))
        self._create(sets, n, device, _lib.lib.ssd_moa_create)
        self._state_sets = self.num_policies   # the tiled state is grouped per weight set

    def _create(self, sets, n, device, create):
        """Checks the weight sets' names and shapes and loads them with `create` (ssd_moa_create[_pool])."""
        self.device = _cuda_device(device)
        self.num_agents = n
        sets = [{k: np.ascontiguousarray(ws[k], dtype=np.float32) for k in
                 ("moa_lstm_w", "moa_lstm_u", "moa_lstm_b", "moa_logits_w", "moa_logits_b")} for ws in sets]
        w = sets[0]
        self.num_policies = P = len(sets)
        self.cell_size = w["moa_lstm_u"].shape[0]
        k_in = w["moa_lstm_w"].shape[0] - FEATURES
        self.num_actions = A = k_in // n if n >= 2 else 0
        shapes = {"moa_lstm_w": (FEATURES + n * A, 4 * self.cell_size), "moa_lstm_u": (self.cell_size, 4 * self.cell_size),
                  "moa_lstm_b": (4 * self.cell_size,), "moa_logits_w": (self.cell_size, (n - 1) * A), "moa_logits_b": ((n - 1) * A,)}
        for q, ws in enumerate(sets):
            for k, shape in shapes.items():
                if ws[k].shape != shape:
                    raise ValueError("weights[%d][%r] has shape %s, expected %s" % (q, k, ws[k].shape, shape))
        if self.cell_size != 128 or k_in != n * A:
            raise ValueError("the MOA kernel is built for cell_size 128 and moa_lstm_w [32 + N A, 512]")
        w = {k: np.ascontiguousarray(np.stack([ws[k] for ws in sets])) for k in w}   # P consecutive arrays behind every pointer
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        self._h = C.c_void_p()
        _lib.check(create(self.device.index, P, n, A, ptr(w["moa_lstm_w"]), ptr(w["moa_lstm_u"]), ptr(w["moa_lstm_b"]),
                          ptr(w["moa_logits_w"]), ptr(w["moa_logits_b"]), C.byref(self._h)))

    def _groups(self, m):
        n, P = self.num_agents, self._state_sets
        if m % n:
            raise ValueError("%d agents are not a whole number of envs of %d agents" % (m, n))
        return P * ((m // P + 127) // 128)

    def initial_state(self, m):
        """Zero (h, c) for m agents in the tiled layout [G, 8, 128, 16]."""
        z = torch.zeros((self._groups(m), self.cell_size // 16, 128, 16), dtype=torch.float32, device=self.device)
        return z, z.clone()

    def state_rows(self, state, m):
        """Tiled state -> agent-major [m, 128] (a copy)."""
        self._groups(m)
        return _state_rows(state, m, self._state_sets)

    def state_from_rows(self, rows):
        """Agent-major [m, 128] -> tiled state, zero padded."""
        self._groups(rows.shape[0])
        return _state_from_rows(rows, self._state_sets)

    def step(self, features, joint_actions, policy_logits, h, c, divergence="kl", clip=float("inf"), counterfactuals=False):
        """-> MOAStep for the M agents of features [M, 32] (float32, ConvToFCNet.features of the step's observations).

        joint_actions: the actions the step took, an integer tensor of M elements ([B, N] or [M], agent-major); a value outside
        0..A-1 is a zero one-hot input and makes influence NaN for every agent of its env.  policy_logits [M, A]: the policy's
        logits of that step (PolicyStep.logits).  divergence 'kl' or 'jsd'; influence = clamp(sum over the others, -clip, clip).
        counterfactuals=True also returns the [M, A, N-1, A] logits of every own action."""
        return self._step(features, None, joint_actions, policy_logits, h, c, divergence, clip, counterfactuals)

    def _step(self, features, ids, joint_actions, policy_logits, h, c, divergence, clip, counterfactuals):
        """ssd_moa_step, or ssd_moa_pool_step on `ids` (None: the former)."""
        if divergence not in _DIVERGENCES:
            raise ValueError("divergence must be 'kl' or 'jsd', not %r" % (divergence,))
        clip = float(clip)
        if not clip >= 0.0:
            raise ValueError("clip must be >= 0 (inf: no clamp), not %r" % (clip,))
        n, A = self.num_agents, self.num_actions
        if not isinstance(features, torch.Tensor) or features.dtype != torch.float32 or features.device != self.device \
                or features.dim() != 2 or features.shape[1] != FEATURES:
            raise ValueError("features must be a float32 [M, %d] tensor on %s" % (FEATURES, self.device))
        m = features.shape[0]
        g = self._groups(m)
        _, given = _step_mode("given", joint_actions, m, A, self.device)
        if ids is not None and (not isinstance(ids, torch.Tensor) or ids.dtype != torch.uint8 or ids.device != self.device
                                or tuple(ids.shape) not in ((m,), (m // n, n))):
            raise ValueError("policy_ids must be a uint8 tensor of shape [%d, %d] or [%d] on %s" % (m // n, n, m, self.device))
        if not isinstance(policy_logits, torch.Tensor) or policy_logits.dtype != torch.float32 or policy_logits.device != self.device \
                or tuple(policy_logits.shape) != (m, A):
            raise ValueError("policy_logits must be a float32 [%d, %d] tensor on %s" % (m, A, self.device))
        if tuple(h.shape) != (g, self.cell_size // 16, 128, 16) or h.shape != c.shape:
            raise ValueError("(h, c) must be in the tiled layout of initial_state / state_from_rows")
        x, h, c, pl = _aligned(features), _aligned(h), _aligned(c), policy_logits.contiguous()
        h_new, c_new = torch.empty_like(h), torch.empty_like(c)
        pred = torch.empty((m, n - 1, A), dtype=torch.float32, device=self.device)
        cf = torch.empty((m, A, n - 1, A), dtype=torch.float32, device=self.device) if counterfactuals else None
        ipa = torch.empty((m, n - 1), dtype=torch.float32, device=self.device)
        infl = torch.empty((m,), dtype=torch.float32, device=self.device)
        p = lambda t: C.c_void_p(t.data_ptr() if t is not None else None)
        io = (p(pl), p(h), p(c), p(h_new), p(c_new), p(pred), p(cf), p(ipa), p(infl), m, _DIVERGENCES[divergence], clip, self._stream())
        if ids is None:
            _lib.check(_lib.lib.ssd_moa_step(self._h, p(x), p(given), *io))
        else:
            _lib.check(_lib.lib.ssd_moa_pool_step(self._h, p(x), p(ids.contiguous()), p(given), *io))
        return MOAStep(pred, infl, ipa, h_new, c_new, cf)


class MOAPool(MOANet):
    """K MOA weight sets (1 <= K <= 255, each a dict as for MOANet) loaded once; every `step` takes `policy_ids`, a uint8
    tensor on the device of M elements ([B, N] or [M], agent-major): agent m is evaluated with weight_sets[policy_ids[m]], and
    the ids may differ from call to call -- typically the tensor the PolicyPool call of the same step took (K seeds of an MOA
    experiment on one GPU, cross-play teams).  An id >= K means "no MOA for this agent": nothing is written for it (its rows
    of pred, influence, influence_per_agent, counterfactual, h' and c' are left as they were in the output buffers, which
    `step` allocates uninitialised) and its row of policy_logits is not read; its action still enters the other agents'
    inputs, and an action outside 0..A-1 still makes influence NaN for its whole env.  The recurrent state is the shared
    network's tiled layout [ceil(M/128), 8, 128, 16], independent of the ids; an agent that was skipped wants a fresh state row
    (state_from_rows) before it returns to a pool MOA.  The id values are checked on the device only.  Calls on one MOA pool
    must be ordered on one stream: the grouping of the agents by id uses scratch that belongs to the pool."""

    def __init__(self, weight_sets, num_agents, device="cuda:0"):
        sets = list(weight_sets) if isinstance(weight_sets, (list, tuple)) else [weight_sets]
        if not sets:
            raise ValueError("no weight sets")
        self._create(sets, int(num_agents), device, _lib.lib.ssd_moa_create_pool)
        self._state_sets = 1   # agent-major, whatever the ids

    def step(self, features, policy_ids, joint_actions, policy_logits, h, c, divergence="kl", clip=float("inf"), counterfactuals=False):
        """-> MOAStep as MOANet.step, agent m evaluated with weight set policy_ids[m] (ssd_moa_pool_step); rows of skipped agents
        (id >= K) are not written."""
        return self._step(features, policy_ids, joint_actions, policy_logits, h, c, divergence, clip, counterfactuals)
