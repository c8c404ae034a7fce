"""CPU oracle for the MARLClassification hot path (TEST INFRASTRUCTURE ONLY).

This module is a functional, CPU-only restatement of the reference algorithm
(Ipsedo/MARLClassification): the batched multi-agent episode rollout and the
actor-critic loss.  It exists to CHECK the CUDA product path; nothing under
``marlclassification_b200/`` may import it.  Only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` use it.

Pinning: the reference holds no golden vectors of its own (its tests check
shapes/bounds only), so this restatement is pinned against outputs of the
reference itself, generated in the build container by ``oracle/make_golden.py``
(imports ``/root/reference`` unmodified, records every random draw) and
committed under ``tests/golden/``.  ``tests/test_oracle_golden.py`` holds the
oracle to those fixtures (bit-exact positions/patches, <=1e-5 on floats).

The arithmetic of the reference lives in third-party torch (ATen); the oracle
uses the same ATen CPU primitives (``F.linear``, ``F.conv2d``, ``F.group_norm``,
``F.layer_norm``) so fp32 rounding matches the reference closely.

Parameters are passed as a dict keyed by the reference's ``state_dict`` names
(prefix ``_ModelsWrapper__``), so reference checkpoints plug in directly.

Every function cites the reference file:line it follows
(paths relative to ``marl_classification/``).
"""

from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

P = "_ModelsWrapper__"
CNN = P + "map_obs._Generic2dCnnModule__layers."
LSTM_B = P + "belief_unit._LSTMCellWrapper__lstm."
LSTM_A = P + "action_unit._LSTMCellWrapper__lstm."

# (in,out) channels + GroupNorm groups per conv block -- networks/vision.py:59-113
CNN_SPECS = {
    "mnist": ([(1, 8), (8, 16)], [2, 4], True),
    "resisc45": ([(3, 16), (16, 32), (32, 64)], [2, 4, 8], False),
    "skin_cancer": ([(3, 16), (16, 32), (32, 64)], [2, 4, 8], False),
    "aid": ([(3, 16), (16, 32), (32, 64), (64, 128)], [2, 4, 8, 16], False),
    "worldstrat": (
        [(3, 16), (16, 32), (32, 64), (64, 128), (128, 256)],
        [2, 4, 8, 16, 32],
        False,
    ),
}


@dataclass
class OracleConfig:
    """Mirror of the fields of config.py:18-31 that the path consumes."""

    ft_extr: str
    f: int
    n_b: int
    n_a: int
    n_m: int
    n_m_o: int
    n_d: int
    nb_class: int
    nl_b: int
    nl_a: int
    actions: List[List[int]] = field(
        default_factory=lambda: [[1, 0], [-1, 0], [0, 1], [0, -1]]
    )

    @property
    def cnn_layers(self) -> List[Tuple[int, int]]:
        return CNN_SPECS[self.ft_extr][0]

    @property
    def cnn_groups(self) -> List[int]:
        return CNN_SPECS[self.ft_extr][1]

    @property
    def ch0_only(self) -> bool:
        return CNN_SPECS[self.ft_extr][2]

    @property
    def cnn_out(self) -> int:
        # vision.py:41-45
        w = self.f
        for _ in self.cnn_layers:
            w = (w - 3 + 2) // 2 + 1
        return self.cnn_layers[-1][1] * w * w


# --------------------------------------------------------------------------
# Environment (core/environment.py)
# --------------------------------------------------------------------------
def to_tensor_batch(u8_hwc: torch.Tensor) -> torch.Tensor:
    """torchvision ``ToTensor`` on a batch of decoded images (registry.py:56-57 applied per sample by
    the DataLoader of train.py:91-107): u8[B,H,W,C] -> f32[B,C,H,W] = permute, cast, true-divide by 255."""
    return u8_hwc.permute(0, 3, 1, 2).contiguous().to(torch.float32).div(255)


def observation_masked(img: torch.Tensor, pos: torch.Tensor, f: int) -> torch.Tensor:
    """The reference's own algorithm, environment.py:96-126: per-dim window
    masks, AND-ed and broadcast over [Na,B,C,H,W], then ``masked_select``.
    Used as the timed CPU baseline (this IS what the reference executes)."""
    B, C = img.shape[0], img.shape[1]
    sizes = list(img.shape[2:])
    Na = pos.shape[0]
    nd = len(sizes)
    full = None
    for d, s in enumerate(sizes):
        ar = torch.arange(s, device=pos.device).view(1, 1, s)
        lo = pos[:, :, d, None]
        m = (lo <= ar) & (ar < lo + f)
        shape = [Na, B] + [1] * nd
        shape[2 + d] = s
        m = m.view(shape)
        full = m if full is None else (full & m)
    full = full.unsqueeze(2)
    return img.unsqueeze(0).masked_select(full).view(Na, B, C, *([f] * nd))


def observation(img: torch.Tensor, pos: torch.Tensor, f: int) -> torch.Tensor:
    """Closed form of environment.py:96-126 for 2-D images:
    obs[a,b,c,i,j] = img[b,c,pos[a,b,0]+i,pos[a,b,1]+j] (pure data movement)."""
    Na, B, _ = pos.shape
    ar = torch.arange(f, device=pos.device)
    rows = pos[:, :, 0, None] + ar  # [Na,B,f]
    cols = pos[:, :, 1, None] + ar
    b_idx = torch.arange(B, device=pos.device).view(1, B, 1, 1, 1)
    c_idx = torch.arange(img.shape[1], device=pos.device).view(1, 1, -1, 1, 1)
    return img[b_idx, c_idx, rows[:, :, None, :, None], cols[:, :, None, None, :]]


def transition(
    pos: torch.Tensor, moves: torch.Tensor, f: int, sizes: Sequence[int]
) -> torch.Tensor:
    """environment.py:128-150 as integer arithmetic: the move is applied only
    if EVERY dim stays inside (0 <= p+m and p+m+f < S, strict), else the agent
    stays where it is.  The reference does this in fp32 and casts back; values
    are small integers so the two agree exactly."""
    new = pos + moves
    ok = torch.ones(pos.shape[:2], dtype=torch.bool, device=pos.device)
    for d, s in enumerate(sizes):
        ok &= (new[:, :, d] >= 0) & (new[:, :, d] + f < s)
    return torch.where(ok.unsqueeze(-1), new, pos)


def normalized_positions(pos: torch.Tensor, sizes: Sequence[int], dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """environment.py:74-81: float(pos) / float(size), true fp32 division (what the reference and the
    engine compute, whatever precision the networks run in), returned as ``dtype``."""
    s = torch.tensor([[list(sizes)]], dtype=torch.float32, device=pos.device)
    return (pos.to(torch.float32) / s).to(dtype)


# --------------------------------------------------------------------------
# Networks (networks/*.py)
# --------------------------------------------------------------------------
def cnn_forward(p: Dict[str, torch.Tensor], cfg: OracleConfig, x: torch.Tensor) -> torch.Tensor:
    """vision.py:23-77: k x [conv3x3 s2 p1 -> GroupNorm(eps 1e-5) -> SiLU],
    flatten C-major.  MnistCnn keeps channel 0 only (vision.py:64)."""
    if cfg.ch0_only:
        x = x[:, 0:1]
    for li, g in enumerate(cfg.cnn_groups):
        cw, cb = p[f"{CNN}{3 * li}.weight"], p[f"{CNN}{3 * li}.bias"]
        gw, gb = p[f"{CNN}{3 * li + 1}.weight"], p[f"{CNN}{3 * li + 1}.bias"]
        x = F.conv2d(x, cw, cb, stride=2, padding=1)
        x = F.group_norm(x, g, gw, gb, eps=1e-5)
        x = F.silu(x)
    return x.flatten(1)


def lin_ln_silu(p, name: str, i: int, x: torch.Tensor) -> torch.Tensor:
    """Linear -> LayerNorm(eps 1e-5) -> SiLU: the block shared by message.py:
    26-33, state.py:13-17, policy.py:11-14, prediction.py:10-13."""
    w, b = p[f"{P}{name}.{i}.weight"], p[f"{P}{name}.{i}.bias"]
    g, be = p[f"{P}{name}.{i + 1}.weight"], p[f"{P}{name}.{i + 1}.bias"]
    y = F.linear(x, w, b)
    return F.silu(F.layer_norm(y, (y.shape[-1],), g, be, 1e-5))


def aggregate_messages(msg: torch.Tensor) -> torch.Tensor:
    """message.py:5-17: mean over the OTHER agents; zeros if alone."""
    na = msg.shape[0]
    if na == 1:
        return torch.zeros_like(msg)
    return (msg.sum(0) - msg) / (na - 1)


def lstm_cell(p, prefix: str, u, h, c):
    """recurrent.py:20-35 -> nn.LSTMCell: gates i,f,g,o;
    c' = s(f)c + s(i)tanh(g); h' = s(o)tanh(c')."""
    g = F.linear(u, p[prefix + "weight_ih"], p[prefix + "bias_ih"]) + F.linear(
        h, p[prefix + "weight_hh"], p[prefix + "bias_hh"]
    )
    i, f_, gg, o = g.chunk(4, dim=-1)
    c2 = torch.sigmoid(f_) * c + torch.sigmoid(i) * torch.tanh(gg)
    h2 = torch.sigmoid(o) * torch.tanh(c2)
    return h2, c2


def step_forward(p, cfg: OracleConfig, patch, msg, npos, hid, record: Optional[dict] = None):
    """models.py:78-138, one step of every network for all Na*Nb rows.
    patch [Na,Nb,C,f,f]; msg [Na,Nb,n_m]; npos [Na,Nb,2];
    hid = (h, c, h^, c^).  Returns probs, values, preds, new_msg, new_hid.
    ``record`` (a dict) receives the LSTM input u [Na*Nb, Kin]."""
    na, nb = patch.shape[:2]
    h, c, hc, cc = hid
    b_t = cnn_forward(p, cfg, patch.flatten(0, 1)).view(na, nb, -1)
    d_bar = lin_ln_silu(p, "decode_msg", 3, lin_ln_silu(p, "decode_msg", 0, aggregate_messages(msg)))
    lam = lin_ln_silu(p, "map_pos", 0, npos)
    u = torch.cat((b_t, d_bar, lam), dim=2).flatten(0, 1)
    if record is not None:
        record["u"] = u
    h2, c2 = lstm_cell(p, LSTM_B, u, h.flatten(0, 1), c.flatten(0, 1))
    h2, c2 = h2.view(na, nb, -1), c2.view(na, nb, -1)
    new_msg = lin_ln_silu(p, "encode_msg", 3, lin_ln_silu(p, "encode_msg", 0, h2))
    hc2, cc2 = lstm_cell(p, LSTM_A, u, hc.flatten(0, 1), cc.flatten(0, 1))
    hc2, cc2 = hc2.view(na, nb, -1), cc2.view(na, nb, -1)
    # policy.py:11-17 (softmax probabilities) and 22-28 (critic, flatten(-2,-1))
    pol = lin_ln_silu(p, "policy", 0, hc2)
    probs = F.softmax(F.linear(pol, p[P + "policy.3.weight"], p[P + "policy.3.bias"]), dim=-1)
    cri = lin_ln_silu(p, "critic", 0, hc2)
    values = F.linear(cri, p[P + "critic.3.weight"], p[P + "critic.3.bias"]).squeeze(-1)
    # prediction.py:10-15 (raw logits)
    prd = lin_ln_silu(p, "predict", 0, h2)
    preds = F.linear(prd, p[P + "predict.3.weight"], p[P + "predict.3.bias"])
    return probs, values, preds, new_msg, (h2, c2, hc2, cc2)


@dataclass
class Rollout:
    step_preds: torch.Tensor  # [T,Na,Nb,Nc]
    step_log_probas: torch.Tensor  # [T,Na,Nb]
    step_values: torch.Tensor  # [T,Na,Nb]
    step_pos: torch.Tensor  # [T,Na,Nb,2] int64, AFTER each move
    step_probs: torch.Tensor  # [T,Na,Nb,nA] (extra: for sampling tests)
    patches: List[torch.Tensor]  # T+1 observations (o_0 .. o_T)
    actions: torch.Tensor  # [T,Na,Nb] int64
    final_hidden: Tuple[torch.Tensor, ...]
    # per-step values (rollout(record=True)): for each step t a dict with the LSTM input "u" [Na*Nb, Kin]
    # (CNN features | decoded message | position features), the new state "h", "c", "h_caret", "c_caret"
    # [Na,Nb,n] and the message "msg" [Na,Nb,n_m] it emits
    steps: Optional[List[Dict[str, torch.Tensor]]] = None


def rollout(
    p: Dict[str, torch.Tensor],
    cfg: OracleConfig,
    img: torch.Tensor,
    pos0: torch.Tensor,
    hidden0: Sequence[torch.Tensor],
    actions: Optional[torch.Tensor],
    nb_step: int,
    *,
    faithful_gather: bool = False,
    generator: Optional[torch.Generator] = None,
    record: bool = False,
) -> Rollout:
    """episode.py:32-82 + agent.py:40-68 + environment.py:23-68 with the three
    random sites injected: initial positions (environment.py:33-43), initial
    recurrent state (models.py:148-159) and the per-step action sample
    (agent.py:53-55).  ``actions=None`` samples with torch.multinomial.  Runs in the dtype of ``img``
    (fp64 parameters, image and state give an fp64 reference); ``record`` keeps the per-step values
    in ``Rollout.steps``."""
    sizes = list(img.shape[2:])
    gather = observation_masked if faithful_gather else observation
    table = torch.tensor(cfg.actions, dtype=torch.long, device=img.device)
    na, nb = pos0.shape[:2]
    pos = pos0.clone()
    hid = tuple(hidden0)
    msg = torch.zeros(na, nb, cfg.n_m, dtype=img.dtype, device=img.device)
    obs = gather(img, pos, cfg.f)
    patches = [obs]
    preds_l, logp_l, val_l, pos_l, prob_l, act_l = [], [], [], [], [], []
    steps = [] if record else None
    for t in range(nb_step):
        npos = normalized_positions(pos, sizes, img.dtype)
        rec = {} if record else None
        probs, values, preds, msg, hid = step_forward(p, cfg, obs, msg, npos, hid, rec)
        if record:
            rec.update(h=hid[0], c=hid[1], h_caret=hid[2], c_caret=hid[3], msg=msg)
            steps.append(rec)
        if actions is None:
            a = torch.multinomial(probs.flatten(0, 1), 1, True, generator=generator).view(na, nb)
        else:
            a = actions[t]
        logp = torch.gather(probs, -1, a.unsqueeze(-1)).squeeze(-1).log()
        pos = transition(pos, table[a], cfg.f, sizes)
        obs = gather(img, pos, cfg.f)
        patches.append(obs)
        preds_l.append(preds)
        logp_l.append(logp)
        val_l.append(values)
        pos_l.append(pos)
        prob_l.append(probs)
        act_l.append(a)
    return Rollout(
        torch.stack(preds_l),
        torch.stack(logp_l),
        torch.stack(val_l),
        torch.stack(pos_l),
        torch.stack(prob_l),
        patches,
        torch.stack(act_l),
        hid,
        steps,
    )


# --------------------------------------------------------------------------
# Loss (training/functions.py, training/trainer.py:73-111)
# --------------------------------------------------------------------------
def classification_rewards(step_preds: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
    """functions.py:7-32: (ln Nc - CE(pred[t,a,b], y_b)) / ln Nc."""
    T, na, nb, nc = step_preds.shape
    ce = F.cross_entropy(
        step_preds.reshape(-1, nc), targets.view(1, 1, nb).expand(T, na, nb).reshape(-1), reduction="none"
    ).view(T, na, nb)
    return (math.log(nc) - ce) / math.log(nc)


def discounted_returns(rewards: torch.Tensor, gamma: float) -> torch.Tensor:
    """functions.py:35-51: flip-cumsum-flip of r*gamma^t, divided by gamma^t (0/0 = NaN from t = 1 on at
    gamma = 0, as in the reference)."""
    T = rewards.shape[0]
    g = (gamma ** torch.arange(T, dtype=rewards.dtype, device=rewards.device)).view(T, *([1] * (rewards.dim() - 1)))
    return (rewards * g).flip(0).cumsum(0).flip(0) / g


def standardize(x: torch.Tensor, eps: float = 1e-8) -> torch.Tensor:
    """functions.py:54-55: global mean / unbiased std."""
    return (x - x.mean()) / (x.std() + eps)


@dataclass
class LossParts:
    loss: torch.Tensor
    path: torch.Tensor  # path_loss.sum(0).mean()
    error: torch.Tensor  # error.mean()
    actor: torch.Tensor  # actor_loss.sum(0).mean()
    critic: torch.Tensor  # critic_loss.sum(0).mean()


def a2c_loss(step_preds, step_logp, step_values, targets, gamma: float, adv_stats=None) -> LossParts:
    """trainer.py:75-111 (+ the meter reads at 119-122).  ``adv_stats=(mean, std)`` overrides
    the statistics of ``standardize`` (data-parallel shards use the GLOBAL batch's)."""
    T, na, nb, nc = step_preds.shape
    vote = step_preds.mean(dim=1).reshape(T * nb, nc)
    error = F.cross_entropy(vote, targets.repeat(T), reduction="none").view(T, 1, nb)
    returns = discounted_returns(classification_rewards(step_preds, targets), gamma)
    raw_adv = returns - step_values
    adv = standardize(raw_adv) if adv_stats is None else (raw_adv - adv_stats[0]) / (adv_stats[1] + 1e-8)
    path = -step_logp * adv.detach()
    actor = path + error
    critic = F.smooth_l1_loss(step_values, returns.detach(), reduction="none")
    loss = (actor + critic).sum(0).mean()
    return LossParts(loss, path.sum(0).mean(), error.mean(), actor.sum(0).mean(), critic.sum(0).mean())


def loss_and_grads(p, cfg, img, targets, pos0, hidden0, actions, nb_step, gamma):
    """One train iteration's numbers: rollout -> loss -> autograd grads
    (trainer.py:73-115).  Returns (Rollout, LossParts, {name: grad})."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
    ro = rollout(leaf, cfg, img, pos0, hidden0, actions, nb_step)
    parts = a2c_loss(ro.step_preds, ro.step_log_probas, ro.step_values, targets, gamma)
    names = list(leaf)
    grads = torch.autograd.grad(parts.loss, [leaf[k] for k in names], allow_unused=True)
    return ro, parts, {k: (g if g is not None else torch.zeros_like(leaf[k])) for k, g in zip(names, grads)}


def train_steps(p, cfg, img, targets, pos0, hidden0, actions, nb_step, gamma, lr, n_steps, parts_out=None):
    """``n_steps`` optimisation steps of trainer.py:66-116 on ONE batch with the same injected draws
    every step: rollout -> loss -> ``backward`` -> ``th.optim.Adam(lr)`` (trainer.py:33 defaults:
    betas (0.9, 0.999), eps 1e-8).  Returns (final params, [loss per step]); a list ``parts_out``
    receives each step's [loss, path, error, actor, critic]."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
    opt = torch.optim.Adam(list(leaf.values()), lr=lr)
    losses = []
    for _ in range(n_steps):
        ro = rollout(leaf, cfg, img, pos0, hidden0, actions, nb_step)
        parts = a2c_loss(ro.step_preds, ro.step_log_probas, ro.step_values, targets, gamma)
        opt.zero_grad()
        parts.loss.backward()
        opt.step()
        losses.append(float(parts.loss.detach()))
        if parts_out is not None:
            parts_out.append([float(getattr(parts, k).detach()) for k in ("loss", "path", "error", "actor", "critic")])
    return {k: v.detach() for k, v in leaf.items()}, losses


def confusion_matrix(batches, nb_class: int, window_size=None):
    """metrics.py:25-108: the meter keeps the last ``window_size`` (argmax prediction, target) batches
    (all when None), rebuilds the matrix from their concatenation with ``bincount`` (rows = true
    class), and derives per-class precision (diag / column sum) and recall (diag / row sum), 0 where
    the denominator is 0.  ``batches``: iterable of (y_proba [B, Nc], y_true [B]).
    Returns (conf_mat int64 [Nc, Nc], precision f32 [Nc], recall f32 [Nc])."""
    kept = []
    for y_proba, y_true in batches:
        if window_size is not None and len(kept) >= window_size:  # metrics.py:38-44
            kept.pop(0)
        kept.append((y_proba.argmax(dim=1), y_true))
    y_pred = torch.cat([a for a, _ in kept])
    y_true = torch.cat([b for _, b in kept])
    cm = torch.bincount(y_true * nb_class + y_pred, minlength=nb_class**2).reshape(nb_class, nb_class)
    diag = torch.diagonal(cm, 0)

    def ratio(tot):
        out = torch.zeros(nb_class)
        mask = tot != 0
        out[mask] = diag[mask] / tot[mask]
        return out

    return cm, ratio(cm.sum(dim=0)), ratio(cm.sum(dim=1))


def init_params(cfg: OracleConfig, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Random parameters with the reference's shapes and init distribution
    (init.py:6-29: orthogonal(gain sqrt2) weights, zero biases, norm affine
    (1,0)) -- for tests that need a weight set without the reference around.
    Biases / affines are then perturbed so they are exercised by parity tests."""
    g = torch.Generator().manual_seed(seed)
    p: Dict[str, torch.Tensor] = {}

    def ortho(*shape):
        w = torch.empty(*shape)
        flat = torch.randn(shape[0], int(math.prod(shape[1:])), generator=g)
        if flat.shape[0] < flat.shape[1]:
            q, r = torch.linalg.qr(flat.t())
            q = (q * torch.sign(torch.diagonal(r))).t()
        else:
            q, r = torch.linalg.qr(flat)
            q = q * torch.sign(torch.diagonal(r))
        w.copy_(q.reshape(shape) * math.sqrt(2.0))
        return w

    def small(n):
        return 0.1 * torch.randn(n, generator=g)

    for li, (ci, co) in enumerate(cfg.cnn_layers):
        p[f"{CNN}{3 * li}.weight"] = ortho(co, ci, 3, 3)
        p[f"{CNN}{3 * li}.bias"] = small(co)
        p[f"{CNN}{3 * li + 1}.weight"] = 1 + small(co)
        p[f"{CNN}{3 * li + 1}.bias"] = small(co)

    def lin(name, i, n_in, n_out, norm=True):
        p[f"{P}{name}.{i}.weight"] = ortho(n_out, n_in)
        p[f"{P}{name}.{i}.bias"] = small(n_out)
        if norm:
            p[f"{P}{name}.{i + 1}.weight"] = 1 + small(n_out)
            p[f"{P}{name}.{i + 1}.bias"] = small(n_out)

    k_in = cfg.cnn_out + cfg.n_m_o + cfg.n_d
    lin("map_pos", 0, 2, cfg.n_d)
    lin("encode_msg", 0, cfg.n_b, 2 * cfg.n_m)
    lin("encode_msg", 3, 2 * cfg.n_m, cfg.n_m)
    lin("decode_msg", 0, cfg.n_m, 2 * cfg.n_m)
    lin("decode_msg", 3, 2 * cfg.n_m, cfg.n_m_o)
    for pre, n in ((LSTM_B, cfg.n_b), (LSTM_A, cfg.n_a)):
        p[pre + "weight_ih"] = ortho(4 * n, k_in)
        p[pre + "weight_hh"] = ortho(4 * n, n)
        p[pre + "bias_ih"] = small(4 * n)
        p[pre + "bias_hh"] = small(4 * n)
    lin("policy", 0, cfg.n_a, cfg.nl_a)
    lin("policy", 3, cfg.nl_a, len(cfg.actions), norm=False)
    lin("critic", 0, cfg.n_a, cfg.nl_a)
    lin("critic", 3, cfg.nl_a, 1, norm=False)
    lin("predict", 0, cfg.n_b, cfg.nl_b)
    lin("predict", 3, cfg.nl_b, cfg.nb_class, norm=False)
    return p
