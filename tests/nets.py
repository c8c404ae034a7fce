"""Network shapes and oracle inputs shared by the GPU test modules (not a test module itself)."""
import torch

from oracle import marl_oracle as O
from tests.conftest import oracle_config

MOVES1 = [[1, 0], [-1, 0], [0, 1], [0, -1]]
MOVES3 = [[3, 0], [-3, 0], [0, 3], [0, -3]]


def model_config(ft, f, n, n_m, n_m_o, n_d, nl_b, nl_a, nc, actions):
    """A ``ModelConfig`` dict (marl.json schema) with equal belief / action widths ``n``."""
    return dict(ft_extr_str=ft, window_size=f, hidden_size_belief=n, hidden_size_action=n, hidden_size_msg=n_m,
                hidden_size_msg_output=n_m_o, hidden_size_state=n_d, state_dim=2, actions=actions, nb_class=nc,
                hidden_size_linear_belief=nl_b, hidden_size_linear_action=nl_a)


C1_NET = model_config("mnist", 6, 64, 16, 24, 8, 96, 96, 10, MOVES1)
C2_NET = model_config("resisc45", 12, 256, 64, 96, 16, 384, 384, 45, MOVES1)
SHIPPED_AID_NET = model_config("aid", 24, 768, 128, 192, 16, 1024, 1024, 30, MOVES3 + [[0, 0]])


def oracle_case(spec, seed=99):
    """Inputs of a ``spec`` (mc, na, nb, T, C, H, W): oracle config, parameters, images, labels, initial positions
    and states, and actions the oracle sampled itself (an on-distribution trajectory both sides replay)."""
    ocfg = oracle_config(spec["mc"])
    params = O.init_params(ocfg, seed=7)
    na, nb, T = spec["na"], spec["nb"], spec["T"]
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(nb, spec["C"], spec["H"], spec["W"], generator=g)
    y = torch.randint(ocfg.nb_class, (nb,), generator=g)
    pos0 = torch.stack([torch.randint(spec["H"] - ocfg.f, (na, nb), generator=g),
                        torch.randint(spec["W"] - ocfg.f, (na, nb), generator=g)], -1)
    hidden0 = [torch.randn(na, nb, n, generator=g) for n in (ocfg.n_b, ocfg.n_b, ocfg.n_a, ocfg.n_a)]
    actions = O.rollout(params, ocfg, img, pos0, hidden0, None, T, generator=g).actions
    return ocfg, params, img, y, pos0, hidden0, actions
