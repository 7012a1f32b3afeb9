"""Checkpoint parity + resume (SURVEY 8f-3): save_model writes the reference's dictionary layout, load_model restores
networks, Adam state and step counters; checkpoints written the way the reference writes them load as warm starts."""
import os
import types

import numpy as np
import torch


def _ppo(seed, sizes_p=(5, 64, 64, 2), sizes_v=(5, 64, 64, 1)):
    from rl_replicas_b200.algorithms import PPO
    from rl_replicas_b200.networks import MLP
    from rl_replicas_b200.policies import GaussianPolicy
    from rl_replicas_b200.value_function import ValueFunction
    torch.manual_seed(seed)
    pnet, vnet = MLP(list(sizes_p)), MLP(list(sizes_v))
    policy = GaussianPolicy(pnet, torch.optim.Adam(pnet.parameters(), lr=3e-4),
                            torch.nn.Parameter(torch.full((sizes_p[-1],), -0.5)))
    algo = PPO(policy, ValueFunction(vnet, torch.optim.Adam(vnet.parameters(), lr=1e-3)), None, None)
    algo.current_total_steps = 0
    return algo


def _fake_adam_progress(optimizer, steps):
    """Populate Adam state the way `steps` real updates would leave it (any values: the test is about round-tripping)."""
    for group in optimizer.param_groups:
        for p in group["params"]:
            optimizer.state[p] = {"step": torch.tensor(float(steps)), "exp_avg": torch.randn_like(p),
                                  "exp_avg_sq": torch.rand_like(p)}


def test_ppo_checkpoint_round_trip(tmp_path):
    a = _ppo(0)
    _fake_adam_progress(a.policy.optimizer, 37)
    _fake_adam_progress(a.value_function.optimizer, 80)
    a.current_total_steps = 123456
    path = os.path.join(tmp_path, "model.pt")
    a.save_model(17, path)
    ckpt = torch.load(path, weights_only=False)
    assert set(ckpt) == {"epoch", "total_steps", "policy_state_dict", "policy_optimizer_state_dict",
                         "value_function_state_dict", "value_function_optimizer_state_dict"}  # ref ppo.py:296-306
    assert list(ckpt["policy_state_dict"]) == ["network.0.weight", "network.0.bias", "network.2.weight", "network.2.bias",
                                               "network.4.weight", "network.4.bias"]
    b = _ppo(1)
    assert b.load_model(path) == 17 and b.current_total_steps == 123456
    for ma, mb in ((a.policy, b.policy), (a.value_function, b.value_function), (a.policy, b.old_policy)):
        for pa, pb in zip(ma.network.parameters(), mb.network.parameters()):
            assert torch.equal(pa, pb)
    for oa, ob in ((a.policy.optimizer, b.policy.optimizer), (a.value_function.optimizer, b.value_function.optimizer)):
        for pa, pb in zip(oa.param_groups[0]["params"], ob.param_groups[0]["params"]):
            for k in ("step", "exp_avg", "exp_avg_sq"):
                assert torch.equal(torch.as_tensor(oa.state[pa][k]), torch.as_tensor(ob.state[pb][k]))
    # the engine-facing readers see the restored state (this is what the next train() uploads)
    from rl_replicas_b200.algorithms._onpolicy import describe_mlp, read_adam_state
    m, v, step = read_adam_state(b.policy.optimizer, describe_mlp(b.policy.network)[3])
    assert step == 37 and m.shape == v.shape


def _td3(seed, o=17, a=6, h=256):
    from rl_replicas_b200.algorithms import TD3
    from rl_replicas_b200.networks import MLP
    from rl_replicas_b200.policies import DeterministicPolicy, RandomPolicy
    from rl_replicas_b200.q_function import QFunction
    from rl_replicas_b200.replay_buffer import ReplayBuffer
    torch.manual_seed(seed)
    pnet = MLP([o, h, h, a], torch.nn.ReLU, torch.nn.Tanh)
    qs = [MLP([o + a, h, h, 1], torch.nn.ReLU) for _ in range(2)]
    env = types.SimpleNamespace(action_space=types.SimpleNamespace(high=np.ones(a, np.float32), shape=(a,)),
                                spec=types.SimpleNamespace(id="stub"))
    algo = TD3(DeterministicPolicy(pnet, torch.optim.Adam(pnet.parameters(), lr=1e-3)), RandomPolicy(None),
               QFunction(qs[0], torch.optim.Adam(qs[0].parameters(), lr=1e-3)),
               QFunction(qs[1], torch.optim.Adam(qs[1].parameters(), lr=1e-3)), env, None, ReplayBuffer(), None)
    algo.current_total_steps = 0
    return algo


def test_td3_checkpoint_round_trip(tmp_path):
    a = _td3(0, h=32)
    for m in (a.policy, a.q_function_1, a.q_function_2):
        _fake_adam_progress(m.optimizer, 11)
    with torch.no_grad():
        for t in (a.target_policy, a.target_q_function_1, a.target_q_function_2):
            for p in t.network.parameters():
                p.add_(0.25)  # targets differ from the online networks, as after polyak averaging
    path = os.path.join(tmp_path, "model.pt")
    a.save_model(5, path)
    b = _td3(1, h=32)
    assert b.load_model(path) == 5
    pairs = ((a.policy, b.policy), (a.q_function_1, b.q_function_1), (a.q_function_2, b.q_function_2),
             (a.target_policy, b.target_policy), (a.target_q_function_1, b.target_q_function_1),
             (a.target_q_function_2, b.target_q_function_2))
    for ma, mb in pairs:
        for pa, pb in zip(ma.network.parameters(), mb.network.parameters()):
            assert torch.equal(pa, pb)
    assert not any(p.requires_grad for p in b.target_policy.network.parameters())


class _ReferenceMLP(torch.nn.Module):
    """The reference's network layout (ref networks/mlp.py): Linear / activation pairs in ``self.network``, so the
    state-dict keys read network.<i>.weight / network.<i>.bias."""

    def __init__(self, sizes, activation, output_activation=torch.nn.Identity):
        super().__init__()
        layers = []
        for i in range(len(sizes) - 1):
            layers += [torch.nn.Linear(sizes[i], sizes[i + 1]),
                       activation() if i < len(sizes) - 2 else output_activation()]
        self.network = torch.nn.Sequential(*layers)

    def forward(self, x):
        return self.network(x)


# Adam's param-group keys in torch 2.5.1, the version the reference pins (pyproject.toml): newer torch adds others
_ADAM_GROUP_KEYS_TORCH_2_5 = {"params", "lr", "betas", "eps", "weight_decay", "amsgrad", "maximize", "foreach",
                              "capturable", "differentiable", "fused"}


def _trained(sizes, activation, output_activation=torch.nn.Identity):
    """A network and its Adam state dict after a few real steps (moments and a step count), laid out as torch 2.5.1
    writes it."""
    net = _ReferenceMLP(sizes, activation, output_activation)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    for _ in range(3):
        opt.zero_grad()
        net(torch.randn(8, sizes[0])).pow(2).mean().backward()
        opt.step()
    sd = opt.state_dict()
    sd["param_groups"] = [{k: v for k, v in g.items() if k in _ADAM_GROUP_KEYS_TORCH_2_5} for g in sd["param_groups"]]
    return net, sd


def _reference_checkpoints(directory):
    """{algorithm: path} of checkpoints with the dictionaries the reference's save_model writes (ref ppo.py:296-306;
    vpg.py and trpo.py use the same keys; td3.py:367-382), built from plain torch modules at the shapes of the shipped
    benchmark checkpoints: HalfCheetah [64, 32] nets (17 -> 64 -> 32 -> 6 policy, 17 -> 64 -> 32 -> 1 value, tanh;
    run_ppo.py:28-29), used here for PPO, VPG and TRPO, and TD3 on Hopper (11 -> 256 -> 256 -> 3 policy, relu with tanh
    output; 14 -> 256 -> 256 -> 1 critics).  TRPO's
    policy optimizer is the conjugate-gradient one, whose state dict holds its hyper-parameters and no per-parameter
    state (ref optimizers/conjugate_gradient_optimizer.py:100-119)."""
    torch.manual_seed(0)
    paths = {}
    for epoch, algo in enumerate(("ppo", "vpg", "trpo"), start=1):
        (pnet, popt), (vnet, vopt) = _trained([17, 64, 32, 6], torch.nn.Tanh), _trained([17, 64, 32, 1], torch.nn.Tanh)
        if algo == "trpo":
            popt = {"state": {"max_constraint": 0.01, "n_conjugate_gradients": 10, "max_backtracks": 15,
                              "backtrack_ratio": 0.8, "hvp_damping_coefficient": 1e-5},
                    "param_groups": [{"params": list(range(6))}]}
        paths[algo] = os.path.join(directory, algo + ".pt")
        torch.save({"epoch": 100 * epoch, "total_steps": 400000 * epoch,
                    "policy_state_dict": pnet.state_dict(), "policy_optimizer_state_dict": popt,
                    "value_function_state_dict": vnet.state_dict(), "value_function_optimizer_state_dict": vopt},
                   paths[algo])
    pnet, popt = _trained([11, 256, 256, 3], torch.nn.ReLU, torch.nn.Tanh)
    ckpt = {"epoch": 300, "total_steps": 1000000,
            "policy_state_dict": pnet.state_dict(), "policy_optimizer_state_dict": popt,
            "target_policy_state_dict": _ReferenceMLP([11, 256, 256, 3], torch.nn.ReLU, torch.nn.Tanh).state_dict()}
    for q in ("q_function_1", "q_function_2"):
        qnet, qopt = _trained([14, 256, 256, 1], torch.nn.ReLU)
        ckpt.update({f"{q}_state_dict": qnet.state_dict(), f"{q}_optimizer_state_dict": qopt,
                     f"target_{q}_state_dict": _ReferenceMLP([14, 256, 256, 1], torch.nn.ReLU).state_dict()})
    paths["td3"] = os.path.join(directory, "td3.pt")
    torch.save(ckpt, paths["td3"])
    return paths


def test_reference_layout_checkpoints_load_as_warm_starts(tmp_path):
    """One checkpoint per algorithm family: layer sizes come from the file, the loaded module reproduces a plain-torch
    evaluation of the stored weights."""
    seen = set()
    for algo_name, path in _reference_checkpoints(str(tmp_path)).items():
        seen.add(algo_name)
        ckpt = torch.load(path, map_location="cpu", weights_only=False)
        sd = ckpt["policy_state_dict"]
        ws = [v for k, v in sd.items() if k.endswith("weight")]
        sizes = [ws[0].shape[1]] + [w.shape[0] for w in ws]
        if "q_function_1_state_dict" in ckpt:
            algo = _td3(0, o=sizes[0], a=sizes[-1], h=sizes[1])
            epoch = algo.load_model(path)
            x = torch.randn(4, sizes[0])
            want = x
            for i, w in enumerate(ws):
                want = torch.nn.functional.linear(want, w, sd[f"network.{2 * i}.bias"])
                want = torch.tanh(want) if i == len(ws) - 1 else torch.relu(want)
            assert torch.allclose(algo.policy.network(x), want, atol=1e-6)
            assert int(algo.q_function_1.optimizer.state_dict()["state"][0]["step"]) > 0
        elif "value_function_state_dict" in ckpt and "q_function_state_dict" not in ckpt:
            vs = [v for k, v in ckpt["value_function_state_dict"].items() if k.endswith("weight")]
            algo = _ppo(0, tuple(sizes), tuple([vs[0].shape[1]] + [w.shape[0] for w in vs]))
            epoch = algo.load_model(path)
            x = torch.randn(4, sizes[0])
            want = x
            for i, w in enumerate(ws):
                want = torch.nn.functional.linear(want, w, sd[f"network.{2 * i}.bias"])
                if i < len(ws) - 1:
                    want = torch.tanh(want)
            assert torch.allclose(algo.policy.network(x), want, atol=1e-6)
        else:
            continue
        assert epoch == ckpt["epoch"] and algo.current_total_steps == ckpt["total_steps"]
    assert seen == {"ppo", "vpg", "trpo", "td3"}
