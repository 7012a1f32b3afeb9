"""TD3 / DDPG (csrc/offpolicy.cu) at the shapes the engine accepts beyond the benchmark's 256-256 networks and B = 256:
ragged M, N and K tiles, K past one prefetch round, a single-row minibatch, 1- to 4-layer networks whose policy and
critic depths differ, and an action limit at which the target clamp bites.  Every case is checked three ways:
  * step 0 (Q-values and TD losses) against a float64 evaluation from the initial parameters (north-star bar 1e-5);
  * the whole trajectory -- every network, targets included, Q-values and losses -- against the numpy oracle (2e-5);
  * every execution path (graph replay, persistent kernel, device gather) bit-identical to plain launches on
    host-staged minibatches.
Two sharp tests on frozen learners (lr = 0) pin the rounding of the polyak update and of the TD target to the
reference's: each product and the sum rounded separately (ref utils.py:47-57, td3.py:337-339)."""
import types

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import offpolicy as OP
from oracle import onpolicy as O

pytestmark = pytest.mark.gpu
F32 = np.float32
GAMMA = 0.99

# name: obs / act widths, policy and critic hidden widths, minibatch B; optional policy_delay (TD3), polyak rho,
# action limit, done fraction, TD3 only
CASES = {
    "reference_default": dict(O=11, A=3, p=[256, 256], q=[256, 256], B=100, done=0.3),  # learn(minibatch_size=100)
    "td3_paper": dict(O=17, A=6, p=[400, 300], q=[400, 300], B=100),                    # K = 400: two prefetch rounds
    "wide_observation": dict(O=376, A=17, p=[256, 256], q=[256, 256], B=256),           # [s | a] split at 376, K = 393
    "one_row": dict(O=3, A=1, p=[64, 64], q=[64, 64], B=1),
    "odd_widths": dict(O=11, A=3, p=[40, 24], q=[40, 24], B=33, delay=3, done=0.3),
    "large_minibatch": dict(O=11, A=3, p=[64, 64], q=[64, 64], B=1000),                 # dW with K = 1000
    "policy_1_critic_2": dict(O=8, A=2, p=[], q=[64], B=64, rho=0.9),
    "policy_4_critic_4": dict(O=8, A=2, p=[64, 48, 32], q=[64, 48, 32], B=100, rho=0.9),
    "policy_4_critic_2": dict(O=8, A=2, p=[64, 48, 32], q=[64], B=100, delay=3),
    "action_limit": dict(O=11, A=3, p=[64, 64], q=[64, 64], B=100, high=0.4, rho=0.9, td3_only=True),
}
MATRIX = [pytest.param(name, twin, id=f"{name}-{'td3' if twin else 'ddpg'}")
          for name, c in CASES.items() for twin in (True, False) if twin or not c.get("td3_only")]
# execution paths: (device gather, B200RL_OFFPOLICY_GRAPH, B200RL_OFFPOLICY_MEGAKERNEL)
PATHS = {"plain": (True, "0", "0"), "graph": (True, "1", "0"), "persistent": (True, "0", "1")}


def mlp_layers(rng, sizes, bias=0.05):
    return [(rng.standard_normal((o, i)).astype(F32) / np.sqrt(i), bias * rng.standard_normal(o).astype(F32))
            for i, o in zip(sizes[:-1], sizes[1:])]


def copy_layers(layers):
    return [(w.copy(), b.copy()) for w, b in layers]


def flat(m):
    return torch.nn.utils.parameters_to_vector(m.parameters()).detach().numpy().copy()


def make_learner(twin, pl, qls, tpl, tqls, high=1.0, lr=1e-3, rho=0.995, delay=2):
    """TD3 (twin) / DDPG through the public classes with networks of any sizes: pl / qls the online policy and
    critic(s), tpl / tqls their targets, all as lists of (W, b)."""
    from rl_replicas_b200.algorithms import DDPG, TD3
    from rl_replicas_b200.algorithms._onpolicy import describe_mlp, write_flat
    from rl_replicas_b200.networks import MLP
    from rl_replicas_b200.policies import DeterministicPolicy, RandomPolicy
    from rl_replicas_b200.q_function import QFunction
    load = lambda module, layers: write_flat(describe_mlp(module)[3], O.flatten_layers(layers))
    psizes, qsizes = O.layer_sizes(pl), O.layer_sizes(qls[0])
    pnet = MLP(psizes, torch.nn.ReLU, torch.nn.Tanh)
    load(pnet, pl)
    policy = DeterministicPolicy(pnet, torch.optim.Adam(pnet.parameters(), lr=lr))
    qfs = []
    for ql in qls:
        n = MLP(qsizes, torch.nn.ReLU)
        load(n, ql)
        qfs.append(QFunction(n, torch.optim.Adam(n.parameters(), lr=lr)))
    A = psizes[-1]
    env = types.SimpleNamespace(action_space=types.SimpleNamespace(high=np.full(A, high, F32), shape=(A,)),
                                spec=types.SimpleNamespace(id="stub"))
    if twin:
        algo = TD3(policy, RandomPolicy(None), qfs[0], qfs[1], env, None, None, None, gamma=GAMMA, polyak_rho=rho,
                   policy_delay=delay)
        targets = [algo.target_policy, algo.target_q_function_1, algo.target_q_function_2]
    else:
        algo = DDPG(policy, RandomPolicy(None), qfs[0], env, None, None, None, gamma=GAMMA, polyak_rho=rho)
        targets = [algo.target_policy, algo.target_q_function]
    for t, layers in zip(targets, [tpl] + list(tqls)):
        load(t.network, layers)
    algo.current_total_steps = 0  # what save_model records
    return algo


def networks(algo):
    """{oracle name: flat parameters} of every network of the learner, targets included."""
    qs = [algo.q_function_1, algo.q_function_2] if algo.n_q == 2 else [algo.q_function]
    tqs = [algo.target_q_function_1, algo.target_q_function_2] if algo.n_q == 2 else [algo.target_q_function]
    out = {"policy": flat(algo.policy.network), "target_policy": flat(algo.target_policy.network)}
    for i, (q, t) in enumerate(zip(qs, tqs)):
        out[f"q{i + 1}"], out[f"target_q{i + 1}"] = flat(q.network), flat(t.network)
    return out


def adam_moments(algo):
    mods = [algo.policy] + ([algo.q_function_1, algo.q_function_2] if algo.n_q == 2 else [algo.q_function])
    out = []
    for m in mods:
        st = m.optimizer.state
        for p in m.network.parameters():
            out += [st[p]["exp_avg"].numpy().ravel().copy(), st[p]["exp_avg_sq"].numpy().ravel().copy(),
                    np.array([float(st[p]["step"])])]
    return out


class _Columns:
    """Transition columns handed to ReplayBuffer.add_experience the way a PackedExperience hands them."""

    def __init__(self, cols):
        self.cols = cols

    def transition_columns(self):
        return self.cols


def replay(rng, O_dim, A, n=2000, high=1.0, done=0.01, rew=None):
    from rl_replicas_b200.replay_buffer import ReplayBuffer
    rb = ReplayBuffer()
    rewards = rng.standard_normal(n) if rew is None else np.full(n, rew, np.float64)
    rb.add_experience(_Columns((rng.standard_normal((n, O_dim)).astype(F32),
                                rng.uniform(-high, high, (n, A)).astype(F32), rewards,
                                rng.standard_normal((n, O_dim)).astype(F32), rng.random(n) < done)))
    return rb


def train(algo, rb, S, B, seed, device_replay=True):
    algo.use_device_replay = device_replay
    np.random.seed(seed)
    torch.manual_seed(seed)
    algo.train(rb, S, B)
    return {k: v.copy() for k, v in algo.last_train_output.items()}


def replay_draws(rb, S, B, A, seed, noisy):
    """The minibatches and target-smoothing noise train() drew: the same numpy / torch streams, consumed the same way."""
    np.random.seed(seed)
    torch.manual_seed(seed)
    mbs = [rb.sample_minibatch(B) for _ in range(S)]
    noise = np.stack([torch.randn(B, A).numpy() for _ in range(S)]) if noisy else None
    return mbs, noise


def setup(name, twin):
    """Initial networks (targets drawn apart from the online networks, so that a target read from the wrong network
    shows), replay content and hyper-parameters of one case."""
    c = CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)) + twin)
    ps, qs = [c["O"]] + c["p"] + [c["A"]], [c["O"] + c["A"]] + c["q"] + [1]
    n_q = 2 if twin else 1
    pl, qls = mlp_layers(rng, ps), [mlp_layers(rng, qs) for _ in range(n_q)]
    tpl, tqls = mlp_layers(rng, ps), [mlp_layers(rng, qs) for _ in range(n_q)]
    hp = dict(high=c.get("high", 1.0), rho=c.get("rho", 0.995), delay=c.get("delay", 2) if twin else 1)
    # At least two policy steps and two polyak updates, and no more: every step is another chance for a ReLU input within
    # rounding of 0 to gate the gradient differently in two correct float32 runs.  The wide-observation DDPG run meets
    # one (|z| = 1.2e-7 max|z| in the policy) in its 4th step, and 22000 policy weights then differ by up to 4e-4.
    S = 2 * hp["delay"] if twin else 3
    rb = replay(rng, c["O"], c["A"], high=hp["high"], done=c.get("done", 0.01))
    return (pl, qls, tpl, tqls), hp, rb, S, c["B"]


class _OracleAdam(O.AdamState):
    """The oracle's Adam, remembering each element's first gradient (see network_error)."""

    def apply(self, flat, grad):
        if self.step == 0:
            self.g1 = np.abs(grad.astype(np.float64))
        return super().apply(flat, grad)


def network_error(got, want, adam=None):
    """(rel_err, elements held to the looser bound) of a trained network against the oracle's.  Adam's first update of
    an element, lr * g / (|g| + eps), amplifies the rounding error of a gradient within a few eps of 0 by up to
    lr / eps = 1e5: a gradient of 6e-10 that float64 sums make 2.5e-10 moves its weight by 3.3e-5 (reference_default,
    DDPG, numpy against numpy).  So the elements whose first gradient is nonzero and below 10 eps -- a few in 10^3 --
    only have to agree to within one Adam step (2 lr); everywhere else the gain is at most lr eps / (10 eps)^2 ~ 800 on
    gradient errors of ~1e-9, and the 2e-5 bar holds."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = max(np.max(np.abs(want)), 1e-30)
    loose = np.zeros(want.shape, bool) if adam is None else (adam.g1 > 0) & (adam.g1 < 10 * adam.eps)
    assert loose.mean() < 1e-2, loose.mean()
    d = np.abs(got - want)
    if loose.any():
        assert d[loose].max() <= 2 * adam.lr, d[loose].max()
    return float(np.max(d[~loose], initial=0.0) / scale), int(loose.sum())


def forward64(layers, x, hidden, out):
    h = np.asarray(x, np.float64)
    for i, (w, b) in enumerate(layers):
        z = h @ w.astype(np.float64).T + b.astype(np.float64)
        kind = out if i == len(layers) - 1 else hidden
        h = np.tanh(z) if kind == "tanh" else np.maximum(z, 0.0) if kind == "relu" else z
    return h


def step0_float64(nets, mb, eps, high):
    """Q(s, a) of every critic and the TD losses of step 0 in float64 (td3.py:325-358; ddpg.py:275-282 when eps is
    None): initial parameters, the step's minibatch rows and noise."""
    pl, qls, tpl, tqls = nets
    obs, act, nobs = (np.asarray(mb[k], np.float64) for k in ("observations", "actions", "next_observations"))
    rew, done = np.asarray(mb["rewards"], np.float32).astype(np.float64), np.asarray(mb["dones"], np.float64)
    a2 = forward64(tpl, nobs, "relu", "tanh")
    if eps is not None:
        a2 = np.clip(a2 + np.clip(0.2 * eps.astype(np.float64), -0.5, 0.5), -high, high)
    tq = np.min([forward64(t, np.concatenate([nobs, a2], 1), "relu", "identity")[:, 0] for t in tqls], axis=0)
    y = rew + GAMMA * (1.0 - done) * tq
    qs = [forward64(q, np.concatenate([obs, act], 1), "relu", "identity")[:, 0] for q in qls]
    return qs, [float(np.mean((q - y) ** 2)) for q in qs]


@pytest.mark.parametrize("name,twin", MATRIX)
def test_step0_against_float64_and_trajectory_against_oracle(name, twin):
    nets, hp, rb, S, B = setup(name, twin)
    pl, qls, tpl, tqls = nets
    algo = make_learner(twin, *nets, **hp)
    out = train(algo, rb, S, B, seed=7)
    A = O.layer_sizes(pl)[-1]
    mbs, noise = replay_draws(rb, S, B, A, seed=7, noisy=twin)
    # step 0 against float64
    q64, l64 = step0_float64(nets, mbs[0], None if noise is None else noise[0], hp["high"])
    errs0 = {}
    for i in range(len(qls)):
        errs0[f"q{i + 1}_values[0]"] = rel_err(out[f"q{i + 1}_values"][0], q64[i])
        errs0[f"q{i + 1}_losses[0]"] = rel_err(out[f"q{i + 1}_losses"][0], l64[i])
    print(f"{name} step 0 vs float64:", {k: f"{v:.2e}" for k, v in errs0.items()})
    for k, v in errs0.items():
        assert v < 1e-5, (k, v, errs0)
    # the whole trajectory against the oracle on the same minibatches and noise
    onets = {"policy": copy_layers(pl), "target_policy": copy_layers(tpl)}
    for i in range(len(qls)):
        onets[f"q{i + 1}"], onets[f"target_q{i + 1}"] = copy_layers(qls[i]), copy_layers(tqls[i])
    adams = {k: _OracleAdam(O.flatten_layers(onets[k]).size, 1e-3) for k in onets if not k.startswith("target")}
    logs = OP.offpolicy_train(onets, adams, mbs, noise, gamma=GAMMA, rho=hp["rho"], action_limit=hp["high"],
                              policy_delay=hp["delay"], twin=twin)
    assert len(out["policy_losses"]) == len(logs["policy_losses"]) == len(range(0, S, hp["delay"]))
    errs = {"policy_losses": rel_err(out["policy_losses"], np.asarray(logs["policy_losses"]))}
    for i in range(len(qls)):
        errs[f"q{i + 1}_values"] = rel_err(out[f"q{i + 1}_values"], np.stack(logs[f"q{i + 1}_values"]))
        errs[f"q{i + 1}_losses"] = rel_err(out[f"q{i + 1}_losses"], np.asarray(logs[f"q{i + 1}_losses"]))
    loose = {}
    for k, v in networks(algo).items():
        errs[k], loose[k] = network_error(v, O.flatten_layers(onets[k]), adams.get(k))
    print(f"{name} trajectory vs oracle:", {k: f"{v:.2e}" for k, v in errs.items()},
          "elements within one Adam step:", {k: n for k, n in loose.items() if n})
    for k, v in errs.items():
        assert v < 2e-5, (k, v, errs)


@pytest.mark.parametrize("name,twin", MATRIX)
def test_every_path_is_bit_identical_to_plain_launches_on_staged_minibatches(name, twin, monkeypatch):
    """Graph replay, the persistent kernel and the device gather of the replay rows change where the work runs, not
    what it computes.  Two calls per learner: the second replays the captured graph / the built program."""
    nets, hp, rb, S, B = setup(name, twin)

    def run(device_replay, graph, mega):
        monkeypatch.setenv("B200RL_OFFPOLICY_GRAPH", graph)
        monkeypatch.setenv("B200RL_OFFPOLICY_MEGAKERNEL", mega)
        algo = make_learner(twin, *nets, **hp)
        outs = [train(algo, rb, S, B, seed=11 + call, device_replay=device_replay) for call in range(2)]
        return outs, networks(algo)

    ref_outs, ref_nets = run(False, "0", "0")
    for dev, graph, mega in ((False, "1", "0"), (False, "0", "1"), (True, "0", "0"), (True, "1", "0"),
                             (True, "0", "1")):
        outs, nets_ = run(dev, graph, mega)
        what = f"device gather={dev} graph={graph} persistent={mega}"
        for call, (a, b) in enumerate(zip(outs, ref_outs)):
            assert a.keys() == b.keys()
            for k in a:
                np.testing.assert_array_equal(a[k], b[k], err_msg=f"call {call} {k} {what}")
        for k in ref_nets:
            np.testing.assert_array_equal(nets_[k], ref_nets[k], err_msg=f"{k} {what}")


@pytest.mark.parametrize("twin", [True, False])
def test_engine_reuse_across_minibatch_sizes_matches_a_fresh_learner(twin, tmp_path):
    """One learner trains with (B = 256, S = 8), then (B = 100, S = 5) on the same engine (smaller shapes reuse the
    allocations), then B = 257 (the engine is rebuilt).  Each call gives what a fresh learner, loaded from a checkpoint
    of the state before the call, computes on the same random streams."""
    rng = np.random.default_rng(41)
    ps, qs = [11, 40, 24, 3], [14, 40, 24, 1]
    n_q = 2 if twin else 1
    nets = (mlp_layers(rng, ps), [mlp_layers(rng, qs) for _ in range(n_q)], mlp_layers(rng, ps),
            [mlp_layers(rng, qs) for _ in range(n_q)])
    rb = replay(rng, 11, 3, done=0.1)
    algo = make_learner(twin, *nets)
    engines = []
    for call, (B, S) in enumerate([(256, 8), (100, 5), (257, 5)]):
        ckpt = str(tmp_path / f"before_{call}.pt")
        algo.save_model(call, ckpt)
        out = train(algo, rb, S, B, seed=50 + call)
        engines.append(algo._engine)
        fresh = make_learner(twin, *nets)
        fresh.load_model(ckpt)
        want = train(fresh, rb, S, B, seed=50 + call)
        assert (fresh._engine.max_minibatch, fresh._engine.max_steps) == (B, S)
        for k in want:
            np.testing.assert_array_equal(out[k], want[k], err_msg=f"call {call} (B={B}, S={S}): {k}")
        got_nets, want_nets = networks(algo), networks(fresh)
        for k in want_nets:
            np.testing.assert_array_equal(got_nets[k], want_nets[k], err_msg=f"call {call} (B={B}, S={S}): {k}")
        for a, b in zip(adam_moments(algo), adam_moments(fresh)):
            np.testing.assert_array_equal(a, b, err_msg=f"call {call} (B={B}, S={S}): Adam state")
    assert engines[1] is engines[0] and engines[2] is not engines[0]
    assert (engines[2].max_minibatch, engines[2].max_steps) == (257, 5)


def _frozen(twin, nets, rho, path, monkeypatch, delay=2):
    """A learner whose three Adam optimizers have lr = 0: p - 0 * (m / denom) leaves every online parameter
    bit-unchanged, so the targets see the same online networks at every polyak update."""
    dev, graph, mega = PATHS[path]
    monkeypatch.setenv("B200RL_OFFPOLICY_GRAPH", graph)
    monkeypatch.setenv("B200RL_OFFPOLICY_MEGAKERNEL", mega)
    algo = make_learner(twin, *nets, lr=0.0, rho=rho, delay=delay)
    algo.use_device_replay = dev
    return algo


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("twin", [True, False], ids=["td3", "ddpg"])
def test_polyak_rounds_both_products_and_the_sum_separately(twin, path, monkeypatch):
    """target <- rho * target + (1 - rho) * param with float32 tensors rho and 1 - rho (ref utils.py:47-57): two
    rounded products and a rounded sum, never a fused multiply-add."""
    rng = np.random.default_rng(21)
    ps, qs = [11, 64, 64, 3], [14, 64, 64, 1]
    n_q = 2 if twin else 1
    nets = (mlp_layers(rng, ps), [mlp_layers(rng, qs) for _ in range(n_q)], mlp_layers(rng, ps),
            [mlp_layers(rng, qs) for _ in range(n_q)])
    rho, S, delay = 0.995, 6, 2
    algo = _frozen(twin, nets, rho, path, monkeypatch, delay)
    before = networks(algo)
    out = train(algo, replay(rng, 11, 3), S, 64, seed=3, device_replay=algo.use_device_replay)
    n_pol = len(range(0, S, delay if twin else 1))
    assert len(out["policy_losses"]) == n_pol
    after = networks(algo)
    for src in ["policy", "q1"] + (["q2"] if twin else []):
        np.testing.assert_array_equal(after[src], before[src], err_msg=f"{src} moved with lr = 0")
        p, t = before[src], before["target_" + src]
        for _ in range(n_pol):
            t = F32(rho) * t + F32(1.0 - rho) * p  # numpy float32: each product and the sum rounded on its own
        np.testing.assert_array_equal(after["target_" + src], t, err_msg=f"target_{src} after {n_pol} updates ({path})")


def _td_pair(rng):
    """(r, c) from U(0.5, 1) whose TD target r + f32(gamma) * c rounds differently when the product is kept exact (a
    fused multiply-add; emulated in float64, exact here because both terms are of the same magnitude)."""
    g = F32(GAMMA)
    for _ in range(1000):
        r, c = rng.uniform(0.5, 1.0, 2).astype(F32)
        y_sep = F32(r + F32(g * F32(1) * c))
        y_fused = F32(np.float64(r) + np.float64(g) * np.float64(c))
        if y_sep != y_fused:
            return r, c, y_sep
    raise AssertionError("no (r, c) pair separates the two roundings")


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("twin", [True, False], ids=["td3", "ddpg"])
def test_td_target_rounds_like_the_reference(twin, path, monkeypatch):
    """y = r + gamma * (1 - d) * min(Q1', Q2') with every operation rounded (td3.py:337-339).  Every critic ends in a
    zero-weight Linear, so on the device Q == its bias exactly: online b, target c.  rho = 1 keeps the targets at c for
    every step, and b is the separately rounded y, so each Q loss is exactly 0 -- a fused TD target leaves ulp^2."""
    rng = np.random.default_rng(31)
    r, c, y = _td_pair(rng)
    ps, qs = [11, 64, 64, 3], [14, 64, 64, 1]
    n_q = 2 if twin else 1

    def critic(bias):
        layers = mlp_layers(rng, qs)
        layers[-1] = (np.zeros_like(layers[-1][0]), np.full(1, bias, F32))
        return layers

    nets = (mlp_layers(rng, ps), [critic(y) for _ in range(n_q)], mlp_layers(rng, ps), [critic(c) for _ in range(n_q)])
    algo = _frozen(twin, nets, 1.0, path, monkeypatch)
    S, B = 4, 64
    out = train(algo, replay(rng, 11, 3, done=0.0, rew=r), S, B, seed=4, device_replay=algo.use_device_replay)
    for i in range(n_q):
        np.testing.assert_array_equal(out[f"q{i + 1}_values"], np.full((S, B), y, F32), err_msg=f"q{i + 1} ({path})")
        np.testing.assert_array_equal(out[f"q{i + 1}_losses"], np.zeros(S, F32), err_msg=f"q{i + 1} loss ({path})")
