"""Golden outputs of the reference for the CPU differential tests that used to import it at test time:
    python tests/golden/make_golden_reference_cpu.py   ->  tests/golden/envelope_port.npz, tests/golden/termination.npz
(needs the reference, imported through oracle/ref_harness.py)

envelope_port.npz (tests/test_port_vs_reference.py): for per in {0, 1}, the reference Envelope's initial Q-net, the replay indices and weight
sets its three updates drew, and its Q-net after them.
termination.npz (tests/test_dyna_cpu.py): the reference's termination rules on the seeded batch of the test (bit-packed), and the rule its
ModelEnv picks for each env id."""

import os
import sys

import numpy as np
import torch as th

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh  # noqa: E402
from oracle.envelope_update_port import synthetic_store  # noqa: E402

# shared with the tests: the inputs are regenerated there from these seeds
PORT_CFG = dict(OBS=12, A=5, D=3, W=6, B=16, N=512, NET=[32, 32], SEED=3, STORE_SEED=1, STEPS=3)
TERMINATION_RULES = ("false", "mountaincar", "minecart", "hopper", "lunarlander", "humanoid")
ENV_IDS = ("mo-hopper-v4", "mo-halfcheetah-v4", "mo-humanoid-v4", "mo-lunar-lander-v2", "mo-reacher-v4", "mo-mountaincar-v0", "minecart-v0",
           "mo-highway-v0", "mo-highway-fast-v0")


def termination_batch(n=4000):
    """Random batches that hit both outcomes of every rule, NaN / inf rows included."""
    rng = np.random.default_rng(0)
    obs = (rng.standard_normal((n, 9)) * np.array([0.3, 0.3, 1, 1, 1, 1, 1, 1, 1])).astype(np.float32)
    nobs = (rng.standard_normal((n, 9)) * np.array([0.6, 0.15, 1, 1, 1, 1, 0.6, 0.6, 40])).astype(np.float32)
    nobs[:, 0] += 0.9  # heights / positions around the hopper, humanoid and mountain-car thresholds
    nobs[:, 6:8] += 0.8
    nobs[5, 3], nobs[6, 4], nobs[7, 8] = np.nan, np.inf, 250.0
    act = rng.integers(0, 2, (n, 4)).astype(np.float32)
    rew = (rng.standard_normal((n, 3)) * (rng.random((n, 1)) < 0.5)).astype(np.float32)
    return obs, act, nobs, rew


def envelope_port_golden(out):
    envm = rh.import_reference("morl_baselines.multi_policy.envelope.envelope")
    wm = rh.import_reference("morl_baselines.common.weights")
    c = PORT_CFG
    for per in (0, 1):
        th.manual_seed(0)
        agent = envm.Envelope(rh.FakeEnv(obs_dim=c["OBS"], n_actions=c["A"], reward_dim=c["D"]), batch_size=c["B"], num_sample_w=c["W"],
                              per=bool(per), buffer_size=c["N"], net_arch=c["NET"], log=False, seed=c["SEED"], device="cpu")
        store = synthetic_store(c["N"], c["OBS"], c["A"], c["D"], seed=c["STORE_SEED"])
        rb = agent.replay_buffer
        rb.obs[:], rb.next_obs[:], rb.actions[:], rb.rewards[:], rb.dones[:] = (store[k] for k in ("obs", "next_obs", "actions", "rewards", "dones"))
        rb.size, rb.ptr = c["N"], 0
        if per:
            rb.tree.batch_set(np.arange(c["N"]), np.full(c["N"], rb.min_priority))
        for k, v in agent.q_net.state_dict().items():
            out[f"per{per}/init/{k}"] = v.numpy().copy()
        rng = np.random.default_rng(c["SEED"])  # mirrors agent.np_random
        agent.global_step = 1
        idx_all, w_all = [], []
        for step in range(c["STEPS"]):
            np.random.seed(50 + step)
            # replicate the reference's draws: replay indices from the global RNG first, then the weights from the agent's generator
            state = np.random.get_state()
            idx_all.append(rb.tree.sample(c["B"]) if per else np.random.choice(c["N"], c["B"], replace=True))
            np.random.set_state(state)
            w_all.append(th.tensor(wm.random_weights(c["D"], c["W"], dist="gaussian", rng=rng)).float().numpy())
            agent.update()
        out[f"per{per}/idx"] = np.stack(idx_all).astype(np.int64)
        out[f"per{per}/wset"] = np.stack(w_all)
        for k, v in agent.q_net.state_dict().items():
            out[f"per{per}/final/{k}"] = v.numpy().copy()


def termination_golden(out):
    ref = rh.import_reference("morl_baselines.common.model_based.utils")
    obs, act, nobs, rew = termination_batch()
    for name in TERMINATION_RULES:
        want = np.asarray(getattr(ref, f"termination_fn_{name}")(obs, act, nobs, rew), dtype=bool)
        assert want.shape == (len(obs), 1), (name, want.shape)
        out[f"rule/{name}"] = np.packbits(want[:, 0])
    by_fn = {getattr(ref, f"termination_fn_{name}"): name for name in TERMINATION_RULES}
    out["env_ids"] = np.array(ENV_IDS)
    out["env_rules"] = np.array([by_fn[ref.ModelEnv(None, env_id).termination_func] for env_id in ENV_IDS])


def main():
    assert rh.reference_available(), "needs the reference"
    port, term = {}, {}
    envelope_port_golden(port)
    termination_golden(term)
    np.savez_compressed(os.path.join(HERE, "envelope_port.npz"), **port)
    np.savez_compressed(os.path.join(HERE, "termination.npz"), **term)
    print(len(port), "arrays in envelope_port.npz,", len(term), "in termination.npz")


if __name__ == "__main__":
    main()
