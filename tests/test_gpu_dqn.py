"""DQN data path (maze_dqn_observe / push / sample / select) against the oracle's -v1 observation
and direction mask: every transition in the ring is a transition the oracle envs made, sampled
batches unpack to the right windows, and the masked epsilon-greedy draws the reference's
distribution."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from conftest import load_golden  # noqa: E402
from oracle.env_port import ClosedFormEnv  # noqa: E402


def _setup(B_per_maze=4, visit_bits=False):
    import maze_b200 as mb
    z, meta = load_golden("bestdir")
    rows = [m for m in meta if m["shape"] >= 15][:6]
    mazes = [dict(grid=z[f"m{m['id']}_grid"], start=tuple(m["start"]), goal=tuple(m["goal"]), toroidal=m["topology"] == "torus") for m in rows]
    pool = mb.MazePool.from_grids([m["grid"] for m in mazes], [m["start"] for m in mazes], [m["goal"] for m in mazes],
                                  [m["toroidal"] for m in mazes])
    B = B_per_maze * len(mazes)
    env_maze = np.arange(B) % len(mazes)
    batch = mb.MazeBatch(pool, B, env_maze=torch.from_numpy(env_maze.astype(np.int32)).cuda(), visit_layout="cell", visit_bits=visit_bits)
    envs = [ClosedFormEnv(mazes[k]["grid"], mazes[k]["start"], mazes[k]["goal"], mazes[k]["toroidal"], enrich=True) for k in env_maze]
    return mb, batch, envs


def _state_of(obs):
    vec = np.concatenate([obs["agent"], obs["target"], obs["best dir"]]).astype(np.float32)   # off_policy_trainer.py:156
    return vec, np.asarray(obs["window"], dtype=np.float32)


@pytest.mark.parametrize("visit_bits", [False, True])
def test_replay_holds_exactly_the_oracle_transitions_and_samples_unpack(visit_bits):
    from maze_b200.dqn import DeviceReplay, unpack_windows
    mb, batch, envs = _setup(visit_bits=visit_bits)
    B, T = batch.num_envs, 120
    mem = DeviceReplay(batch, capacity=B * T, seed=3)
    batch.reset()
    mem.observe()
    obs = [e.reset()[0] for e in envs]
    vec0, win0 = mem.current_state()
    for i in range(B):
        v, w = _state_of(obs[i])
        np.testing.assert_array_equal(vec0[i].cpu().numpy(), v)
        np.testing.assert_array_equal(win0[i].cpu().numpy(), w)
    expected = set()
    pending = [False] * B
    rng = np.random.default_rng(1)
    for t in range(T):
        acts = rng.integers(0, 4, B).astype(np.uint8)
        a_d = torch.from_numpy(acts).cuda()
        batch.step(a_d, mode=mb.cabi.STEP_AUTORESET)
        mem.push(a_d)
        for i, env in enumerate(envs):
            if pending[i]:
                obs[i], _ = env.reset()
                pending[i] = False
                continue
            nobs, r, trunc, term, _ = env.step(int(acts[i]))
            v, w = _state_of(obs[i])
            nv, nw = _state_of(nobs)
            expected.add((v.tobytes(), w.tobytes(), int(acts[i]), np.float32(r).tobytes(), nv.tobytes(), nw.tobytes()))
            pending[i] = bool(trunc or term)
            obs[i] = nobs
    n = len(mem)
    got = set()
    wins, nwins = unpack_windows(mem.win[:n]).cpu().numpy(), unpack_windows(mem.next_win[:n]).cpu().numpy()
    vec, nvec = mem.vec[:n].cpu().numpy(), mem.next_vec[:n].cpu().numpy()
    act, rew = mem.action[:n].cpu().numpy(), mem.reward[:n].cpu().numpy()
    for k in range(n):
        got.add((vec[k].tobytes(), wins[k].tobytes(), int(act[k]), rew[k].tobytes(), nvec[k].tobytes(), nwins[k].tobytes()))
    assert got == expected and n >= len(expected) > B * T // 2
    # sampling: every drawn transition is one of the stored ones, and the draw covers the ring
    (sv, sw), sa, sr, (snv, snw) = mem.sample(4096)
    sv, sw, sa, sr, snv, snw = (x.cpu().numpy() for x in (sv, sw, sa, sr, snv, snw))
    assert sw.shape == (4096, 3, 15, 15) and sa.dtype == np.int64
    drawn = {(sv[k].tobytes(), sw[k].tobytes(), int(sa[k]), sr[k].tobytes(), snv[k].tobytes(), snw[k].tobytes()) for k in range(4096)}
    assert drawn <= expected and len(drawn) > 0.5 * min(len(expected), 4096)
    (sv2, _), _, _, _ = mem.sample(4096)
    assert not np.array_equal(sv2.cpu().numpy(), sv)          # a fresh draw each call


def test_ring_wraps_and_len_saturates():
    from maze_b200.dqn import DeviceReplay
    mb, batch, envs = _setup(2)
    B = batch.num_envs
    mem = DeviceReplay(batch, capacity=5 * B)
    batch.reset(); mem.observe()
    acts = torch.zeros(B, dtype=torch.uint8, device="cuda")
    for t in range(12):
        batch.step(acts, mode=0)
        mem.push(acts)
    assert int(mem.pushed.item()) == 12 * B and len(mem) == 5 * B
    (v, w), a, r, _ = mem.sample(64)
    assert torch.isfinite(v).all() and set(np.unique(w.cpu().numpy())) <= {0.0, 1.0}


def test_masked_epsilon_greedy_matches_reference_distribution():
    """eps = 1: every action comes from np.random.choice(4, p=mask/mask.sum()) with the reference's
    probs=True mask; eps = 0: argmax of the q-values."""
    from maze_b200.dqn import MaskedEpsilonGreedy
    mb, batch, envs = _setup(1)
    B = batch.num_envs
    batch.reset()
    for e in envs:
        e.reset()
    rng = np.random.default_rng(5)
    for t in range(6):   # walk a little so that the 0.25 "back" weight is in play
        acts = rng.integers(0, 4, B).astype(np.uint8)
        batch.step(torch.from_numpy(acts).cuda(), mode=0)
        for i, e in enumerate(envs):
            e.step(int(acts[i]))
    masks = np.stack([np.asarray(e.mask_direction(probs=True), dtype=np.float64) for e in envs])
    np.testing.assert_array_equal(batch.direction_mask(probs=True).cpu().numpy(), masks.astype(np.float32))
    q = torch.randn(B, 4, device="cuda")
    greedy = MaskedEpsilonGreedy(batch, 0.0, 0.0, 100.0)
    np.testing.assert_array_equal(greedy.select(q).cpu().numpy(), q.argmax(1).cpu().numpy())
    explore = MaskedEpsilonGreedy(batch, 1.0, 1.0, 100.0, seed=9)
    N = 6000
    counts = np.zeros((B, 4))
    for _ in range(N):
        a = explore.select(q).cpu().numpy()
        counts[np.arange(B), a] += 1
    p = masks / masks.sum(1, keepdims=True)
    assert (counts[p == 0] == 0).all()
    assert np.abs(counts / N - p).max() < 4.5 * np.sqrt(0.25 / N)
    assert int(explore.steps_done.cpu()[0]) == N


def test_sampling_without_replacement_is_random_sample():
    """ReplayMemory.sample is random.sample(memory, batch_size) (lib/replay_memory.py:20-21): a batch holds DISTINCT
    transitions.  The ring's default reproduces that (first n images of a keyed pseudo-random permutation of the stored
    slots): a batch of the whole ring is a permutation of it, every smaller batch is duplicate-free, every slot is equally
    likely, and different draws give different batches.  without_replacement=False is the round-1 behaviour
    (independent uniform draws, duplicates expected)."""
    from maze_b200.dqn import DeviceReplay
    mb, batch, _ = _setup(B_per_maze=8)
    B = batch.num_envs
    N = 3000                                              # stored transitions: not a power of two
    mem = DeviceReplay(batch, capacity=4096, seed=11)
    assert mem._c.without_replacement == 1
    mem.reward[:N] = torch.arange(N, dtype=torch.float32, device="cuda")    # tag every slot
    mem.pushed.fill_(N)
    _, _, reward, _ = mem.sample(N)
    assert torch.equal(reward.sort()[0], torch.arange(N, dtype=torch.float32, device="cuda"))
    counts = torch.zeros(N, device="cuda")
    first = None
    for d in range(300):
        r = mem.sample_packed(500)[5]
        assert r.unique().numel() == 500 and r.max() < N
        counts += torch.bincount(r.long(), minlength=N).float()
        if d == 0:
            first = r.clone()
        elif d == 1:
            assert not torch.equal(first, r)
    expected = 300 * 500 / N                               # 50 per slot; binomial sd ~ 6.5
    assert counts.min() > expected - 6 * 6.5 and counts.max() < expected + 6 * 6.5
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert chi2 < N * (1 - 500 / N) + 6 * (2 * N) ** 0.5   # hypergeometric draws: variance a little below binomial
    # n larger than what is stored: the reference's agent returns before sampling (ddqn_agent.py:114-115); here the draws
    # fall back to independent ones instead of failing on the device
    r = mem.sample_packed(4000)[5]
    assert r.max() < N and r.unique().numel() < 4000
    loose = DeviceReplay(batch, capacity=4096, seed=11, without_replacement=False)
    loose.reward[:N] = torch.arange(N, dtype=torch.float32, device="cuda")
    loose.pushed.fill_(N)
    assert loose.sample_packed(2000)[5].unique().numel() < 2000
