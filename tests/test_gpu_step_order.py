"""maze_step runs its CTAs in reverse order on every other launch.  At a batch size that takes the two-envs-per-thread
kernel with a partial last CTA (which then runs first), consecutive maze_step launches of both parities must give
bit for bit what maze_step_many gives over the same action tape."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _golden_pool(mb):
    from conftest import load_golden
    grids, starts, goals, tors = [], [], [], []
    z, meta = load_golden("metrics")
    for m in meta:
        grids.append(z[f"m{m['id']}_grid"]); starts.append(m["start"]); goals.append(m["goal"]); tors.append(bool(m["no_border"]))
    for name in ("bestdir", "bestdir81"):
        z, meta = load_golden(name)
        for m in meta:
            grids.append(z[f"m{m['id']}_grid"]); starts.append(m["start"]); goals.append(m["goal"]); tors.append(m["topology"] == "torus")
    return mb.MazePool.from_grids(grids, starts, goals, tors)


@pytest.mark.parametrize("visit_layout", ["cell", "tile"])
def test_alternating_cta_order_matches_step_many(visit_layout):
    import maze_b200 as mb
    pool = _golden_pool(mb)
    M = pool.num_mazes
    B, K = 65536 + 77, 8                      # 129 CTAs of 512 envs, the last one holding 77
    env_maze = torch.from_numpy((np.arange(B) % M).astype(np.int32)).cuda()
    mode = mb.cabi.STEP_AUTORESET | mb.cabi.STEP_WIN_NEXT
    rng = np.random.default_rng(11)
    warm = torch.from_numpy(rng.integers(0, 4, (256, B)).astype(np.uint8)).cuda()
    one = mb.MazeBatch(pool, B, env_maze=env_maze.clone(), stats=True, pool_stride=5, visit_layout=visit_layout, visit_bits=True)
    many = mb.MazeBatch(pool, B, env_maze=env_maze.clone(), stats=True, pool_stride=5, visit_layout=visit_layout, visit_bits=True)
    one.reset(); many.reset()
    one.step_many(warm, mode); many.step_many(warm, mode)   # episodes at every stage: some envs end and restart below
    ended = 0
    for burst in range(2):                    # 8 launches per burst: both parities, twice
        tape = torch.from_numpy(rng.integers(0, 4, (K, B)).astype(np.uint8)).cuda()
        ref = {k: [] for k in ("agent", "best_dir", "reward", "terminated", "truncated")}
        for t in range(K):
            one.step(tape[t], mode)
            for k in ref:
                ref[k].append(getattr(one, k).clone())
        tr = many.step_many(tape, mode, trace=True)
        for k in ref:
            got, want = tr[k], torch.stack(ref[k])
            if k == "reward":
                got, want = got.view(torch.int64), want.view(torch.int64)
            assert torch.equal(got, want), (burst, k)
        ended += int((tr["terminated"].bool() | tr["truncated"].bool()).sum().item())
        for k in ("state", "env_maze", "agent", "target", "best_dir", "terminated", "truncated", "visits", "ep_return", "stats", "visit_bits"):
            assert torch.equal(getattr(many, k), getattr(one, k)), (burst, k)
        assert torch.equal(many.reward.view(torch.int64), one.reward.view(torch.int64)), burst
    assert ended > 0
