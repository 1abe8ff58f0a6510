"""maze_window / maze_direction_mask through the C ABI vs the golden vectors recorded from the
unmodified reference's -v1 ("Enrich") envs and get_mask_direction(probs=True).  Bit-exact."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from conftest import GOLDEN, load_golden  # noqa: E402


def _replay(meta, z, visit_layout, on_step, visit_bits=False):
    import maze_b200 as mb
    pool = mb.MazePool.from_grids([z[f"m{m['id']}_grid"] for m in meta], [m["start"] for m in meta],
                                  [m["goal"] for m in meta], [m["topology"] == "torus" for m in meta])
    pairs = [(k, m, j) for k, m in enumerate(meta) for j in m["tapes"]]
    env_maze = torch.tensor([k for k, _, _ in pairs], dtype=torch.int32, device="cuda")
    batch = mb.MazeBatch(pool, len(pairs), env_maze=env_maze, visit_layout=visit_layout, visit_bits=visit_bits)
    tapes = [z[f"m{m['id']}_t{j}_action"] for _, m, j in pairs]
    T = max(len(t) for t in tapes)
    acts = np.zeros((T, len(pairs)), dtype=np.uint8)
    for e, t in enumerate(tapes):
        acts[:len(t), e] = t
    acts_d = torch.from_numpy(acts).cuda()
    batch.reset()
    on_step(batch, pairs, 0)
    for t in range(T):
        batch.step(acts_d[t], mode=0)
        on_step(batch, pairs, t + 1)


@pytest.mark.parametrize("name", ["steps", "steps81"])
@pytest.mark.parametrize("visit_layout", ["cell", "tile", "cell+bits", "tile+bits"])
def test_window_matches_reference_traces(name, visit_layout):
    """"+bits": the non_visited channel comes from the one-bit-per-block visited map (maze_env_batch.visit_bits, the -v1
    default of MazeVectorEnv) instead of the visit counters."""
    visit_bits = visit_layout.endswith("+bits")
    visit_layout = visit_layout.split("+")[0]
    z, meta = load_golden(name)
    meta = [m for m in meta if m["enrich"]]
    assert len(meta) >= (5 if name == "steps" else 1)
    checked = [0]

    def on_step(batch, pairs, t):
        win = batch.compute_window().cpu().numpy()
        an, tn = batch.agent_norm.cpu().numpy(), batch.target_norm.cpu().numpy()
        for e, (_, m, j) in enumerate(pairs):
            pre = f"m{m['id']}_t{j}_"
            if t > len(z[pre + "action"]):
                continue
            np.testing.assert_array_equal(win[e], z[pre + "window"][t].astype(np.float32), err_msg=f"{pre} step {t}")
            np.testing.assert_array_equal(an[e].view(np.uint64), z[pre + "agent"][t].view(np.uint64), err_msg=f"{pre} step {t}")
            np.testing.assert_array_equal(tn[e].view(np.uint64), z[pre + "target"][t].view(np.uint64))
            checked[0] += 1

    _replay(meta, z, visit_layout, on_step, visit_bits=visit_bits)
    assert checked[0] > (2000 if name == "steps" else 400)


def test_direction_mask_matches_reference_traces(golden_steps):
    z, meta = golden_steps
    checked = [0]

    def on_step(batch, pairs, t):
        probs = batch.direction_mask(probs=True).cpu().numpy()
        plain = batch.direction_mask(probs=False).cpu().numpy()
        for e, (_, m, j) in enumerate(pairs):
            pre = f"m{m['id']}_t{j}_"
            if t > len(z[pre + "action"]):
                continue
            ref = z[pre + "mask"][t]
            np.testing.assert_array_equal(probs[e], ref, err_msg=f"{pre} step {t}")
            assert set(np.unique(plain[e])) <= {0.0, 1.0}
            np.testing.assert_array_equal(plain[e][ref != 0.25], ref[ref != 0.25])
            checked[0] += 1

    _replay(meta, z, "cell", on_step)
    assert checked[0] > 5000


@pytest.mark.parametrize("visit_bits", [False, True])
def test_window_against_oracle_with_autoreset(visit_bits):
    """Window after autoresets and revisits, both topologies, vs the closed-form oracle (with the visited bitmap: it must be
    cleared by every episode start)."""
    from oracle.env_port import ClosedFormEnv
    import maze_b200 as mb
    z, meta = load_golden("bestdir")
    rows = [m for m in meta if m["shape"] >= 15][:8]
    mazes = [dict(grid=z[f"m{m['id']}_grid"], start=m["start"], goal=m["goal"], toroidal=m["topology"] == "torus") for m in rows]
    pool = mb.MazePool.from_grids([m["grid"] for m in mazes], [m["start"] for m in mazes], [m["goal"] for m in mazes],
                                  [m["toroidal"] for m in mazes])
    B = len(mazes)
    batch = mb.MazeBatch(pool, B, visit_layout="cell", visit_bits=visit_bits)
    envs = [ClosedFormEnv(m["grid"], m["start"], m["goal"], m["toroidal"], enrich=True) for m in mazes]
    batch.reset()
    obs = [e.reset()[0] for e in envs]
    pending = [False] * B
    rng = np.random.default_rng(3)
    for t in range(500):
        acts = rng.integers(0, 4, B).astype(np.uint8)
        batch.step(torch.from_numpy(acts).cuda(), mode=mb.cabi.STEP_AUTORESET)
        win = batch.compute_window().cpu().numpy()
        for i, env in enumerate(envs):
            if pending[i]:
                o, _ = env.reset()
                pending[i] = False
            else:
                o, _, tr, te, _ = env.step(int(acts[i]))
                pending[i] = bool(tr or te)
            np.testing.assert_array_equal(win[i], o["window"], err_msg=f"env {i} step {t}")


@pytest.mark.parametrize("toroidal", [False, True])
def test_render_matches_the_replayed_drawing_calls(toroidal):
    """maze_render against oracle/render.py (lib/maze_view.py's draw calls replayed on a numpy canvas)
    along one episode: fresh frame, trail outlines on every block the agent has left, agent square."""
    import maze_b200 as mb
    from oracle.render import Canvas
    pool = mb.MazePool(2, (21, 21))
    pool.generate(algorithms=["r-prim", "dfs"], toroidal=toroidal, seed=3)
    batch = mb.MazeBatch(pool, 2, env_maze=torch.tensor([0, 1], dtype=torch.int32, device="cuda"))
    batch.reset()
    meta = pool.meta_host()
    canv = [Canvas(pool.grid_host(m), (int(meta[m, 2]) & 0xffff, int(meta[m, 2]) >> 16)) for m in range(2)]
    frames = batch.render().cpu().numpy()
    assert frames.shape == (2, 21 * 16, 21 * 16, 3) and frames.dtype == np.uint8
    for m in range(2):
        assert np.array_equal(frames[m], canv[m].frame())
    rng = np.random.default_rng(5)
    moved_any = False
    for t in range(120):
        before = batch.agent.cpu().numpy().copy()
        batch.step(torch.from_numpy(rng.integers(0, 4, 2).astype(np.uint8)).cuda(), 0)
        after = batch.agent.cpu().numpy()
        if batch.terminated.any() or batch.truncated.any():
            break
        for m in range(2):
            if (before[m] != after[m]).any():
                canv[m].move_to(after[m])
                moved_any = True
        if t % 10 == 9:
            frames = batch.render().cpu().numpy()
            for m in range(2):
                assert np.array_equal(frames[m], canv[m].frame()), (t, m)
    assert moved_any
    one = batch.render([1]).cpu().numpy()
    assert np.array_equal(one[0], batch.render().cpu().numpy()[1])


def test_render_matches_frames_of_the_reference_view():
    """maze_render against frames of the UNMODIFIED lib/maze_view.py (tests/golden/render.npz; the reference's views driven on a
    software pygame -- they draw rectangles only, which rasterise exactly): frame after reset, then after every action of a
    scripted walk (moves, blocked moves, wraps on the torus) for as long as the first episode lasts.  Deviation, by design:
    maze_render draws the trail of the CURRENT episode (it is derived from the visit state), the reference's surface keeps
    the trails of earlier episodes until the maze changes -- so frames after a reset are not compared."""
    import maze_b200 as mb
    z = np.load(f"{GOLDEN}/render.npz")
    checked = 0
    for k in range(int(z["count"])):
        grid, frames, acts, pos = z[f"grid{k}"], z[f"frames{k}"], z[f"actions{k}"], z[f"pos{k}"]
        open_grid = (grid != 0).astype(np.uint8)
        pool = mb.MazePool.from_grids([open_grid], [tuple(z[f"start{k}"])], [tuple(z[f"goal{k}"])], bool(z[f"toroidal{k}"]))
        batch = mb.MazeBatch(pool, 1, env_maze=torch.zeros(1, dtype=torch.int32, device="cuda"))
        batch.reset()
        got = batch.render().cpu().numpy()[0]
        assert got.shape == frames[0].shape
        np.testing.assert_array_equal(got, frames[0], err_msg=f"maze {k}: frame after reset")
        for t, a in enumerate(acts):
            batch.step(torch.tensor([a], dtype=torch.uint8, device="cuda"), 0)
            if bool(batch.terminated.any()) or bool(batch.truncated.any()):
                break
            assert tuple(batch.agent.cpu().numpy()[0]) == tuple(pos[t]), (k, t)     # the env moves exactly when the view does
            np.testing.assert_array_equal(batch.render().cpu().numpy()[0], frames[1 + t], err_msg=f"maze {k} step {t}")
            checked += 1
    assert checked > 150


def test_bordered_flag_follows_a_pool_that_is_reconfigured_after_the_batch_was_built():
    """MAZE_BATCH_BORDERED selects the window / push kernels without torus code: a batch built over an empty (or bordered) pool
    must drop the flag when the pool's slots become toroidal, or its windows would clamp where they have to wrap."""
    import maze_b200 as mb
    pool = mb.MazePool(4, (21, 21))
    early = mb.MazeBatch(pool, 64, visit_bits=True, visit_layout="tile")
    assert early._c.flags & mb.cabi.BATCH_BORDERED
    pool.generate(algorithms="dfs", toroidal=True, seed=4)
    late = mb.MazeBatch(pool, 64, visit_bits=True, visit_layout="tile")
    assert not (late._c.flags & mb.cabi.BATCH_BORDERED)
    g = torch.Generator(device="cuda").manual_seed(1)
    for b in (early, late):
        b.reset()
    for _ in range(30):
        acts = torch.randint(0, 4, (64,), dtype=torch.uint8, device="cuda", generator=g)
        early.step(acts, 0)
        late.step(acts, 0)
    w_early, w_late = early.compute_window().clone(), late.compute_window().clone()
    assert not (early._c.flags & mb.cabi.BATCH_BORDERED)
    assert torch.equal(w_early, w_late)
    pool.generate(algorithms="dfs", toroidal=False, seed=5)      # every slot bordered again
    assert not pool.any_toroidal
    early.reset()
    early.compute_window()
    assert early._c.flags & mb.cabi.BATCH_BORDERED
