"""Error behaviour of the C ABI: every bad argument is reported as a negative MAZE_E_* code with a
message, nothing throws, nothing is launched."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _raw():
    import maze_b200 as mb
    pool = mb.MazePool(4, (21, 21))
    pool.generate(seed=1)
    batch = mb.MazeBatch(pool, 8)
    return mb, pool, batch, mb.cabi.lib(), pool.ctx.handle


def test_null_and_range_errors_have_codes_and_messages():
    mb, pool, batch, lib, ctx = _raw()
    st = mb.cabi.current_stream(pool.device)
    E = mb.cabi
    assert lib.maze_step(None, C.byref(batch._c), None, 0, st) == E.E_NULL
    assert lib.maze_step(ctx, C.byref(batch._c), None, 0, st) == E.E_NULL
    assert b"actions" in lib.maze_last_error(ctx)
    assert lib.maze_fields(ctx, None, mb.cabi.ptr(pool.meta), mb.cabi.ptr(pool.table), None, 4, pool.slot, st) == E.E_NULL
    assert lib.maze_fields(ctx, mb.cabi.ptr(pool.grids), mb.cabi.ptr(pool.meta), mb.cabi.ptr(pool.table), None, 0, pool.slot, st) == E.E_RANGE
    # generators stage one maze on chip: shapes above MAZE_GEN_MAX_DIM - 2 and even shapes are refused
    args = lambda h, w, cand=1: (ctx, mb.cabi.ptr(pool.grids), mb.cabi.ptr(pool.meta), mb.cabi.ptr(pool.table), None, None,  # noqa: E731
                                 4, pool.slot, h, w, 1, 0, cand, None, st)
    assert lib.maze_generate(*args(20, 21)) == E.E_SHAPE
    assert lib.maze_generate(*args(131, 131)) == E.E_SHAPE
    assert lib.maze_generate(*args(41, 41)) == E.E_RANGE          # does not fit the 21x21 slots
    assert lib.maze_generate(*args(21, 21, 0)) == E.E_RANGE       # candidates
    assert lib.maze_generate(*args(21, 21)) == 0
    # a batch with a misaligned / missing buffer
    bad = mb.cabi.MazeEnvBatch.from_buffer_copy(batch._c)
    bad.reward = batch.reward.data_ptr() + 4
    acts = torch.zeros(8, dtype=torch.uint8, device="cuda")
    assert lib.maze_step(ctx, C.byref(bad), mb.cabi.ptr(acts), 0, st) == E.E_ALIGN
    bad = mb.cabi.MazeEnvBatch.from_buffer_copy(batch._c)
    bad.visits = None
    assert lib.maze_reset(ctx, C.byref(bad), None, st) == E.E_NULL
    bad = mb.cabi.MazeEnvBatch.from_buffer_copy(batch._c)
    bad.num_envs = 0
    assert lib.maze_step(ctx, C.byref(bad), mb.cabi.ptr(acts), 0, st) == E.E_RANGE
    torch.cuda.synchronize()
    # the good batch still works afterwards
    batch.reset()
    batch.step(acts, mode=0)
    assert batch.state_host()["steps"].tolist() == [1] * 8


def test_host_side_validation():
    mb, pool, batch, lib, ctx = _raw()
    from maze_b200.agents import QAgent
    with pytest.raises(ValueError):
        pool.generate(algorithms="kruskal")
    with pytest.raises(ValueError):
        pool.generate(shapes=(22, 21))
    with pytest.raises(ValueError):
        mb.MazeBatch(pool, 4, visit_layout="diagonal")
    with pytest.raises(ValueError):
        mb.MazeBatch(pool, 4, visit_layout="env")
    with pytest.raises(ValueError):
        mb.MazeVectorEnv(8, shape=(21, 21), on_win="regenerate", num_mazes=4)     # needs one slot per env
    with pytest.raises(ValueError):
        mb.MazeVectorEnv(8, shape=(11, 11), enrich=True)                          # no 15x15 window in an 11x11 maze
    with pytest.raises(ValueError):
        mb.MazeVectorEnv(8, shape=(21, 21), grow=4)                               # curriculum needs on_win='regenerate'
    with pytest.raises(ValueError):
        QAgent(batch, 0.1, 0.9, 100, 0.05, 0.9, 1e-3, envs_per_agent=100)
    agent = QAgent(batch, 0.1, 0.9, 100, 0.05, 0.9, 1e-3, capacity=16)            # far too small: must be detected
    batch.reset()
    agent.rollout(200)
    with pytest.raises(mb.cabi.MazeError):
        agent.core.check_overflow()


def test_single_env_and_odd_batch_sizes():
    """B = 1 and B not a multiple of the CTA tile behave like any other batch."""
    from oracle.vector import OracleVector
    mb, pool, _, _, _ = _raw()
    meta = pool.meta_host()
    mazes = [dict(grid=pool.grid_host(m), start=(int(meta[m, 2]) & 0xffff, int(meta[m, 2]) >> 16),
                  goal=(int(meta[m, 3]) & 0xffff, int(meta[m, 3]) >> 16), toroidal=False) for m in range(4)]
    for B in (1, 513, 777):
        env_maze = np.arange(B) % 4
        batch = mb.MazeBatch(pool, B, env_maze=torch.from_numpy(env_maze.astype(np.int32)).cuda())
        ora = OracleVector(mazes, env_maze, autoreset=True)
        batch.reset(); ora.reset()
        rng = np.random.default_rng(B)
        for t in range(40):
            acts = rng.integers(0, 4, B).astype(np.uint8)
            batch.step(torch.from_numpy(acts).cuda(), mode=mb.cabi.STEP_AUTORESET)
            ref = ora.step(acts)
            np.testing.assert_array_equal(batch.agent.cpu().numpy(), ref["agent"])
            np.testing.assert_array_equal(batch.reward.cpu().numpy().view(np.uint64), ref["reward"].view(np.uint64))


def test_errors_of_the_abi_9_entry_points():
    """maze_step_many, maze_difficulty_ext, maze_pack / maze_unpack, maze_collection_encode, maze_render,
    maze_window alignment: bad arguments come back as MAZE_E_* codes with a message."""
    mb, pool, batch, lib, ctx = _raw()
    st = mb.cabi.current_stream(pool.device)
    E, ptr = mb.cabi, mb.cabi.ptr
    acts = torch.zeros((4, 8), dtype=torch.uint8, device="cuda")
    assert lib.maze_step_many(ctx, C.byref(batch._c), None, 4, 0, None, 0, st) == E.E_NULL
    assert lib.maze_step_many(ctx, C.byref(batch._c), ptr(acts), 0, 0, None, 0, st) == E.E_RANGE
    assert lib.maze_step_many(ctx, C.byref(batch._c), ptr(acts), 4, E.STEP_WIN_QUEUE, None, 0, st) == E.E_RANGE
    assert b"maze_step" in lib.maze_last_error(ctx)
    tr = E.MazeStepTrace(agent=batch.agent.data_ptr() + 4)
    assert lib.maze_step_many(ctx, C.byref(batch._c), ptr(acts), 4, 0, C.byref(tr), 0, st) == E.E_ALIGN
    out = torch.empty((4, E.METRIC_WORDS), dtype=torch.float64, device="cuda")
    assert lib.maze_difficulty_ext(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, 21, 21, ptr(out), None, st) == E.E_NULL
    assert lib.maze_difficulty_ext(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, 20, 21, ptr(out), ptr(out), st) == E.E_SHAPE
    packed = torch.empty((4, 56), dtype=torch.uint8, device="cuda")
    assert lib.maze_pack(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, 7, ptr(packed), 56, st) == E.E_RANGE        # format
    assert lib.maze_pack(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, E.PACK_BITMAP, ptr(packed), pool.slot, st) == E.E_RANGE   # stride > slot / 8
    assert lib.maze_pack(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, E.PACK_BITMAP, None, 56, st) == E.E_NULL
    assert lib.maze_unpack(ctx, ptr(packed), 56, E.PACK_BITMAP, ptr(pool.grids), ptr(pool.meta), None, 0, pool.slot, st) == E.E_RANGE
    assert lib.maze_unpack(ctx, ptr(packed), 56, E.PACK_BITMAP, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot + 1, st) == E.E_RANGE   # slot % 16
    coll = torch.empty((4, 3, 21, 21), dtype=torch.int32, device="cuda")
    assert lib.maze_collection_encode(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, 41, 41, ptr(coll), st) == E.E_RANGE
    assert lib.maze_collection_encode(ctx, ptr(pool.grids), ptr(pool.meta), None, 4, pool.slot, 21, 21, None, st) == E.E_NULL
    img = torch.empty((1, 21 * 16, 21 * 16, 3), dtype=torch.uint8, device="cuda")
    assert lib.maze_render(ctx, C.byref(batch._c), None, 1, ptr(img), 21 * 16 + 1, 21 * 16, st) == E.E_RANGE
    assert lib.maze_render(ctx, C.byref(batch._c), None, 9, ptr(img), 21 * 16, 21 * 16, st) == E.E_RANGE    # n > num_envs
    assert lib.maze_render(ctx, C.byref(batch._c), None, 1, None, 21 * 16, 21 * 16, st) == E.E_NULL
    win = torch.empty(8 * 675 + 4, dtype=torch.float32, device="cuda")
    assert lib.maze_window(ctx, C.byref(batch._c), win.data_ptr() + 4, None, None, st) == E.E_ALIGN
    torch.cuda.synchronize()
    # nothing was launched or damaged: the pool still scores and steps
    assert torch.isfinite(pool.difficulty()).all()
    batch.reset()
    batch.step_many(acts, 0)
    assert batch.state_host()["steps"].tolist() == [4] * 8


def test_windows_of_odd_batch_sizes_are_complete():
    """maze_window serves 8 envs per CTA with 16-byte stores: batch sizes that are not multiples of 8
    (tail CTA, scalar tail stores) must produce the same windows as the same envs in a larger batch."""
    import maze_b200 as mb
    pool = mb.MazePool(3, (21, 21))
    pool.generate(algorithms=["r-prim", "dfs", "prim&kill"], seed=4)
    rng = np.random.default_rng(1)
    tape = torch.from_numpy(rng.integers(0, 4, (30, 16)).astype(np.uint8)).cuda()
    ref = None
    for B in (16, 13, 9, 1):
        batch = mb.MazeBatch(pool, B, env_maze=torch.arange(B, dtype=torch.int32, device="cuda") % 3, visit_layout="tile")
        batch.reset()
        for t in range(30):
            batch.step(tape[t, :B].contiguous(), 0)
        w = batch.compute_window().cpu().numpy()
        if ref is None:
            ref = w
            assert ref.sum() > 0
        assert np.array_equal(w, ref[:B]), B
