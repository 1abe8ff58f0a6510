"""oracle/render.py against frames of the unmodified lib/maze_view.py (tests/golden/render.npz, made by
make_golden_render.py on a software pygame: the reference draws rectangles only, which rasterise exactly)."""
import numpy as np

from conftest import GOLDEN
from oracle.render import Canvas


def test_canvas_reproduces_the_reference_frames():
    z = np.load(f"{GOLDEN}/render.npz")
    total = 0
    for k in range(int(z["count"])):
        grid, start = z[f"grid{k}"], z[f"start{k}"]
        frames, moved, pos = z[f"frames{k}"], z[f"moved{k}"], z[f"pos{k}"]
        c = Canvas(grid, start)
        assert frames[0].shape == (grid.shape[0] * 16, grid.shape[1] * 16, 3)
        np.testing.assert_array_equal(c.frame(), frames[0], err_msg=f"maze {k}: frame after construction")
        for t in range(len(moved)):
            if moved[t]:
                c.move_to(pos[t])
            np.testing.assert_array_equal(c.frame(), frames[1 + t], err_msg=f"maze {k} step {t}")
            total += 1
        assert moved.any() and not moved.all()      # both a successful and a blocked move are in the walk
        c.move_to(start)                            # _reset_agent (maze_view.py:154-158): trail on the block left, agent at the start
        np.testing.assert_array_equal(c.frame(), frames[-1], err_msg=f"maze {k}: frame after _reset_agent")
    assert total == 240
