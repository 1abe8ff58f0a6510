"""CPU oracle for the batched-maze hot path.  TEST INFRASTRUCTURE ONLY.

This package restates, on the CPU, the algorithms of the reference
(Fabri000/Maze-Solving-Agent-Gymnasium) that the CUDA path replaces.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` legs may import
it; the product package (`maze-solving-agent-gymnasium_b200/`) never does and fails loudly
when its CUDA library is missing.

Parity status: PINNED.  Every function here is checked against outputs of the unmodified
reference imported in the build container (tests/golden/make_golden.py generated the committed
fixtures under tests/golden/*.npz) and against the reference's only known-answer material, the
literal 15x15 maze of testing_Mccledon.py:4-20 (values in BASELINE.md section 2).

Modules
  grid.py        A* (depth-limited, partial) port, BFS distance fields, block-grid helpers
  env_port.py    PortEnv: step/reset exactly as the reference computes them (A* per step);
                 ClosedFormEnv: the O(1) table-driven restatement the kernels implement
  generation.py  r-prim / dfs / prim&kill generators + goal selection + validity checks
  gen_stream.py  bit-exact model of the device generators' random stream (Philox-keyed PCG32)
  gen_exact.py   exact generator output distributions on small lattices, best-of-k, chi-square
  metrics.py     McClendon difficulty/complexity, Kim-Crawfis L / D / DE and the unused
                 Kim-Crawfis metrics (density, T, J, CR, AC/FDE/BDE, L_DE, *_sharp)
  qlearn.py      tabular Q / double-Q update rules
  mazeset.py     packed maze-set records (.mzs files) and the auto-encoder channel encode
"""
