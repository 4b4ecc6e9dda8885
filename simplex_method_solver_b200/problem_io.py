"""Problem files of the reference GUI (SURVEY.md §8f, N3) and a batched loader for them.

Format written by ``MainWindow.save_state`` (/root/reference/src/main.py:387-395) and parsed by
``load_state`` (main.py:417-482): one constraint per line as ``a1,a2,b``, then the gradient as
``g1,g2,0``, then the integer plot limit ``lim`` on the last line (no trailing newline).  The
solver sees ``constraints = [[a1, a2, b], ...]`` and ``function = [g1, g2]`` (main.py:309-312).
"""
from __future__ import annotations

from typing import Iterable, NamedTuple

import numpy as np


class Problem(NamedTuple):
    rows: list          # [[a1, a2, b], ...]
    grad: list          # [g1, g2, g3] as stored (the solver uses grad[:-1])
    lim: int


def dumps(rows, grad, lim: int) -> str:
    """main.py:387-395: ``str()`` of every coefficient, comma separated; lim last, no newline."""
    out = [",".join(map(str, r)) for r in rows]
    out.append(",".join(map(str, grad)))
    return "\n".join(out) + "\n" + str(lim)


def loads(text: str) -> Problem:
    """main.py:417-482: at least two lines; every data line has exactly three numbers."""
    lines = text.splitlines()
    if len(lines) < 2:
        raise ValueError("bad file format: at least a gradient line and a limit line are needed")
    data, rows, grad = lines[:-1], [], None
    for k, line in enumerate(data):
        vals = line.strip().split(",")
        if len(vals) != 3:
            raise ValueError(f"bad format in line {k + 1}: {line.strip()}")
        nums = list(map(float, vals))
        if k < len(data) - 1:
            rows.append(nums)
        else:
            grad = nums
    return Problem(rows, grad, int(lines[-1].strip()))


def save(path: str, rows, grad, lim: int) -> None:
    with open(path, "w", encoding="utf-8") as fh:
        fh.write(dumps(rows, grad, lim))


def load(path: str) -> Problem:
    with open(path, "r", encoding="utf-8") as fh:
        return loads(fh.read())


def solver_inputs(problem: Problem):
    """(constraints, function) as ``compute_solution`` passes them (main.py:309-312)."""
    return [list(map(float, r)) for r in problem.rows], list(problem.grad)[:-1]


def batch_tables(problems: Iterable[Problem]) -> tuple[np.ndarray, int, int]:
    """Problems of one shape -> the [B, cells] reference-flat array ``solve_batched`` takes.

    Returns (tables, n, m).  Raises if the shapes differ: problems of mixed shapes go to
    ``batched.solve_ragged([solver_inputs(p) for p in problems], ...)`` in one call.
    """
    flat, shape = [], None
    for p in problems:
        rows, c = solver_inputs(p)
        n, m = len(rows), len(c)
        if shape is None:
            shape = (n, m)
        elif shape != (n, m):
            raise ValueError(f"mixed shapes in one batch: {shape} and {(n, m)}")
        flat.append(np.concatenate([np.asarray(rows, dtype=np.float64).reshape(-1), np.asarray(c, dtype=np.float64)]))
    if shape is None:
        raise ValueError("empty batch")
    return np.stack(flat), shape[0], shape[1]
