"""An independent reader of .smx files (the reference's format, src/smatrix.c:30-72), in numpy only: it
shares no code with the library or with the C checker, so it can judge both.

    512-byte header   8 x 0x17, u64 offset of the first directory block
    directory block   u64 entries, u64 next block (0 = last), entries x {u32 row, u64 row offset};
                      an entry with offset 0 ends its block
    row block         8 x 0x23, u64 size, size x {u32 column, u32 value}

`read(path)` parses a file into {row: (size, cells)} (cells: a (size, 2) uint32 array in slot order) and
asserts the structure.  `unreachable(size, cells)` applies the reference's reachability rule: its probe for
a column starts at `column % size` (column 0 at slot 0) and stops at the first empty slot
(column == 0 and value == 0), so every non-empty cell must be found from its home without crossing one.
The reference's loader clears every slot whose value is 0 (:533-540); `cleared(cells)` is what it sees.
"""
from __future__ import annotations

import numpy as np

HEAD = 512
DIR_HEAD = 16
ENTRY = np.dtype([("row", "<u4"), ("off", "<u8")])   # 12 bytes, packed
ROW_HEAD = 16


def read(path: str, min_size: int = 16) -> dict[int, tuple[int, np.ndarray]]:
    """{row: (size, cells)} of every directory entry, after checking the magics, the directory chain (no
    loop, every block inside the file), row blocks inside the file, power-of-two sizes >= min_size,
    no row listed twice and no column twice in a row."""
    d = np.fromfile(path, dtype=np.uint8)
    assert len(d) >= HEAD, "shorter than the header"
    assert (d[:8] == 0x17).all(), "header magic"
    at = int(d[8:16].view("<u8")[0])
    rows: dict[int, tuple[int, np.ndarray]] = {}
    seen = set()
    while at:
        assert at not in seen, "the directory chain loops"
        seen.add(at)
        assert at + DIR_HEAD <= len(d), "directory block past the end of the file"
        entries, nxt = (int(v) for v in d[at:at + 16].view("<u8"))
        assert entries <= 4194304 and at + DIR_HEAD + entries * ENTRY.itemsize <= len(d), "directory block size"
        ents = np.frombuffer(d, ENTRY, entries, at + DIR_HEAD)
        ends = np.flatnonzero(ents["off"] == 0)
        ents = ents[: ends[0] if len(ends) else entries]
        for row, off in zip(ents["row"].tolist(), ents["off"].tolist()):
            assert row not in rows, f"row {row} listed twice"
            assert off + ROW_HEAD <= len(d) and (d[off:off + 8] == 0x23).all(), f"row {row}: block magic"
            size = int(d[off + 8:off + 16].view("<u8")[0])
            assert size >= min_size and size & (size - 1) == 0, f"row {row}: size {size}"
            assert off + ROW_HEAD + 8 * size <= len(d), f"row {row}: block past the end of the file"
            cells = np.frombuffer(d, "<u4", 2 * size, off + ROW_HEAD).reshape(size, 2)
            cols = cells[~empty(cells), 0]
            assert len(np.unique(cols)) == len(cols), f"row {row}: a column twice"
            rows[row] = (size, cells)
        at = nxt
    return rows


def empty(cells: np.ndarray) -> np.ndarray:
    return (cells[:, 0] == 0) & (cells[:, 1] == 0)


def cleared(cells: np.ndarray) -> np.ndarray:
    """The row as the reference's positional load leaves it: slots with value 0 emptied."""
    out = cells.copy()
    out[out[:, 1] == 0] = 0
    return out


def unreachable(size: int, cells: np.ndarray) -> np.ndarray:
    """Columns of the non-empty cells that the reference's probe does not find."""
    occ = ~empty(cells)
    slots = np.flatnonzero(occ)
    if occ.all() or len(slots) == 0:
        return np.zeros(0, np.uint32)
    holes = np.flatnonzero(~occ)
    # run[p] = consecutive non-empty slots ending at p, going backwards (cyclically)
    k = np.searchsorted(holes, slots, side="right") - 1
    prev_hole = np.where(k >= 0, holes[np.maximum(k, 0)], holes[-1] - size)
    run = slots - prev_hole
    cols = cells[slots, 0]
    home = (cols.astype(np.uint64) % np.uint64(size)).astype(np.int64)   # column 0 -> slot 0
    dist = (slots - home) % size
    return cols[dist >= run]


def check_row(row: int, size: int, cells: np.ndarray) -> None:
    """The reachability rule on the row as written, and again as the reference's loader sees it."""
    bad = unreachable(size, cells)
    assert len(bad) == 0, f"row {row}: columns {bad[:8].tolist()} are not found from their home slot"
    bad = unreachable(size, cleared(cells))
    assert len(bad) == 0, f"row {row}: columns {bad[:8].tolist()} are hidden once the zero-valued slots are cleared"


def live(cells: np.ndarray) -> list[tuple[int, int]]:
    """The non-empty cells, sorted by column."""
    c = cells[~empty(cells)]
    return sorted(map(tuple, c.tolist()))
