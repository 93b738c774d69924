"""Host checks of the time-series plumbing (mdproptools_b200/dynamical/series.py): the per-group rank split, the molecule
layout, the lag rule, the batch form of the frame merge under two gloo ranks, and the input errors raised before any frame
is parsed."""
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import MASS, NUM_ATOMS, NUM_MOLS, ROOT


def test_rank_blocks_split_every_group_into_disjoint_contiguous_blocks():
    from mdproptools_b200 import dist
    from mdproptools_b200.dynamical.series import rank_blocks
    rng = np.random.default_rng(3)
    sizes = [0, 1, 2, 7, 100]
    members = [np.sort(rng.choice(10 ** 6, n, replace=False)) for n in sizes]         # non-contiguous indices
    for w in range(1, 6):
        seen = [[] for _ in sizes]
        for r in range(w):
            sel, counts = rank_blocks(members, "cpu", r, w)
            sel = sel.numpy()
            assert sel.dtype == np.int64 and counts == [len(range(*dist.shard_range(n, r, w))) for n in sizes]
            parts = np.split(sel, np.cumsum(counts)[:-1])
            for g, (idx, part) in enumerate(zip(members, parts)):                       # group order
                lo, hi = dist.shard_range(len(idx), r, w)
                assert np.array_equal(part, idx[lo:hi]), (w, r, g)
                seen[g].append(part)
        for g, idx in enumerate(members):                                               # disjoint and covering
            got = np.concatenate(seen[g])
            assert np.array_equal(got, idx) and len(np.unique(got)) == len(idx), (w, g)


def test_molecule_layout_matches_membership_and_checks_atom_count():
    from mdproptools_b200.common.com_mols import atom_masses, mol_membership
    from mdproptools_b200.dynamical.series import MoleculeLayout
    for num_mols, num_atoms in ((NUM_MOLS, NUM_ATOMS), ([2, 3], [2, 1]), ([0, 4, 1], [3, 2, 5])):
        lay = MoleculeLayout(num_mols, num_atoms, MASS)
        for a, b in zip((lay.mol_type, lay.mol_id, lay.seg_off), mol_membership(num_mols, num_atoms)):
            assert np.array_equal(a, b)
        assert lay.type_off.dtype == np.int64
        assert np.array_equal(lay.type_off, np.concatenate(([0], np.cumsum(num_mols))).astype(np.int64))
        assert [m.tolist() for m in lay.type_members()] == [list(range(lay.type_off[g], lay.type_off[g + 1]))
                                                             for g in range(len(num_mols))]
        n = int(np.dot(num_mols, num_atoms))
        lay.check(n)
        for bad in (n - 1, n + 1):
            with pytest.raises(ValueError, match=rf"^Length of values \({n}\) does not match length of index \({bad}\)$"):
                lay.check(bad)
    types = np.array([1.0, 9.0, 3.0, 3.0])
    row = np.array([2.0, 4.0, 6.0, 8.0])
    assert np.array_equal(MoleculeLayout([1], [4], MASS).masses(types, row), atom_masses(types, MASS))
    got = MoleculeLayout([1], [4]).masses(types, row)
    assert np.array_equal(got, row) and got is not row and got.dtype == np.float64


@pytest.mark.parametrize("max_lag, want", [(None, 5), (0, None), (1, 1), (11, 11), (16, 11)])
def test_lag_count(max_lag, want):
    from mdproptools_b200.dynamical.series import lag_count
    if want is None:
        with pytest.raises(ValueError, match=r"max_lag must be at least 1 \(11 frames\)"):
            lag_count(max_lag, 11)
    else:
        assert lag_count(max_lag, 11) == want
    with pytest.raises(ValueError, match=r"max_lag must be at least 1 \(1 frames\)"):
        lag_count(None, 1)


_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as d
d.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
from mdproptools_b200.common.frames import _merge_frames
r = d.get_rank()
T, G = 11, 4
rng = np.random.default_rng(9)
full = torch.from_numpy(rng.normal(size=(3, G, T)))           # [3, G, T] per-frame results, frame axis last
steps = torch.from_numpy(rng.integers(0, 10 ** 9, T).astype(np.float64))
mine = [i for i in range(T) if i % 2 == r]                     # round-robin frames, in batches of up to 3
batches = [tuple(mine[k:k + 3]) for k in range(0, len(mine), 3)]
got = _merge_frames({{b: full[:, :, list(b)].permute(2, 0, 1) for b in batches}}, T, (3, G), torch.device("cpu"),
                    torch.float64).permute(1, 2, 0)
assert got.numpy().tobytes() == full.numpy().tobytes()
got = _merge_frames({{b: steps[list(b)] for b in batches}}, T, (), torch.device("cpu"), torch.float64)
assert got.numpy().tobytes() == steps.numpy().tobytes()
got = _merge_frames({{i: int(steps[i]) for i in mine}}, T, (), torch.device("cpu"))        # single frames, int64
assert got.tolist() == [int(s) for s in steps]
d.destroy_process_group()
print("rank", r, "ok")
"""


def test_two_rank_gloo_batch_merge(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER.format(root=ROOT))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29613", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.count("ok") == 2


def _frames(path, columns, rows, steps=(0, 10)):
    with open(path, "w") as f:
        for s in steps:
            f.write(f"ITEM: TIMESTEP\n{s}\nITEM: NUMBER OF ATOMS\n{len(rows)}\nITEM: BOX BOUNDS pp pp pp\n0 9\n0 9\n0 9\n"
                    f"ITEM: ATOMS {columns}\n" + "".join(" ".join(map(str, row)) + "\n" for row in rows))


def test_errors_before_any_frame_is_parsed(tmp_path):
    """A pattern without files: "no dump frames found" also from the charge flux without a mass table.  A com MSD without
    masses: the mass assertion before the reader is asked for the column.  Neither gets to a device."""
    from mdproptools_b200.dynamical.conductivity import Conductivity
    from mdproptools_b200.dynamical.diffusion import Diffusion
    c = Conductivity("dump.none.*.dump", [1], [2], volume=1000.0, working_dir=str(tmp_path))
    for method in ("get_charge_flux", "calc_cond"):
        with pytest.raises(ValueError, match="no dump frames found"):
            getattr(c, method)()
    _frames(tmp_path / "dump.nomass.lammpstrj", "id type xu yu zu vx vy vz", [(1, 1, 0.5, 0.5, 0.5, 0.1, 0.2, 0.3),
                                                                              (2, 1, 1.5, 1.5, 1.5, 0.1, 0.2, 0.3)])
    d = Diffusion(outputs_dir=str(tmp_path), diff_dir=str(tmp_path))
    com = dict(msd_type="com", num_mols=[1], num_atoms_per_mol=[2])
    for call in (lambda: d.get_msd_from_dump("dump.nomass.lammpstrj", **com),
                 lambda: d.get_msd_all_origins("dump.nomass.lammpstrj", **com),
                 lambda: d.get_vacf("dump.nomass.lammpstrj", vacf_type="com", num_mols=[1], num_atoms_per_mol=[2])):
        with pytest.raises(AssertionError, match="Missing atom masses in dump file."):
            call()
    with pytest.raises(AssertionError, match="Missing atom masses in dump file."):
        Conductivity("dump.nomass.lammpstrj", [1], [2], volume=1000.0, working_dir=str(tmp_path)).get_charge_flux()
