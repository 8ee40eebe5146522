"""tools/gen_fe_ptx.py, the generator of the device's fe_mul / fe_sq PTX (elastic_elgamal_b200/csrc/fe_ptx.cuh): its
PTX-subset interpreter agrees with Python big integers on edge and random operands for both 2^256 = 38 folds, and the
committed fe_ptx.cuh is what the generator produces."""
import importlib.util
import pathlib
import re
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
GEN = ROOT / "tools" / "gen_fe_ptx.py"
COMMITTED = ROOT / "elastic_elgamal_b200" / "csrc" / "fe_ptx.cuh"


def test_generated_sequences_match_big_integers():
    spec = importlib.util.spec_from_file_location("gen_fe_ptx", GEN)
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    for fold in (gen.fold, gen.fold_shift):      # the default fold and the EG_FE_SHIFT_FOLD variant
        gen.FOLD = fold
        gen.check(2000)                          # every pair of its edge operands (2^256 - 1, p, 2^256 - 38, ...) + random


def lines(text):
    """The generator declares its internal registers in set order, which varies between runs: `.reg` lines compare as sets
    of names, every other line exactly."""
    out = []
    for line in text.splitlines():
        m = re.search(r"\.reg \.u32 ([^;]*);", line)
        out.append(frozenset(n.strip() for n in m.group(1).split(",")) if m else line)
    return out


def test_committed_fe_ptx_is_generated(tmp_path):
    out = tmp_path / "fe_ptx.cuh"
    subprocess.run([sys.executable, str(GEN), "--out", str(out)], check=True, stdout=subprocess.DEVNULL)
    new, committed = lines(out.read_text()), lines(COMMITTED.read_text())
    diff = [i + 1 for i, (a, b) in enumerate(zip(new, committed)) if a != b]
    assert len(new) == len(committed) and not diff, f"fe_ptx.cuh differs from the generator's output at lines {diff[:8]}"
