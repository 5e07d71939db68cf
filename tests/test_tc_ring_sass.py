"""CPU test (no GPU): the converter warps of the tensor-core sampler kernels release a Y ring slot only after their reads of
it have been performed, read in the machine code nvcc makes of gemm_tc.cu with the library's flags.

k_l1_fwd_ts and k_l1_bwd_ts stream raw Y tiles through a ring of shared-memory slots.  The TMA writes a slot through the
async proxy and completes its `yfull` barrier; the converter warps read the tile with generic-proxy loads and arrive on the
slot's `yempty` barrier, after which the TMA may refill the slot at once.  An arrive does not wait for earlier loads by
itself, so a load still in flight when the TMA overwrites the slot returns bytes of the next fill: a wrong gradient or
activation with no fault and no error, seen only when a CTA walks more tiles than the ring holds (0f26c18 found exactly
this in k_l1_fwd_ts).  Two things hold the arrive back:

- k_l1_fwd_ts has a proxy fence before the arrive (`fence.proxy.async.shared::cta`, MEMBAR + FENCE.VIEW.ASYNC in SASS):
  the arrive issues only once the loads have been performed.  Removing it brings the race back.
- k_l1_bwd_ts has no fence.  It is safe because every register its loads write is read (scaled by dz) before the arrive,
  and the SM issues in order, so the arrive waits on the scoreboard of every load.  Nothing in the source pins that: a
  compile that scheduled the arrive above a consumer, or a source edit that released the slot before the conversion
  loop, would make the backward read the next fill.  The test accepts a MEMBAR instead of the consumers.

The barriers are found by the offsets the kernels' barrier layouts give them: in k_l1_fwd_ts yfull = bars + 32 and
yempty = bars + 40 (bytes 0x100, 0x140); in k_l1_bwd_ts yfull = bars + 10 and yempty = bars + 18 (bytes 0x50, 0x90),
which SASS addresses past the 64 KB of mask stages in front of the Y ring (0x10050, 0x10090).  Only the low 16 bits of the
immediate are compared.  The converter path is the straight-line code from the last yfull try-wait before an arrive to
the arrive."""
import os
import re
import subprocess

import pytest

from test_step_tail_sass import _tool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FWD_TS = ("_Z11k_l1_fwd_tsILb0ELb0E", "_Z11k_l1_fwd_tsILb0ELb1E", "_Z11k_l1_fwd_tsILb1ELb0E", "_Z11k_l1_fwd_tsILb1ELb1E")
BWD_TS = "_Z11k_l1_bwd_ts"
BARS = {"fwd": (0x100, 0x140), "bwd": (0x50, 0x90)}        # (yfull[0], yempty[0]) byte offsets from bars
RING = 8                                                     # slots of both barrier arrays

_INSN = re.compile(r"/\*[0-9a-f]{4,}\*/\s+(@!?U?P(?:\d|T)\s+)?([A-Z][A-Z0-9_.]*)\s*(.*?)\s*;")
_BAR_ADDR = re.compile(r"\[[^\]]*?(?:\+0x([0-9a-f]+))?\]")
_REG = re.compile(r"\bR(\d+)(?:\.64)?\b")


def _functions(sass):
    return {m.group(1): m.group(2)
            for m in re.finditer(r"Function : (\S+)\n(.*?)(?=\n\s*Function :|\Z)", sass, re.S)}


def _insns(body):
    """[(opcode, operand text)] in address order"""
    return [(m.group(2), m.group(3)) for m in _INSN.finditer(body)]


def _bar_offset(ops):
    m = _BAR_ADDR.search(ops)
    return int(m.group(1), 16) & 0xFFFF if m and m.group(1) else 0


def _is_bar(op, ops, kind, base):
    return op.startswith(kind) and base <= _bar_offset(ops) < base + 8 * RING


def _converter_paths(insns, which):
    """for every yempty arrive: the instructions from the last yfull try-wait before it up to the arrive"""
    yfull, yempty = BARS[which]
    out = []
    for i, (op, ops) in enumerate(insns):
        if not _is_bar(op, ops, "SYNCS.ARRIVE", yempty):
            continue
        j = i - 1
        while j >= 0 and not _is_bar(*insns[j], "SYNCS.PHASECHK", yfull):
            j -= 1
        assert j >= 0, f"yempty arrive #{len(out)} has no yfull try-wait before it"
        out.append(insns[j + 1:i])
    return out


def _load_dests(op, ops):
    """registers a generic or shared-memory load writes (LD.E.128 R4 -> R4..R7)"""
    if not re.match(r"LDS?(\.|$)", op):
        return []
    m = re.match(r"R(\d+)", ops)
    if not m:
        return []
    width = 4 if ".128" in op else 2 if ".64" in op else 1
    return [int(m.group(1)) + w for w in range(width)]


def _sources(ops):
    """registers an instruction reads: every register operand but the first (the destination), and all of them inside an
    address; a .64 register names a pair"""
    regs = set()
    first = ops.split(",")[0]
    rest = ops[len(first):]
    for part in [rest] + re.findall(r"\[[^\]]*\]", first):
        for m in _REG.finditer(part):
            r = int(m.group(1))
            regs.add(r)
            if m.group(0).endswith(".64"):
                regs.add(r + 1)
    return regs


@pytest.fixture(scope="module")
def sass(tmp_path_factory):
    nvcc, cuobjdump = _tool("nvcc"), _tool("cuobjdump")
    if not nvcc or not cuobjdump:
        pytest.skip("nvcc / cuobjdump not available")
    from grapes_b200.build import NVCC_FLAGS
    cubin = str(tmp_path_factory.mktemp("ring_sass") / "gemm_tc.cubin")
    subprocess.run([nvcc] + NVCC_FLAGS + ["-cubin", "-o", cubin, os.path.join(ROOT, "grapes_b200", "csrc", "gemm_tc.cu")],
                   check=True, capture_output=True)
    return _functions(subprocess.run([cuobjdump, "-sass", cubin], check=True, capture_output=True, text=True).stdout)


def test_bwd_ts_converters_consume_every_load_before_releasing_the_slot(sass):
    names = [n for n in sass if n.startswith(BWD_TS)]
    assert len(names) == 1, names
    paths = _converter_paths(_insns(sass[names[0]]), "bwd")
    assert paths, "k_l1_bwd_ts: no arrive on a yempty barrier"
    for p, path in enumerate(paths):
        pending = {}                          # register -> index of the load that wrote it, not yet read
        last_load = -1
        for i, (op, ops) in enumerate(path):
            for r in _sources(ops):
                pending.pop(r, None)
            if op.startswith("MEMBAR") and i > last_load:
                pending.clear()
            for r in _load_dests(op, ops):
                pending[r] = i
                last_load = i
        assert last_load >= 0, (f"k_l1_bwd_ts arrive #{p}: no load of the tile between the yfull wait and the yempty "
                                f"arrive -- the slot is released before it is read")
        assert not pending, (f"k_l1_bwd_ts arrive #{p}: the loads into " + ", ".join(f"R{r}" for r in sorted(pending)) +
                             " are read by nothing before the yempty arrive and no MEMBAR holds it back")


def test_fwd_ts_converters_fence_before_releasing_the_slot(sass):
    for name in FWD_TS:
        full = [n for n in sass if n.startswith(name)]
        assert len(full) == 1, (name, full)
        paths = _converter_paths(_insns(sass[full[0]]), "fwd")
        assert paths, f"{full[0]}: no arrive on a yempty barrier"
        for p, path in enumerate(paths):
            ops = [op for op, _ in path]
            loads = [i for i, (op, o) in enumerate(path) if _load_dests(op, o)]
            assert loads, f"{full[0]} arrive #{p}: no load of the tile between the yfull wait and the yempty arrive"
            after = ops[loads[-1] + 1:]
            membar = next((i for i, op in enumerate(after) if op.startswith("MEMBAR")), None)
            assert membar is not None, f"{full[0]} arrive #{p}: no MEMBAR between the last tile load and the yempty arrive"
            assert any(op.startswith("FENCE.VIEW.ASYNC") for op in after[membar + 1:]), \
                f"{full[0]} arrive #{p}: no FENCE.VIEW.ASYNC after the MEMBAR, before the yempty arrive"
