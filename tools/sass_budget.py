#!/usr/bin/env python3
"""Static SASS instruction budget of the stream kernels' transform (no GPU needed).

Builds the library (from the working tree, or from a git revision with --rev) with -Xptxas -v, disassembles it with
cuobjdump / nvdisasm (source line info with inlining) and, for every default (fp16-storage) stream-kernel instantiation
of capi.cu, reports

  * registers, the register cap its thread count and __launch_bounds__ allow, and spills;
  * for the ring-path kernels: the SASS of the transform's interior-tile code per 8 elements (one 16-byte chunk),
    split into arithmetic, memory and control / addressing (everything else), with the most frequent opcodes of the
    last class.

The interior-tile code is found through the line info: every instruction whose inline chain passes through the one
source line of conv_stream.cuh that transforms a chunk of an interior tile (`interior_chunk(k)`; `chunk(id, true)` up
to 445bc78).  If those instructions form a loop (a backward branch inside them), the loop body is counted, i.e. the
steady state; otherwise the whole straight-line address range they span.  Chunks in the counted code = STS.128 into the A stage / (2 with split
hi / lo operands, else 1).

    python tools/sass_budget.py [--rev GIT_REV] [--out FILE]
"""
from __future__ import annotations

import argparse
import collections
import re
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

REPO = Path(__file__).resolve().parent.parent
CUDA = Path("/usr/local/cuda/bin")
PRO = {"PRO_NORM": 1, "PRO_NORM_RES": 2, "PRO_FIR": 3, "PRO_NORM_RES_X": 4}
ARITH = {"FFMA", "FFMA2", "FMUL", "FMUL2", "FADD", "FADD2", "MUFU", "FMNMX", "FMNMX2", "F2FP", "HADD2", "HFMA2",
         "HMUL2", "HMNMX2", "F2F"}
MEMORY = {"LDS", "STS", "LDG", "STG", "LD", "ST", "LDL", "STL", "LDSM", "ATOMS", "ATOMG", "RED"}
INTERIOR_CALL = re.compile(r"\bchunk\(id, true\)|\binterior_chunk\(k\)")


def tool(name: str) -> str:
    p = shutil.which(name) or str(CUDA / name)
    if not Path(p).exists():
        raise SystemExit(f"{name} not found")
    return p


def source_tree(rev: str | None, tmp: Path) -> Path:
    if rev is None:
        return REPO
    dst = tmp / "src"
    dst.mkdir()
    arch = subprocess.run(["git", "-C", str(REPO), "archive", rev], check=True, capture_output=True).stdout
    subprocess.run(["tar", "-x", "-C", str(dst)], input=arch, check=True)
    return dst


def build(src: Path, tmp: Path) -> tuple[Path, str]:
    lib = tmp / "lib.so"
    cmd = [tool("nvcc"), "-Xptxas=-v", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "1886,177", "-o", str(lib),
           str(src / "wav2sleep_b200" / "csrc" / "capi.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise SystemExit(f"nvcc failed:\n{res.stderr[-4000:]}")
    return lib, res.stderr


def disassemble(lib: Path, tmp: Path) -> str:
    subprocess.run([tool("cuobjdump"), "-xelf", "all", str(lib)], cwd=tmp, check=True, capture_output=True)
    cubins = sorted(tmp.glob("*.sm_100a.cubin"))
    if not cubins:
        raise SystemExit("no sm_100a cubin in the library")
    return subprocess.run([tool("nvdisasm"), "-gi", "-c", str(cubins[0])], check=True, capture_output=True,
                          text=True).stdout


def default_stream_kernels(src: Path) -> list[dict]:
    """The W2S_STREAM(...) lines of capi.cu: default fp16-storage instantiations."""
    out = []
    pat = re.compile(r"^\s*W2S_STREAM\((\d+), (\d+), (\d), (PRO_\w+), (true|false), (\d+), (\d+), (\d+), (\d+)\)")
    for line in (src / "wav2sleep_b200" / "csrc" / "capi.cu").read_text().splitlines():
        m = pat.match(line)
        if not m:
            continue
        cin, cout, s, pro, ds, mt, nr, na, ntw = m.groups()
        cin, cout, ntw = int(cin), int(cout), int(ntw)
        k = dict(cin=cin, cout=cout, stride=int(s), pro=pro, ds=ds == "true", mt=int(mt), nr=int(nr), na=int(na),
                 ntw=ntw, split=cin <= 16 and cout <= 16)
        k["mangled"] = ("_ZN3w2s18conv_stream_kernelILi{cin}ELi{cout}ELi{stride}ELi{p}ELb{ds}ELb{sp}ELi{mt}ELi{nr}ELi{na}"
                        "ELi{ntw}ELb0ELb0EEEvNS_8ConvArgsENS_10ConvGroup2Eii").format(
            p=PRO[pro], sp=int(k["split"]), **{**k, "ds": int(k["ds"])})
        threads = 32 * (6 + ntw)
        k["threads"] = threads
        k["reg_cap"] = min(255, (65536 // (threads * (2 if threads <= 384 else 1))) // 8 * 8)
        out.append(k)
    return out


def ptxas_info(log: str) -> dict[str, dict]:
    info, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur = m.group(1)
            info[cur] = {}
            continue
        if cur is None:
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m:
            info[cur]["spill_st"], info[cur]["spill_ld"] = int(m.group(1)), int(m.group(2))
        m = re.search(r"Used (\d+) registers", line)
        if m:
            info[cur]["regs"] = int(m.group(1))
    return info


def function_sass(dis: str, mangled: str) -> list[tuple[str | None, str, tuple[tuple[str, int], ...], str]]:
    """(label, opcode, inline chain of (file, line), text) of every instruction of one kernel."""
    head = f".text.{mangled}"
    start = dis.find(f"//--------------------- {head} ")
    if start < 0:
        raise SystemExit(f"{mangled} not in the disassembly")
    end = dis.find("//---------------------", start + 10)
    body = dis[start:end if end > 0 else len(dis)]
    insts, chain, pending, label = [], (), [], None
    for line in body.splitlines():
        s = line.strip()
        m = re.match(r"^(\.L_x_\d+):$", s)
        if m:
            label = m.group(1)
            continue
        if s.startswith("//##"):
            m = re.match(r'//## File "([^"]+)", line (\d+)', s)
            if m:
                pending.append((Path(m.group(1)).name, int(m.group(2))))
            continue
        m = re.match(r"/\*([0-9a-f]+)\*/\s+(.*?);", s)
        if not m:
            continue
        if pending:
            chain, pending = tuple(pending), []
        text = m.group(2).strip()
        op = re.sub(r"^@!?U?P\w+\s+", "", text).split()[0]
        insts.append((label, op, chain, text))
        label = None
    return insts


def interior_lines(src: Path) -> set[int]:
    lines = (src / "wav2sleep_b200" / "csrc" / "conv_stream.cuh").read_text().splitlines()
    hits = {i + 1 for i, t in enumerate(lines) if INTERIOR_CALL.search(t) and not t.strip().startswith("//")}
    if len(hits) != 1:
        raise SystemExit(f"expected one interior-tile chunk call in conv_stream.cuh, found lines {sorted(hits)}")
    return hits


def budget(insts, marker: set[int], split: bool) -> dict | None:
    idx = [i for i, (_, _, ch, _) in enumerate(insts) if any(f == "conv_stream.cuh" and ln in marker for f, ln in ch)]
    if not idx:
        return None
    lo, hi = idx[0], idx[-1]
    at = {lab: i for i, (lab, _, _, _) in enumerate(insts) if lab}
    loop = None
    for i in range(lo, hi + 1):  # backward branches inside the interior code: take the widest loop
        _, op, _, text = insts[i]
        m = re.search(r"\((\.L_x_\d+)\)", text) if op == "BRA" else None
        if m and m.group(1) in at and lo <= at[m.group(1)] < i:
            if loop is None or at[m.group(1)] < loop[0]:
                loop = (at[m.group(1)], i)
    b0, b1 = loop if loop else (lo, hi)
    ops = [insts[i][1] for i in range(b0, b1 + 1)]
    base = [o.split(".")[0] for o in ops]
    sts128 = sum(1 for o in ops if o.startswith("STS.128"))
    chunks = sts128 / (2 if split else 1)
    if chunks == 0:
        return None
    cls = collections.Counter("arith" if b in ARITH else "memory" if b in MEMORY else "other" for b in base)
    other = collections.Counter(b for b in base if b not in ARITH and b not in MEMORY)
    return dict(form="loop" if loop else "straight", n=len(ops), chunks=chunks,
                arith=cls["arith"] / chunks, memory=cls["memory"] / chunks, other=cls["other"] / chunks,
                other_ops=other, arith_ops=collections.Counter(b for b in base if b in ARITH))


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rev", default=None, help="git revision to build instead of the working tree")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory(prefix="sass_budget_") as t:
        tmp = Path(t)
        src = source_tree(args.rev, tmp)
        lib, log = build(src, tmp)
        dis = disassemble(lib, tmp)
        regs = ptxas_info(log)
        marker = interior_lines(src)
        kernels = default_stream_kernels(src)
    head = subprocess.run(["git", "-C", str(REPO), "rev-parse", "--short", args.rev or "HEAD"], capture_output=True,
                          text=True).stdout.strip()
    rev = head if args.rev else f"working tree on {head}"
    rows = [f"# SASS budget of the stream kernels' transform, sm_100a, source: {rev}",
            "# per 8 elements (one 16-byte chunk) of the interior-tile transform; arith = FFMA/FFMA2/FMUL2/FADD2/MUFU/"
            "FMNMX/F2FP/HADD2...,",
            "# memory = LDS/STS/LDG/STG..., other = control / addressing / predicates / conversions / everything else",
            f"{'kernel':44s} {'thr':>4s} {'regs':>4s} {'cap':>4s} {'spill':>7s} {'form':>8s} {'arith':>6s} {'mem':>5s} "
            f"{'other':>6s} {'total':>6s}  top 'other' opcodes"]
    mixes = []
    for k in kernels:
        name = f"<{k['cin']},{k['cout']},s{k['stride']},{k['pro']}{',ds' if k['ds'] else ''},MT{k['mt']},NR{k['nr']},NTW{k['ntw']}>"
        r = regs.get(k["mangled"], {})
        spill = f"{r.get('spill_st', '?')}/{r.get('spill_ld', '?')}"
        line = f"{name:44s} {k['threads']:4d} {r.get('regs', 0):4d} {k['reg_cap']:4d} {spill:>7s}"
        b = None if k["nr"] == 0 else budget(function_sass(dis, k["mangled"]), marker, k["split"])
        if b is None:
            line += f" {'direct' if k['nr'] == 0 else '-':>8s}"
        else:
            tot = b["arith"] + b["memory"] + b["other"]
            top = " ".join(f"{o}:{c / b['chunks']:.1f}" for o, c in b["other_ops"].most_common(8))
            line += f" {b['form']:>8s} {b['arith']:6.1f} {b['memory']:5.1f} {b['other']:6.1f} {tot:6.1f}  {top}"
            mix = " ".join(f"{o}:{c / b['chunks']:.1f}" for o, c in sorted(b["arith_ops"].items()))
            mixes.append(f"{name:44s} {mix}")
        rows.append(line)
    rows.append("# arithmetic opcodes per 8 elements:")
    rows += mixes
    text = "\n".join(rows)
    print(text)
    if args.out:
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    sys.exit(main())
