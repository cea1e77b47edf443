"""SASS evidence for the hand-written kernels: `cuobjdump -sass` of the in-tree extensions (no GPU needed).

    python benchmarks/dump_sass.py            ->  profiles/sass/SUMMARY.md + one listing per selected kernel

SUMMARY.md counts, for EVERY kernel in the four extensions, the instructions that prove which hardware path it uses:
UTCHMMA (tcgen05.mma), UTMALDG / UTMASTG (TMA load / store), UTCBAR (tcgen05.commit), LDTM (tcgen05.ld), SYNCS (mbarrier),
multimem loads / stores (NVLS), vector reductions to global memory, legacy HMMA (must be 0), and the ELECT / BRA.U.ANY
pairs that reveal per-instruction serialisation loops around single-thread instructions.
"""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from b200ddl.ops import _build  # noqa: E402

OUT = os.path.join(ROOT, "profiles", "sass")
COUNT = [("UTCHMMA", r"\bUTCHMMA\b"), ("UTMALDG", r"\bUTMALDG"), ("UTMASTG", r"\bUTMASTG"), ("UTCBAR", r"\bUTCBAR\b"),
         ("LDTM", r"\bLDTM"), ("SYNCS", r"\bSYNCS\."), ("multimem", r"MULTIMEM|\.MMEM|LDGMC|STGMC|REDGMC|\bMM[A-Z]*\.(LD|ST|RED)"),
         ("RED/ATOM.global", r"\b(REDG|RED\.|ATOMG|ATOM\.)"), ("HMMA", r"\bHMMA\b"), ("ELECT", r"\bELECT\b"), ("BRA.U.ANY", r"BRA\.U\.ANY")]
# substrings of demangled names whose full listing is written out
SELECT = ["conv_igemm_kernel<64, 1, true, true>", "conv_igemm_kernel<64, 2, true, true>", "conv_igemm_kernel<256, 1, false, false>",
          "conv_igemm_kernel<256, 2, false, false>", "conv_igemm_kernel<256, 3, false, false>", "conv_igemm_kernel<256, 4, false, false>",
          "allreduce_twoshot_nvls_kernel<(b200::CommDtype)0, 8>", "broadcast_kernel<(b200::CommDtype)0>",
          "softmax_ce_head_kernel", "dwconv3x3_kernel<1>", "dwconv3x3_tiled_kernel<1, 4>", "resize_triangle_batched_kernel", "mbv2_stem_kernel", "weight_prep_batched_kernel", "conv_wgrad_kernel", "stem_fwd_kernel", "stem_wgrad_kernel",
          "allreduce_twoshot_nvls_kernel<(b200::CommDtype)0", "allreduce_sgd_nvls_kernel", "allreduce_twoshot_p2p_kernel<(b200::CommDtype)0, 2>",
          "bn_apply_kernel<true, 1>", "col_reduce_kernel<4>", "bn_bwd_apply_kernel<true>", "sgd_kernel<false>",
          "adam_kernel", "softmax_ce_kernel", "bn_relu_maxpool_fwd_kernel", "tma_probe_kernel", "umma_probe_kernel"]


def demangle(names):
    p = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return p.stdout.split("\n")[:len(names)] if p.returncode == 0 else names


def main():
    os.makedirs(OUT, exist_ok=True)
    for f in os.listdir(OUT):
        os.remove(os.path.join(OUT, f))
    rows, written = [], []
    for ext in _build.EXTENSIONS:
        so = _build.so_path(ext)
        txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
        parts = re.split(r"\n\s*Function : ", txt)[1:]
        names = demangle([p.split("\n")[0].strip() for p in parts])
        for name, body in zip(names, parts):
            ins = [re.sub(r"\s{2,}", "  ", re.sub(r"/\*\s*0x[0-9a-f]{16}\s*\*/", "", l)).rstrip().lstrip()
                   for l in body.split("\n") if re.search(r"/\*[0-9a-f]{4,5}\*/", l)]
            ops = [re.sub(r"^\s*/\*[0-9a-f]{4,5}\*/\s*", "", l).split(";")[0].strip() for l in ins]
            short = re.sub(r"\(.*", "", name).replace("void ", "").replace("b200::", "")
            rows.append((ext, short, len(ops), [sum(bool(re.search(rx, o)) for o in ops) for _, rx in COUNT]))
            if any(s in name for s in SELECT):
                fn = re.sub(r"[^A-Za-z0-9_]+", "_", short).strip("_")[:90] + ".sass"
                with open(os.path.join(OUT, fn), "w") as f:
                    f.write(f"// {name}\n// {ext}.so, sm_100a, {len(ops)} instructions (encodings stripped)\n" + "\n".join(ins) + "\n")
                written.append(fn)
    with open(os.path.join(OUT, "SUMMARY.md"), "w") as f:
        f.write("# SASS summary of the in-tree sm_100a extensions (`python benchmarks/dump_sass.py`)\n\n")
        f.write("Instruction counts per kernel (static occurrences in the SASS).  `UTCHMMA` = tcgen05.mma, `UTMALDG`/`UTMASTG` = TMA, "
                "`UTCBAR` = tcgen05.commit, `LDTM` = tcgen05.ld, `SYNCS` = mbarrier; `HMMA` (legacy mma.sync) must be 0.\n\n")
        f.write("| extension | kernel | instr | " + " | ".join(n for n, _ in COUNT) + " |\n|---|---|---|" + "---|" * len(COUNT) + "\n")
        for ext, short, n, cs in sorted(rows):
            f.write(f"| {ext} | `{short[:110]}` | {n} | " + " | ".join(str(c) if c else "" for c in cs) + " |\n")
        f.write("\nFull listings in this directory: " + ", ".join(f"`{w}`" for w in sorted(set(written))) + "\n")
    print(f"{len(rows)} kernels summarised, {len(set(written))} listings written to {OUT}")


if __name__ == "__main__":
    main()
