"""Write the full SASS of every hot kernel of ops/_C.so, gz-compressed, under profiles/sass/ plus an index with the
tensor-core / TMA / multimem mnemonic counts per kernel (the evidence the north star asks for: UTC*MMA = tcgen05.mma,
LDTM/STTM = tcgen05.ld/st, UTMALDG/UTMASTG = TMA, UTCCP = tcgen05.cp, LDGMC/STGMC... = multimem).

    python tools/dump_sass.py            # after `python -m bert_pytorch_b200.ops.build`
"""
import gzip
import os
import re
import subprocess
import sys
from collections import Counter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "bert_pytorch_b200", "ops", "_C.so")
OUT = os.path.join(ROOT, "profiles", "sass")
HOT = ["gemm_pair_kernel", "gemm_kernel", "gemm_mx", "attn_fwd_row_kernel", "attn_fwd_stream_kernel",
       "attn_bwd_pipe_kernel", "ln_fwd_row_kernel", "ln_bwd3_kernel",
       "fused_allreduce_lamb_kernel", "peer_allreduce_kernel", "lamb_stage1_kernel", "lamb_stage2_kernel",
       "softmax_ce_kernel", "embed_fwd_kernel", "embed_bwd_scatter_kernel", "nsp_head_kernel", "colsum_finalize_kernel",
       "kfac_", "dropout_mask_kernel", "attn_bwd_row2_kernel", "colsum_bf16_kernel"]
MNEMONICS = ["UTCHMMA", "UTCQMMA", "UTCOMMA", "UTCCP", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UTMAREDG", "UBLKCP", "LDGMC",
             "STGMC", "MULTIMEM", "RED", "HMMA", "SYNCS", "UTCBAR", "FFMA2", "FMUL2", "FADD2"]


def main():
    os.makedirs(OUT, exist_ok=True)
    txt = subprocess.run(["cuobjdump", "-sass", SO], capture_output=True, text=True, check=True).stdout
    parts = re.split(r"(?m)^\s*Function : ", txt)
    index = []
    for part in parts[1:]:
        name = part.split("\n", 1)[0].strip()
        if not any(h in name for h in HOT):
            continue
        demangled = subprocess.run(["cu++filt", name], capture_output=True, text=True).stdout.strip() or name
        short = re.sub(r"\(CUtensorMap.*|\((?!bool|int)[^<]*$", "", demangled).replace("b200::", "").replace("void ", "")
        short = re.sub(r"\(bool\)|\(int\)", "", short)
        short = re.sub(r"\(.*", "", short) if "<" not in short else short
        short = re.sub(r"[^A-Za-z0-9_<>,]+", "_", short).strip("_")[:90]
        ops = Counter()
        n_instr = 0
        for line in part.split("\n"):
            m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
            if m:
                n_instr += 1
                base = m.group(1).split(".")[0]
                for k in MNEMONICS:
                    if base.startswith(k):
                        ops[m.group(1) if k in ("UTCHMMA", "UTCQMMA", "UTCOMMA") else k] += 1
        path = os.path.join(OUT, short.replace("<", "_").replace(">", "_").replace(",", "_") + ".sass.gz")
        with gzip.open(path, "wt") as f:
            f.write("Function : " + part)
        index.append((short, n_instr, dict(ops), os.path.basename(path)))
    with open(os.path.join(OUT, "INDEX.md"), "w") as f:
        f.write("# SASS of the hot sm_100a kernels (cuobjdump -sass of bert_pytorch_b200/ops/_C.so, one .sass.gz per kernel)\n\n")
        f.write("| kernel | instructions | tensor-core / TMA / peer mnemonics | file |\n|---|---|---|---|\n")
        for short, n, ops, fn in sorted(index, key=lambda e: e[0]):
            f.write(f"| `{short}` | {n} | {', '.join(f'{k} {v}' for k, v in sorted(ops.items())) or '-'} | {fn} |\n")
    print(f"{len(index)} kernels -> {OUT}")


if __name__ == "__main__":
    main()
