"""Builds libkanzi_b200.so (CUDA kernels + C ABI) in-tree for sm_100a with nvcc. No GPU is needed to build."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libkanzi_b200.so")
SOURCES = ["kz_ans.cu", "kz_ans1.cu", "kz_huffman.cu", "kz_range.cu", "kz_hash.cu", "kz_sbrt.cu", "kz_zrlt.cu", "kz_rolz.cu", "kz_alias.cu", "kz_fsd.cu", "kz_text.cu", "kz_text_par.cu", "kz_utf.cu", "kz_exe.cu", "kz_bwt.cu", "kz_lz.cu", "kz_lz_par.cu", "kz_lz_inv.cu", "kz_concat.cu", "kz_api.cu"]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared",
         "-Xptxas", "-v"]


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    for root in (CSRC, os.path.join(CSRC, "_gen"), os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h", ".cpp", ".inc")) and os.path.getmtime(os.path.join(root, f)) > t:
                return True
    return False


def build(force=False, verbose=False):
    # TEXT's static dictionary is a constant of the kanzi format: csrc/_gen/ is generated from tests/golden/text_dict_en_1024.txt
    import importlib.util

    spec = importlib.util.spec_from_file_location("kz_gen_text_dict", os.path.join(HERE, "gen_text_dict.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.main()
    if not force and not needs_build():
        return OUT
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    tmp = OUT + ".tmp"  # link into a temporary name, then rename: the library never exists half written
    cmd = ["nvcc"] + FLAGS + srcs + ["-o", tmp]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed")
    os.replace(tmp, OUT)
    with open(os.path.join(HERE, "ptxas_info.txt"), "w") as f:
        f.write("".join(ln for ln in r.stderr.splitlines(True) if "Compile time" not in ln))  # registers / spills / smem per kernel of this build (git-ignored)
    return OUT


if __name__ == "__main__":
    build(force=True, verbose=True)
    print(OUT)
