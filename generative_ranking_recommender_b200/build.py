"""In-tree build of librqk_sm100a.so (nvcc, sm_100a only).  Used by __graft_entry__.build() and as
`python -m generative_ranking_recommender_b200.build`."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librqk_sm100a.so")
SOURCES = ["rqk_api.cu", "score_simt.cu", "score_tc.cu", "auction.cu", "centroid.cu", "residual.cu", "encode.cu", "encode_fused.cu", "seed_draw.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-rdc=false",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building librqk_sm100a.so")
    subprocess.check_call([nvcc, "-shared", "-o", LIB, *objs, "-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
