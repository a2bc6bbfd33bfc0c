"""Build the REFERENCE's qigen CPU kernel (cQIGen) into oracle/_ref/cQIGen/ - the compiled CPU baseline SURVEY 8d asks for.

    python oracle/build_qigen.py [threads]

The reference generates its C++ backend with `autogptq_extension/qigen/generate.py` (it writes next to itself, so the
generator runs on a writable scratch copy in a temporary directory - nothing of the reference is copied into this
repository) and bakes the OpenMP thread count in at generation time (`--p`; default 16 = the host cores of the GPU boxes of this pool).  `gekko`
(an optimiser the generator imports for its --search mode) is absent here: a stand-in whose solve() raises sends
`mem_model` to its own closed-form fallback (qlinear_qigen.py:71-87), as SURVEY Appendix B3 verified.
-march=native of the reference's setup.py:197 becomes x86-64-v3 (AVX2 + FMA, what the generated intrinsics use): the
library is built in this container and runs on the GPU box's host.  TEST/BENCH INFRASTRUCTURE: never imported by the product.
"""
import os
import shutil
import subprocess
import sys
import tempfile

REF = "/root/reference/autogptq_extension/qigen"
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref", "cQIGen")


def main():
    if not os.path.isdir(REF):
        sys.exit("reference tree not present (the GPU box only uses the prebuilt oracle/_ref)")
    threads = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    with tempfile.TemporaryDirectory(prefix="agb200_qigen_") as work:
        build(threads, work)


def build(threads, work):
    os.makedirs(os.path.join(work, "autogptq_extension"))
    # file modes are not copied: the sources may be read-only, and the generator writes next to itself
    shutil.copytree(REF, os.path.join(work, "autogptq_extension", "qigen"), copy_function=shutil.copyfile)
    for d, _, _ in os.walk(work):
        os.chmod(d, 0o755)
    stub = os.path.join(work, "stubs", "gekko")
    os.makedirs(stub)
    with open(os.path.join(stub, "__init__.py"), "w") as f:
        f.write("class _V:\n"
                "    def __init__(self, *a, **k): self.value = [1]\n"
                "    def __getattr__(self, n): return _V()\n"
                "    def __call__(self, *a, **k): return _V()\n"
                "    def __mul__(self, o): return _V()\n"
                "    __rmul__ = __add__ = __radd__ = __mul__\n"
                "    def __eq__(self, o): return _V()\n"
                "    __hash__ = None\n"
                "class GEKKO(_V):\n"
                "    def solve(self, *a, **k): raise RuntimeError('gekko stand-in: no solver')\n")
    env = dict(os.environ, PYTHONPATH=os.path.join(work, "stubs") + os.pathsep + os.path.join(work, "autogptq_extension", "qigen"))
    subprocess.run([sys.executable, "autogptq_extension/qigen/generate.py", "--module", "--p", str(threads)], cwd=work, env=env, check=True)
    from torch.utils import cpp_extension

    os.environ["CXX"] = "/usr/bin/g++"      # the toolchain whose libgomp is installed
    os.makedirs(OUT, exist_ok=True)
    cpp_extension.load(name="cQIGen", sources=[os.path.join(work, "autogptq_extension", "qigen", "backend.cpp")],
                       extra_cflags=["-O3", "-mavx", "-mavx2", "-mfma", "-march=x86-64-v3", "-ffast-math", "-ftree-vectorize",
                                     "-faligned-new", "-std=c++17", "-fopenmp", "-fno-signaling-nans", "-fno-trapping-math"],
                       extra_ldflags=["-fopenmp"], build_directory=OUT, verbose=False)
    with open(os.path.join(OUT, "THREADS"), "w") as f:
        f.write(str(threads))
    print("built", os.path.join(OUT, "cQIGen.so"), "threads", threads)


if __name__ == "__main__":
    main()
