"""In-tree build of the CUDA library (``nvcc`` for sm_100a only; no JIT cache)."""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, 'csrc')
LIB_PATH = os.path.join(_HERE, 'libdair_pll_b200.so')
SOURCES = ['cn_kernels.cu', 'cn_tangent.cu', 'cn_tangent_elbow.cu', 'cn_icnn.cu', 'cn_comm.cu', 'cn_adjoint.cu', 'cn_elbow_wf.cu', 'cn_chain.cu', 'cn_icnn_tc.cu', 'cn_icnn_tc_bwd.cu', 'cn_leaf.cu', 'cn_tangent_chain.cu']
HEADERS = ['cn_common.cuh', 'cn_cube.cuh', 'cn_params.cuh', 'cn_elbow.cuh', 'cn_dual.cuh', 'cn_cube_tangent.cuh', 'cn_elbow_tangent.cuh', 'cn_comm.cuh', 'cn_cube_adjoint.cuh', 'cn_elbow_wf.cuh', 'cn_chain.cuh', 'cn_chain_tangent.cuh', 'cn_icnn_tc.cuh', 'cn_launch.cuh', 'cn_reduce.cuh', os.path.join('..', '..', 'include', 'dair_pll_b200.h'), os.path.join('..', '..', 'include', 'dair_pll_b200_warm.h'),
           os.path.join('..', '..', 'include', 'dair_pll_b200_warm_body_tree.h')]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-lineinfo', '-O3', '-std=c++17',
              '-Xcompiler', '-fPIC']


def _nvcc() -> str:
    for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return 'nvcc'


HASH_PATH = LIB_PATH + '.hash'


def sources_present() -> bool:
    return all(os.path.exists(os.path.join(CSRC, f)) for f in SOURCES)


def source_hash() -> str:
    """Content hash of everything the library is compiled from (robust to copies that reset mtimes)."""
    import hashlib
    h = hashlib.sha256(' '.join(NVCC_FLAGS).encode())
    for f in sorted(SOURCES + HEADERS):
        with open(os.path.join(CSRC, f), 'rb') as fh:
            h.update(f.encode() + b'\0' + fh.read())
    return h.hexdigest()


def is_stale() -> bool:
    """True if the library is missing or was built from other sources than the ones present."""
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as fh:
        return fh.read().strip() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile ``csrc/*.cu`` into ``dair_pll_b200/libdair_pll_b200.so`` (cross-compiles without a GPU)."""
    if not force and not is_stale():
        return LIB_PATH
    # translation units are compiled in parallel (the dual-number one is slow), then linked
    objdir = os.path.join(_HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace('.cu', '.o'))
        cmd = [_nvcc()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', '-o', obj, os.path.join(CSRC, src)]
        procs.append((cmd, obj, subprocess.Popen(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    objs = []
    for cmd, obj, proc in procs:
        out, err = proc.communicate()
        if verbose:
            sys.stderr.write(err)
        if proc.returncode != 0:
            raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + out + err)
        objs.append(obj)
    link = [_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', LIB_PATH] + objs
    proc = subprocess.run(link, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError('link failed:\n' + ' '.join(link) + '\n' + proc.stdout + proc.stderr)
    with open(HASH_PATH, 'w') as fh:
        fh.write(source_hash() + '\n')
    return LIB_PATH


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose=True))
