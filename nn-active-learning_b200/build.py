"""Builds libnnal_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OUT = os.path.join(HERE, 'libnnal_b200.so')
SOURCES = ['capi.cu', 'volume.cu', 'forward.cu', 'forward_simt.cu', 'score.cu', 'gemm_tc.cu', 'conv_tc.cu', 'conv_wt.cu', 'fi.cu', 'fi_block.cu', 'sims.cu', 'shrunk.cu', 'sdp.cu', 'influence.cu', 'p2p.cu']
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
         '-Xcompiler', '-fPIC', '-Xcompiler', '-pthread']


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(os.path.dirname(HERE), 'include', 'nnal_b200.h'), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, 'build'), exist_ok=True)
    for s in SOURCES:
        o = os.path.join(HERE, 'build', s.replace('.cu', '.o'))
        cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, s), '-o', o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(o)
    for s, p in procs:
        out = p.communicate()[0].decode()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError('nvcc failed on %s' % s)
        if verbose:
            print(out)
    cmd = [NVCC, '-shared', '-o', OUT] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a', '-lcudart_static',
                                                   '-Xcompiler', '-fPIC', '-Xcompiler', '-pthread', '-lpthread']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        sys.stderr.write(r.stdout.decode())
        raise RuntimeError('link failed')
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
