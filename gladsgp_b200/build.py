"""In-tree nvcc build of libgladsgp_b200.so (sm_100a only).

The shared object lands in gladsgp_b200/ so that it travels with the repository snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libgladsgp_b200.so')
SOURCES = ['ggp_api.cu', 'ggp_loglik.cu', 'ggp_mcmc.cu', 'ggp_predict.cu', 'ggp_quantile.cu', 'ggp_xval.cu', 'ggp_chain_diag.cu', 'ggp_rsvd_tc.cu', 'ggp_ingest.cu', 'ggp_sobol.cu', 'ggp_gp_sens.cu', 'ggp_calib.cu', 'ggp_design.cu', 'ggp_hm.cu', 'ggp_grad_sens.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-fmad=false', '-Xcompiler', '-fPIC', '-Xptxas', '-v']


def _nvcc():
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        raise RuntimeError('nvcc not found')
    return nvcc


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(HERE, '..', 'include', 'gladsgp_b200.h'), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, 'build')
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        if not os.path.exists(src):
            continue
        o = os.path.join(objdir, s.replace('.cu', '.o'))
        objs.append(o)
        procs.append((s, subprocess.Popen([nvcc] + NVCC_FLAGS + ['-c', src, '-o', o],
                                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for s, p in procs:
        out, _ = p.communicate()
        log.append(out)
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError('nvcc failed on %s' % s)
    with open(os.path.join(objdir, 'ptxas.log'), 'w') as f:
        f.write('\n'.join(log))
    if verbose:
        print('\n'.join(log))
    subprocess.check_call([nvcc, '-shared', '-o', LIB, '-gencode', 'arch=compute_100a,code=sm_100a'] + objs + ['-cudart', 'static'])
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
