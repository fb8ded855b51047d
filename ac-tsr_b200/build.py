"""Build libacsr.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python ac-tsr_b200/build.py [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(CSRC, 'libacsr.so')
STAMP = os.path.join(CSRC, '.libacsr.stamp')
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr', '-Xptxas', '-v']


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith('.cu'))


def _nvcc():
    for c in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError('nvcc not found')


def _headers_digest():
    h = hashlib.sha256()
    root = os.path.dirname(HERE)
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(('.cuh', '.h'))]
    files.append(os.path.join(root, 'include', 'acsr.h'))
    for f in files:
        with open(f, 'rb') as fh:
            # paths relative to the checkout: a tree copied or moved after the build stays up to date
            h.update(os.path.relpath(f, root).encode() + b'\0' + fh.read())
    h.update(' '.join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _source_digest(src, hdr):
    with open(os.path.join(CSRC, src), 'rb') as fh:
        return hashlib.sha256(hdr.encode() + fh.read()).hexdigest()


def build(force=False, verbose=False):
    """Compile what changed (one object per .cu, headers invalidate all); returns the path of the shared library."""
    hdr = _headers_digest()
    srcs = _sources()
    digs = {s: _source_digest(s, hdr) for s in srcs}
    total = hashlib.sha256(''.join(s + digs[s] for s in srcs).encode()).hexdigest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == total:
        return LIB
    todo, objs = [], []
    for s in srcs:
        o = os.path.join(CSRC, s[:-3] + '.o')
        objs.append(o)
        st = o + '.stamp'
        if force or not (os.path.exists(o) and os.path.exists(st) and open(st).read().strip() == digs[s]):
            todo.append((s, o))
    log, running = [], []
    jobs = max(1, int(os.environ.get('ACSR_BUILD_JOBS', os.cpu_count() or 4)))

    def reap(block):
        for item in list(running):
            s, o, p = item
            if block or p.poll() is not None:
                out, _ = p.communicate()
                running.remove(item)
                log.append('== %s ==\n%s' % (s, out))
                if p.returncode != 0:
                    for _, _, q in running:
                        q.kill()
                    raise RuntimeError('nvcc failed for %s:\n%s' % (s, out))
                with open(o + '.stamp', 'w') as fh:
                    fh.write(digs[s])
                if block:
                    return
    import time
    for s, o in todo:
        while len(running) >= jobs:
            reap(False)
            if len(running) >= jobs:
                time.sleep(0.2)
        cmd = [_nvcc()] + NVCC_FLAGS + ['-c', os.path.join(CSRC, s), '-o', o]
        running.append((s, o, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    while running:
        reap(True)
    cmd = [_nvcc(), '-shared', '-o', LIB] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a']
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError('link failed:\n' + r.stdout)
    with open(os.path.join(CSRC, 'build.log'), 'a' if len(todo) < len(srcs) else 'w') as fh:
        fh.write('\n'.join(log) + '\n')
    with open(STAMP, 'w') as fh:
        fh.write(total)
    if verbose:
        print('\n'.join(log))
    return LIB


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='--verbose' in sys.argv))
