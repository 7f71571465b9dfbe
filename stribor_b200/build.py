"""Build libstribor_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m stribor_b200.build [--force]

Each ``csrc/*.cu`` is compiled to an object under ``stribor_b200/build/`` (in parallel, re-done only when
the source, a header or the flags changed) and the objects are linked into the shared library.
"""
from __future__ import annotations

import concurrent.futures as cf
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
OUT = os.path.join(HERE, 'libstribor_b200.so')
OBJ = os.path.join(HERE, 'build')

ARCH_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a']
CC_FLAGS = ARCH_FLAGS + ['-lineinfo', '-O3', '-std=c++17', '-Xcompiler', '-fPIC', '-Xptxas', '-v']
# kept for tools that print the one-line equivalent of the build
NVCC_FLAGS = CC_FLAGS + ['-shared']


def sources():
    return sorted(glob.glob(os.path.join(CSRC, '*.cu')))


def _headers():
    return sorted(glob.glob(os.path.join(CSRC, '*.cuh'))) + \
        [os.path.join(os.path.dirname(HERE), 'include', 'stribor_b200.h')]


def _deps():
    return sources() + _headers()


def up_to_date() -> bool:
    if not os.path.exists(OUT):
        return False
    t = os.path.getmtime(OUT)
    return all(os.path.getmtime(p) <= t for p in _deps())


def _digest(paths, extra=''):
    h = hashlib.sha1(extra.encode())
    for p in paths:
        with open(p, 'rb') as f:
            h.update(f.read())
    return h.hexdigest()


def _compile_one(nvcc, src, obj, flags):
    cmd = [nvcc] + flags + ['-c', src, '-o', obj]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return src, ' '.join(cmd), r.returncode, r.stdout


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and up_to_date():
        return OUT
    nvcc = os.environ.get('NVCC', 'nvcc')
    tag = hashlib.sha1(' '.join(CC_FLAGS).encode()).hexdigest()[:8]
    objdir = os.path.join(OBJ, tag)
    os.makedirs(objdir, exist_ok=True)
    hdr = _digest(_headers(), ' '.join(CC_FLAGS))
    jobs, objs = [], []
    for src in sources():
        base = os.path.splitext(os.path.basename(src))[0]
        obj = os.path.join(objdir, base + '.o')
        stamp = obj + '.sha1'
        want = _digest([src], hdr)
        objs.append(obj)
        have = open(stamp).read() if os.path.exists(stamp) and os.path.exists(obj) else ''
        if force or have != want:
            jobs.append((src, obj, stamp, want))
    logs = []
    failed = False
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            futs = {ex.submit(_compile_one, nvcc, s, o, CC_FLAGS): (s, o, st, w) for s, o, st, w in jobs}
            for fu in cf.as_completed(futs):
                s, o, st, w = futs[fu]
                src, cmd, rc, text = fu.result()
                logs.append(cmd + '\n' + text)
                if rc != 0:
                    failed = True
                    if os.path.exists(st):
                        os.remove(st)
                else:
                    with open(st, 'w') as f:
                        f.write(w)
    link_text = ''
    if not failed:
        cmd = [nvcc] + ARCH_FLAGS + ['-shared', '-o', OUT] + objs + ['-lcuda']
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        link_text = ' '.join(cmd) + '\n' + r.stdout
        failed = r.returncode != 0
    text = '\n'.join(logs) + '\n' + link_text
    log = os.path.join(HERE, 'build.log')
    with open(log, 'w') as f:
        f.write(text)
    if verbose or failed:
        print(text)
    if failed:
        raise RuntimeError(f'nvcc failed; see {log}')
    return OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv or '--force' in sys.argv))
