"""In-tree build of libd2d_b200.so (nvcc, sm_100a only).  Cross-compiles without a GPU.

The library is several translation units compiled in parallel and linked into one shared object; objects are cached
under gym_d2d_b200/_obj and rebuilt when a source they include is newer.  `extra` defines (the A/B harness of
profiles/ab.sh) build a differently named library next to the main one.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
from pathlib import Path
from typing import Iterable, List, Optional, Sequence, Tuple

PKG = Path(__file__).resolve().parent
CSRC = PKG / 'csrc'
OBJ = PKG / '_obj'
LIB = PKG / 'libd2d_b200.so'
HEADER = PKG.parent / 'include' / 'd2d_b200.h'
COMMON = ['d2d_internal.h', 'd2d_common.cuh']
# (object name, source, extra defines, headers it includes besides COMMON)
UNITS: List[Tuple[str, str, List[str], List[str]]] = [
    ('abi', 'd2d_abi.cu', [], ['d2d_aux.cuh', 'd2d_launch_plan.h']),
    ('warp2', 'd2d_tu_warp.cu', ['-DD2D_TU_WPB=2'], ['d2d_step_warp.cuh']),
    ('warp4', 'd2d_tu_warp.cu', ['-DD2D_TU_WPB=4'], ['d2d_step_warp.cuh']),
    ('warp8', 'd2d_tu_warp.cu', ['-DD2D_TU_WPB=8'], ['d2d_step_warp.cuh']),
    ('dense', 'd2d_tu_dense.cu', [], ['d2d_step_dense.cuh']),
    ('block', 'd2d_tu_block.cu', [], ['d2d_step_block.cuh']),
]
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC,-fvisibility=hidden']


def _nvcc() -> str:
    for cand in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError('nvcc not found: libd2d_b200.so can only be built with the CUDA toolkit')


def _sources() -> Iterable[Path]:
    return list(CSRC.glob('*.cu*')) + list(CSRC.glob('*.h')) + [HEADER]


def needs_build(lib: Path = LIB) -> bool:
    if not lib.exists():
        return True
    return lib.stat().st_mtime < max(p.stat().st_mtime for p in _sources())


def _compile(name: str, src: str, defines: Sequence[str], deps: Sequence[str], tag: str, force: bool, verbose: bool) -> Path:
    obj = OBJ / f'{name}{tag}.o'
    dep_paths = [CSRC / src, HEADER] + [CSRC / d for d in list(deps) + COMMON]
    if not force and obj.exists() and obj.stat().st_mtime >= max(p.stat().st_mtime for p in dep_paths):
        return obj
    cmd = [_nvcc(), *NVCC_FLAGS, *defines, '-c', '-o', str(obj), str(CSRC / src)]
    if verbose:
        cmd.insert(1, '-Xptxas=-v')
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f'nvcc failed on {src} ({res.returncode}):\n{res.stdout}\n{res.stderr}')
    if verbose:
        print(res.stderr)
    return obj


def build(force: bool = False, verbose: bool = False, extra: Optional[Sequence[str]] = None, out: Optional[Path] = None) -> Path:
    """Compile every CUDA source of the package into gym_d2d_b200/libd2d_b200.so (or `out`, with `extra` nvcc defines)."""
    lib = Path(out) if out is not None else LIB
    extra = list(extra or [])
    if not force and not needs_build(lib):
        return lib
    OBJ.mkdir(exist_ok=True)
    tag = ('-' + hashlib.sha1(' '.join(extra).encode()).hexdigest()[:8]) if extra else ''
    with cf.ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 1)) as pool:
        futs = [pool.submit(_compile, name, src, list(defs) + extra, deps, tag, force, verbose) for name, src, defs, deps in UNITS]
        objs = [f.result() for f in futs]
    lib.parent.mkdir(parents=True, exist_ok=True)
    res = subprocess.run([_nvcc(), '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', str(lib), *map(str, objs)],
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f'link failed ({res.returncode}):\n{res.stdout}\n{res.stderr}')
    return lib


if __name__ == '__main__':
    import sys
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
