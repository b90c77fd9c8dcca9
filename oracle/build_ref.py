"""Build oracle/_ref: the reference's OWN CPU rotated-IoU (utils/detzero_utils/ops/iou3d_nms/src/iou3d_cpu.cpp) compiled from the
sources where they lie in the reference checkout (REF_SRC; never copied), plus a 10-line pybind11 binding of ours.  Used by
tests/golden/make_golden_host.py to record the output that pins the oracle's rotated-IoU restatement.  g++ directly; outputs
only into oracle/_ref/ (git-ignored)."""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = '/root/reference/utils/detzero_utils/ops/iou3d_nms/src/iou3d_cpu.cpp'
OUT = os.path.join(HERE, '_ref')
SO = os.path.join(OUT, 'ref_iou3d_cpu' + (sysconfig.get_config_var('EXT_SUFFIX') or '.so'))


def build(force=False):
    if os.path.exists(SO) and not force:
        return SO
    if not os.path.exists(REF_SRC):
        raise RuntimeError('reference sources not mounted')
    import torch
    from torch.utils import cpp_extension as ce
    os.makedirs(OUT, exist_ok=True)
    inc = ce.include_paths() + ['/usr/local/cuda/include', sysconfig.get_paths()['include'], os.path.dirname(REF_SRC)]
    libdir = os.path.join(os.path.dirname(torch.__file__), 'lib')
    cmd = ['g++', '-O2', '-shared', '-fPIC', '-std=c++17', '-w', '-DTORCH_EXTENSION_NAME=ref_iou3d_cpu',
           '-D_GLIBCXX_USE_CXX11_ABI=%d' % int(torch._C._GLIBCXX_USE_CXX11_ABI)] + ['-I' + i for i in inc] + \
          [REF_SRC, os.path.join(HERE, 'ref_binding.cpp'), '-o', SO, '-L' + libdir, '-Wl,-rpath,' + libdir,
           '-ltorch', '-ltorch_cpu', '-lc10', '-ltorch_python']
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError('oracle/_ref build failed:\n' + r.stderr[-3000:])
    return SO


def load():
    import importlib.util
    import torch  # noqa: F401
    spec = importlib.util.spec_from_file_location('ref_iou3d_cpu', SO)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


if __name__ == '__main__':
    print(build(force='-f' in sys.argv))
