"""Build the reference's own ray-casting extension (tools/ray_iou/lib/dvr/dvr.{cpp,cu}) into oracle/_ref/.

ORACLE / test infrastructure only.  The sources are compiled from where they lie under /root/reference;
dvr.cu does not compile against torch 2.11 as shipped (`AT_DISPATCH_FLOATING_TYPES(x.type(), ...)` at
dvr.cu:371,683,736), so the recipe compiles a scratch copy under /tmp with the 3-token fix
`.type()` -> `.scalar_type()` applied by sed.  Nothing from the reference is copied into the repository;
only the built `dvr_ref.so` lands in oracle/_ref/ (git-ignored, travels to the GPU box).
tests/golden/gen_dvr_ref.py runs it on a GPU and stores its outputs in tests/golden/ref_dvr.npz, against which
tests/test_gpu_parity.py::test_render_forward_vs_reference_kernel pins both the CUDA ray-caster and the C restatement
(oracle/ray_dda.c).
"""
import os
import re
import shutil
import sys
import tempfile

REF = '/root/reference/tools/ray_iou/lib/dvr'
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, '_ref')


def build(verbose=False):
    if not os.path.isdir(REF):
        print('[build_ref] /root/reference not present: skipping (prebuilt oracle/_ref is used if it exists)')
        return None
    os.makedirs(OUT, exist_ok=True)
    so = os.path.join(OUT, 'dvr_ref.so')
    if os.path.exists(so):
        return so
    os.environ.setdefault('TORCH_CUDA_ARCH_LIST', '10.0a')
    os.environ.setdefault('MAX_JOBS', '4')
    from torch.utils.cpp_extension import load
    tmp = tempfile.mkdtemp(prefix='dvr_ref_src_')
    src = open(os.path.join(REF, 'dvr.cu')).read()
    patched, n = re.subn(r'AT_DISPATCH_FLOATING_TYPES\((\w+)\.type\(\)', r'AT_DISPATCH_FLOATING_TYPES(\1.scalar_type()', src)
    assert n == 3, n
    with open(os.path.join(tmp, 'dvr.cu'), 'w') as f:
        f.write(patched)
    bdir = os.path.join(tmp, 'build')
    os.makedirs(bdir)
    load('dvr_ref', sources=[os.path.join(REF, 'dvr.cpp'), os.path.join(tmp, 'dvr.cu')], build_directory=bdir,
         extra_cuda_cflags=['-allow-unsupported-compiler'], verbose=verbose, is_python_module=False)
    shutil.copy(os.path.join(bdir, 'dvr_ref.so'), so)
    shutil.rmtree(tmp, ignore_errors=True)
    print('[build_ref] built', so)
    return so


if __name__ == '__main__':
    build(verbose='-v' in sys.argv)
