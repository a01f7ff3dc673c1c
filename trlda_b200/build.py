"""
Builds the in-tree native pieces of trlda_b200 with explicit compiler invocations (no JIT cache, so the
built files travel with the repository snapshot to the GPU box):

  trlda_b200/libtrlda_b200.so     CUDA kernels + C ABI (include/trlda_b200.h), nvcc, sm_100a only
  trlda_b200/_trlda*.so           CPython extension hosting the reference's Python classes (g++)

nvcc cross-compiles without a GPU, so this also runs in the CPU-only container.
"""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
LIB = os.path.join(HERE, 'libtrlda_b200.so')

NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
NVCC_FLAGS = [
	'-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
	'-Xcompiler', '-fPIC', '-Xcompiler', '-fvisibility=hidden']
CXX = '/usr/bin/g++'


def _newer(target, sources):
	if not os.path.exists(target):
		return True
	t = os.path.getmtime(target)
	return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
	if verbose:
		print(' '.join(cmd), flush=True)
	subprocess.run(cmd, check=True)


def ext_path():
	return os.path.join(HERE, '_trlda' + sysconfig.get_config_var('EXT_SUFFIX'))


def build_library(force=False, verbose=False):
	headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.cuh', '.h'))]
	headers.append(os.path.join(ROOT, 'include', 'trlda_b200.h'))
	sources = [os.path.join(CSRC, 'kernels.cu'), os.path.join(CSRC, 'estep_stream.cu'),
		os.path.join(CSRC, 'estep_tmem.cu'), os.path.join(CSRC, 'sample.cu'), os.path.join(CSRC, 'csc.cu'), os.path.join(CSRC, 'ingest.cu'),
		os.path.join(CSRC, 'topics.cu'), os.path.join(CSRC, 'model.cu')]
	objects = []
	rebuilt = False
	for src in sources:
		obj = os.path.join(CSRC, os.path.basename(src)[:-3] + '.o')
		objects.append(obj)
		if force or _newer(obj, [src] + headers):
			_run([NVCC] + NVCC_FLAGS + ['-c', src, '-o', obj], verbose)
			rebuilt = True
	if rebuilt or _newer(LIB, objects):
		_run([NVCC, '-shared', '-o', LIB] + objects + ['-ldl'], verbose)
	return LIB


def build_extension(force=False, verbose=False):
	src = os.path.join(CSRC, 'pymodule.cpp')
	if not os.path.exists(src):
		return None
	import numpy
	target = ext_path()
	if force or _newer(target, [src, os.path.join(ROOT, 'include', 'trlda_b200.h')]):
		_run([
			CXX, '-O2', '-std=c++17', '-fPIC', '-shared', '-fvisibility=hidden', src, '-o', target,
			'-I' + sysconfig.get_paths()['include'], '-I' + numpy.get_include(), '-I' + os.path.join(ROOT, 'include'),
			'-L' + HERE, '-ltrlda_b200', '-Wl,-rpath,$ORIGIN'], verbose)
	return target


def build_all(force=False, verbose=False):
	build_library(force, verbose)
	build_extension(force, verbose)


if __name__ == '__main__':
	build_all(force='--force' in sys.argv, verbose=True)
