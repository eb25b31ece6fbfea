"""Run-time compilation of user models (models.CudaModel) through NVRTC.

NVRTC is found, in this order:
  1. the file named by MC3B_NVRTC (only that one, when it is set);
  2. nvidia/cuda_nvrtc/lib/libnvrtc.so.12 of the installed nvidia-cuda-nvrtc wheel
     (a dependency of torch);
  3. $CUDA_HOME/lib64/libnvrtc.so.12, then /usr/local/cuda/lib64/libnvrtc.so.12;
  4. the soname libnvrtc.so.12 on the loader's search path.
The first that loads and is 12.8 or newer (the first release that targets sm_100a)
is used; the library dlopen's the same path.

Compiled CUBINs are kept in memory per process, and on disk in the directory named
by MC3B_JIT_CACHE when it is set.  The key covers the source, the parameter count,
the number of inputs, constants and work slots, the dtype, MC3B_VERSION, the NVRTC version and the
embedded kernel headers (not the values of the constants: they are run-time data); the
loader also checks the module's own ABI record, so a stale file is compiled again
rather than launched.
"""
import ctypes
import hashlib
import os
import threading
import time

from . import _lib

_NVRTC = None                 # (path, (major, minor)) once found
_CUBINS = {}                  # key -> bytes
_HANDLES = {}                 # key -> mc3b_user_model_t* (process lifetime)
_LOCK = threading.Lock()
_HEADERS = None


def nvrtc_candidates():
    """NVRTC paths in discovery order."""
    env = os.environ.get('MC3B_NVRTC')
    if env:
        return [env]
    out = []
    try:
        import nvidia
        for d in nvidia.__path__:
            out.append(os.path.join(d, 'cuda_nvrtc', 'lib', 'libnvrtc.so.12'))
    except ImportError:
        pass
    if os.environ.get('CUDA_HOME'):
        out.append(os.path.join(os.environ['CUDA_HOME'], 'lib64', 'libnvrtc.so.12'))
    out.append('/usr/local/cuda/lib64/libnvrtc.so.12')
    out.append('libnvrtc.so.12')
    return out


def _probe(path):
    """(major, minor) of the NVRTC at `path`, or a reason it cannot be used."""
    if os.sep in path and not os.path.exists(path):
        return 'not found'
    try:
        lib = ctypes.CDLL(path)
        major, minor = ctypes.c_int(0), ctypes.c_int(0)
        lib.nvrtcVersion(ctypes.byref(major), ctypes.byref(minor))
    except (OSError, AttributeError) as e:
        return f'cannot be loaded ({e})'
    if (major.value, minor.value) < (12, 8):
        return f'NVRTC {major.value}.{minor.value} cannot target sm_100a (needs 12.8 or newer)'
    return major.value, minor.value


def find_nvrtc():
    """(path, (major, minor)) of the NVRTC to use; Mc3bError listing every path tried."""
    global _NVRTC
    env = os.environ.get('MC3B_NVRTC')
    if _NVRTC is not None and (not env or _NVRTC[0] == env):
        return _NVRTC
    tried = []
    for path in nvrtc_candidates():
        r = _probe(path)
        if isinstance(r, tuple):
            _NVRTC = (path, r)
            return _NVRTC
        tried.append(f'{path}: {r}')
    raise _lib.Mc3bError('no usable NVRTC (12.8 or newer) for user models; tried\n  '
                         + '\n  '.join(tried) + '\nset MC3B_NVRTC to the path of libnvrtc.so.12')


def _headers_digest():
    global _HEADERS
    if _HEADERS is None:
        from .build import jit_headers_digest
        _HEADERS = jit_headers_digest()
    return _HEADERS


def cache_key(source, nmodel, dtype, ninputs=1, nconst=0, nwork=0):
    """Hex key of one compiled model (dtype: _lib.F64 or _lib.F32).  A model of one
    input and no constants or work slots keeps the key it had before models took
    several inputs."""
    _, ver = find_nvrtc()
    h = hashlib.sha256()
    parts = [source, str(int(nmodel)), str(int(dtype)), str(_lib.load().mc3b_version()),
             f'{ver[0]}.{ver[1]}', _headers_digest()]
    if int(ninputs) != 1:
        parts.append(f'ninputs={int(ninputs)}')
    if int(nconst) != 0:
        parts.append(f'nconst={int(nconst)}')
    if int(nwork) != 0:
        parts.append(f'nwork={int(nwork)}')
    for part in parts:
        h.update(part.encode() + b'\0')
    return h.hexdigest()


def _desc(nmodel, dtype, ninputs, nconst, nwork):
    return ctypes.byref(_lib.UserModelDesc(int(nmodel), int(ninputs), int(nconst), int(nwork), int(dtype)))


def compile_cubin(source, nmodel, dtype, name='model', ninputs=1, nconst=0, nwork=0):
    """NVRTC: source -> sm_100a CUBIN bytes.  ValueError with the log when the source
    does not compile."""
    path, _ = find_nvrtc()
    size = ctypes.c_int64(0)
    cap = 1 << 22
    log = ctypes.create_string_buffer(1 << 16)
    lib = _lib.load()
    while True:
        buf = ctypes.create_string_buffer(cap)
        rc = lib.mc3b_user_model_compile_desc(path.encode(), source.encode(), _desc(nmodel, dtype, ninputs, nconst, nwork),
                                              buf, cap, ctypes.byref(size), log, len(log))
        if rc == _lib.ERR_ARG and size.value > cap:
            cap = size.value
            continue
        break
    if rc == _lib.ERR_ARG:
        msg = lib.mc3b_last_error().decode('utf-8', 'replace')
        raise ValueError(f'CudaModel {name!r}: {msg}\n{log.value.decode("utf-8", "replace")}')
    if rc != _lib.OK:
        raise _lib.Mc3bError('mc3b_user_model_compile failed: '
                             + lib.mc3b_last_error().decode('utf-8', 'replace'))
    return buf.raw[:size.value]


def _load(cubin, nmodel, dtype, ninputs=1, nconst=0, nwork=0):
    h = ctypes.c_void_p()
    rc = _lib.load().mc3b_user_model_load_desc(cubin, len(cubin), _desc(nmodel, dtype, ninputs, nconst, nwork),
                                               ctypes.byref(h))
    return h if rc == _lib.OK else rc


def handle(source, nmodel, dtype, name='model', stats=None, ninputs=1, nconst=0, nwork=0):
    """Loaded module of (source, nmodel, dtype, ninputs, nconst, nwork): compiled once per process
    (and taken from MC3B_JIT_CACHE when it is there).  stats, a dict, receives where
    the CUBIN came from ('memory', 'disk', 'nvrtc') and the seconds it took."""
    key = cache_key(source, nmodel, dtype, ninputs, nconst, nwork)
    with _LOCK:
        h = _HANDLES.get(key)
        if h is not None:
            if stats is not None:
                stats.update(origin='memory', seconds=0.0)
            return h
        t0 = time.perf_counter()
        origin = 'memory'
        cubin = _CUBINS.get(key)
        cdir = os.environ.get('MC3B_JIT_CACHE')
        fpath = os.path.join(cdir, key + '.cubin') if cdir else None
        if cubin is None and fpath and os.path.exists(fpath):
            with open(fpath, 'rb') as f:
                cubin = f.read()
            origin = 'disk'
        h = _load(cubin, nmodel, dtype, ninputs, nconst, nwork) if cubin is not None else None
        if not isinstance(h, ctypes.c_void_p):
            # not compiled yet, or a stale file that the loader refused: compile
            cubin = compile_cubin(source, nmodel, dtype, name, ninputs, nconst, nwork)
            origin = 'nvrtc'
            if fpath:
                os.makedirs(cdir, exist_ok=True)
                tmp = f'{fpath}.{os.getpid()}.tmp'
                with open(tmp, 'wb') as f:
                    f.write(cubin)
                os.replace(tmp, fpath)
            h = _load(cubin, nmodel, dtype, ninputs, nconst, nwork)
            if not isinstance(h, ctypes.c_void_p):
                raise _lib.Mc3bError('mc3b_user_model_load failed: '
                                     + _lib.load().mc3b_last_error().decode('utf-8', 'replace'))
        _CUBINS[key] = cubin
        _HANDLES[key] = h
        if stats is not None:
            stats.update(origin=origin, seconds=time.perf_counter() - t0)
        return h


def forget():
    """Drop the in-memory CUBINs (the loaded modules stay: populations may use them);
    the next handle() of a model not loaded yet compiles or reads the disk cache."""
    with _LOCK:
        _CUBINS.clear()
