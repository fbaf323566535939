"""Compile the sm_100a CUDA library in-tree (nvcc cross-compiles without a GPU).

The 64 step-kernel variants are spread over eight translation units (csrc/step_instances.cu compiled once per
(KFUSED, P1BOT, P2BOT)) next to the C-ABI unit, all compiled in parallel and linked into libfootsies_b200.so."""
import concurrent.futures
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(PKG_DIR, "build")
LIB_NAME = "libfootsies_b200.so"
LIB_PATH = os.environ.get("FOOTSIES_B200_LIB") or os.path.join(PKG_DIR, LIB_NAME)   # override: developer experiments only

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",            # fp32 ops round one by one, like the scalar C# expressions they restate
    "-Xcompiler", "-fPIC",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libfootsies_b200.so")


def sources():
    return [os.path.join(CSRC, "footsies_kernels.cu"), os.path.join(CSRC, "step_instances.cu"),
            os.path.join(CSRC, "policy_kernel.cu"), os.path.join(CSRC, "rollout_kernel.cu")]


def deps():
    inc = os.path.join(os.path.dirname(PKG_DIR), "include", "footsies_b200.h")
    return sources() + [os.path.join(CSRC, f) for f in ("state_codec.h", "frame_tables.h", "frame_logic.cuh",
                                                        "tables_host.h", "step_kernel.cuh", "policy_mlp.cuh", "policy_mma.cuh", "device_once.h",
                                                        "rollout_kernel.h", "delay_ring.cuh")] + [inc]


def source_digest(extra_flags=()):
    """sha256 over the contents of every source / header and the compiler flags: what the built library depends on.
    (Content, not mtimes: the tree is copied to GPU boxes and checked out by git, neither of which keeps timestamps.)"""
    import hashlib
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS + list(extra_flags)).encode())
    for d in deps():
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _digest_path(lib_path):
    return lib_path + ".srchash"


def is_stale(lib_path=None, extra_flags=()):
    """True when the library is missing or was built from other sources / flags than the ones in the tree."""
    lib_path = lib_path or LIB_PATH
    if not os.path.exists(lib_path):
        return True
    try:
        with open(_digest_path(lib_path)) as f:
            return f.read().strip() != source_digest(extra_flags)
    except OSError:
        return True


def translation_units():
    """(object name, source, extra defines)"""
    # The policy arithmetic (policy_mlp.cuh) spells its multiply-adds as explicit fmaf; both translation units that use
    # it are compiled with -fmad=false like everything else (the rollout kernel holds the simulator too), so that no
    # other expression is contracted in one and not in the other: their logits and log-probabilities are bit-identical.
    units = [("abi.o", os.path.join(CSRC, "footsies_kernels.cu"), []),
             ("policy.o", os.path.join(CSRC, "policy_kernel.cu"), []),
             ("rollout.o", os.path.join(CSRC, "rollout_kernel.cu"), [])]           # the dispatcher
    for hidden in (32, 64, 128):
        for dense in (0, 1):
            for delay in (0, 1):
                units.append((f"rollout{'_delay' if delay else ''}_h{hidden}_d{dense}.o", os.path.join(CSRC, "rollout_kernel.cu"),
                              [f"-DFG_ROLLOUT_H={hidden}", f"-DFG_ROLLOUT_DENSE={dense}", f"-DFG_ROLLOUT_DELAY={delay}"]))
    for kf in (0, 1):
        for b1 in (0, 1):
            for b2 in (0, 1):
                units.append((f"step_k{kf}_b{b1}{b2}.o", os.path.join(CSRC, "step_instances.cu"),
                              [f"-DFG_INST_KF={kf}", f"-DFG_INST_B1={b1}", f"-DFG_INST_B2={b2}"]))
    return units


def build(force=False, verbose=False, extra_flags=(), lib_path=None):
    """Build libfootsies_b200.so next to this file; returns its path.  Safe to call from several processes at once (one
    rank per GPU under torchrun): an exclusive file lock serialises them, staleness is re-checked under the lock, objects
    go to a per-process directory and the library is moved into place atomically."""
    import fcntl
    import tempfile
    lib_path = lib_path or LIB_PATH
    if not force and not is_stale(lib_path, extra_flags):
        return lib_path
    nvcc = _nvcc()
    obj_root = OBJ_DIR if lib_path == LIB_PATH else lib_path + ".obj"
    os.makedirs(obj_root, exist_ok=True)
    flags = NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else [])
    with open(os.path.join(obj_root, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale(lib_path, extra_flags):      # another process built it while this one waited
                return lib_path
            obj_dir = tempfile.mkdtemp(prefix="obj.", dir=obj_root)

            def compile_one(unit):
                name, src, defs = unit
                out = os.path.join(obj_dir, name)
                res = subprocess.run([nvcc] + flags + defs + ["-c", src, "-o", out], capture_output=True, text=True)
                if res.returncode != 0:
                    raise RuntimeError(f"nvcc failed on {name}:\n" + res.stdout + res.stderr)
                return out, res.stderr

            try:
                units = translation_units()
                with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(units), os.cpu_count() or 2)) as pool:
                    results = list(pool.map(compile_one, units))
                if verbose:
                    for _, log in results:
                        print(log)
                tmp_lib = os.path.join(obj_dir, LIB_NAME)
                res = subprocess.run([nvcc, "-shared", "-o", tmp_lib] + [o for o, _ in results], capture_output=True, text=True)
                if res.returncode != 0:
                    raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
                os.replace(tmp_lib, lib_path)
                with open(_digest_path(lib_path) + ".tmp", "w") as f:
                    f.write(source_digest(extra_flags) + "\n")
                os.replace(_digest_path(lib_path) + ".tmp", _digest_path(lib_path))
            finally:
                shutil.rmtree(obj_dir, ignore_errors=True)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return lib_path


if __name__ == "__main__":
    import sys
    print(build(force=True, verbose="-v" in sys.argv))
