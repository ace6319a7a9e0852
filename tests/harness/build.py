"""Build the test harnesses.

- The broker harness (harness_broker.c + vb_broker.c over the oracle-backed mock ABI) needs nothing but this
  repository: it is always built, into tests/harness/_build/.
- The glue harness compiles the extension glue against pgvector's own headers, so it is built only where the pgvector
  source tree is present (PGVECTOR_SRC, default /root/reference).  It goes to oracle/_ref/harness/, beside the other
  binaries made from pgvector's sources, and is used as shipped where those sources are absent."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.join(os.environ.get("PGVECTOR_SRC", "/root/reference"), "src")
EXT = os.path.join(ROOT, "pgvector_b200", "ext")
OUT = os.path.join(ROOT, "oracle", "_ref", "harness")
BROKER_OUT = os.path.join(HERE, "_build")
SRCS = [os.path.join(HERE, f) for f in ("harness_common.c", "harness_ivf.c", "harness_hnsw.c", "harness_broker.c")] + \
       [os.path.join(EXT, f) for f in ("vb_ivfflat_scan.c", "vb_ivfflat_build.c", "vb_hnsw_scan.c", "vb_hnsw_build.c", "vb_broker.c")] + \
       [os.path.join(EXT, "pgstub", "pgstub_runtime.c")]
BROKER_SRCS = [os.path.join(HERE, "harness_broker.c"), os.path.join(EXT, "vb_broker.c"), os.path.join(HERE, "mock_abi.c")]
CFLAGS = ["-std=gnu11", "-O1", "-g", "-fPIC", "-shared", "-pthread", "-Wall", "-Werror", "-Wno-unused-function", "-Wno-comment"]
FLAGS = CFLAGS + ["-I" + os.path.join(EXT, "pgstub"), "-I" + REF, "-I" + os.path.join(ROOT, "include"), "-I" + EXT, "-I" + HERE]


def paths():
    return os.path.join(OUT, "libvbharness_mock.so"), os.path.join(OUT, "libvbharness_real.so")


def broker_path():
    return os.path.join(BROKER_OUT, "libvbharness_broker.so")


def build_broker(force=False):
    """the broker over the mock ABI; returns the library's path"""
    import oracle
    oracle.build()
    lib = broker_path()
    deps = BROKER_SRCS + [os.path.join(EXT, "vb_broker.h"), os.path.join(ROOT, "include", "vecb200.h"),
                          os.path.join(ROOT, "oracle", "pgv_oracle.h")]
    if force or not os.path.exists(lib) or os.path.getmtime(lib) < max(os.path.getmtime(d) for d in deps):
        os.makedirs(BROKER_OUT, exist_ok=True)
        cmd = ["gcc", *CFLAGS, "-I" + os.path.join(ROOT, "include"), "-I" + EXT, "-o", lib + ".tmp", *BROKER_SRCS,
               "-L" + os.path.join(ROOT, "oracle"), "-l:liboracle.so", "-Wl,-rpath,$ORIGIN/../../../oracle", "-lm"]
        subprocess.run(cmd, check=True, capture_output=True, text=True)
        os.replace(lib + ".tmp", lib)
    return lib


def build(force=False):
    mock, real = paths()
    if not os.path.isdir(REF):
        return os.path.exists(mock), os.path.exists(real)
    os.makedirs(OUT, exist_ok=True)
    deps = SRCS + [os.path.join(HERE, f) for f in ("mock_abi.c", "harness_common.h")] + [os.path.join(EXT, "vb_glue.h"), os.path.join(EXT, "vb_broker.h"),
                                                                                        os.path.join(EXT, "pgstub", "postgres.h"),
                                                                                        os.path.join(ROOT, "include", "vecb200.h")]
    newest = max(os.path.getmtime(d) for d in deps)
    import oracle
    oracle.build()
    if force or not os.path.exists(mock) or os.path.getmtime(mock) < newest:
        cmd = ["gcc", *FLAGS, "-o", mock + ".tmp", *SRCS, os.path.join(HERE, "mock_abi.c"),
               "-L" + os.path.join(ROOT, "oracle"), "-l:liboracle.so", "-Wl,-rpath,$ORIGIN/../..", "-lm"]
        subprocess.run(cmd, check=True, capture_output=True, text=True)
        os.replace(mock + ".tmp", mock)
    lib = os.path.join(ROOT, "pgvector_b200", "libvecb200.so")
    if os.path.exists(lib) and (force or not os.path.exists(real) or os.path.getmtime(real) < newest):
        cmd = ["gcc", *FLAGS, "-o", real + ".tmp", *SRCS, "-L" + os.path.dirname(lib), "-l:libvecb200.so",
               "-Wl,-rpath,$ORIGIN/../../../pgvector_b200", "-lm"]
        subprocess.run(cmd, check=True, capture_output=True, text=True)
        os.replace(real + ".tmp", real)
    return os.path.exists(mock), os.path.exists(real)


if __name__ == "__main__":
    try:
        print(build_broker(force=True), build(force=True))
    except subprocess.CalledProcessError as e:
        print(e.stderr)
        raise
