"""SURVEY.md 8f N3 — the reference's JNI and Ruby glue compile UNCHANGED against include/smatrix.h
and link against our static archive: every smatrix_* symbol they call resolves inside our library.
The glue is the reference's own source, which this repository does not carry: set $LIBSMATRIX_SRC to
the src/ directory of a libsmatrix checkout to run these tests; without it they skip.  No JDK / Ruby
is needed: tests/stubs/ provides just enough of jni.h / ruby.h to compile."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("LIBSMATRIX_SRC", "")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
pytestmark = pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "smatrix_jni.c")),
                                reason="needs the reference's JNI / Ruby glue: set LIBSMATRIX_SRC to libsmatrix's src/")


@pytest.fixture(scope="module")
def archive():
    from libsmatrix_b200 import build
    so = build.build()
    return os.path.join(os.path.dirname(so), "smatrix-static.a")


def _link(tmp_path, src, archive, extra):
    out = tmp_path / (os.path.basename(src) + ".so")
    cmd = ["gcc", "-shared", "-fPIC", "-w", f"-I{ROOT}/include", f"-I{ROOT}/tests/stubs", f"-I{REF}",
           src, archive, "-o", str(out), f"-L{CUDA}/lib64", "-lcudart_static", "-lstdc++", "-ldl",
           "-lrt", "-lpthread"] + extra
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    nm = subprocess.run(["nm", str(out)], capture_output=True, text=True, check=True).stdout
    return nm


def test_jni_glue_links_unchanged(tmp_path, archive):
    nm = _link(tmp_path, os.path.join(REF, "smatrix_jni.c"), archive, ["-Wl,--no-undefined"])
    for sym in ("Java_com_paulasmuth_libsmatrix_SparseMatrix_init",
                "Java_com_paulasmuth_libsmatrix_SparseMatrix_getRowNative",
                "smatrix_open", "smatrix_close", "smatrix_get", "smatrix_set", "smatrix_incr",
                "smatrix_decr", "smatrix_rowlen", "smatrix_getrow"):
        assert re.search(rf" [Tt] {sym}\b", nm), sym      # defined inside the linked object
    assert not re.search(r" U smatrix_", nm)


def test_ruby_glue_links_unchanged(tmp_path, archive):
    # like src/ruby/Makefile:18-19 the interpreter symbols (rb_*) stay undefined until load time
    nm = _link(tmp_path, os.path.join(REF, "smatrix_ruby.c"), archive, [])
    for sym in ("Init_smatrix", "smatrix_rb_incr", "smatrix_open", "smatrix_incr", "smatrix_close"):
        assert re.search(rf" [Tt] {sym}\b", nm), sym
    assert not re.search(r" U smatrix_", nm)
    assert re.search(r" U rb_define_method", nm)


def test_batched_jni_glue_compiles_links_and_runs(tmp_path):
    """N3, second half: examples/jni/smatrix_jni_batch.c (incrBatch / setBatch / getBatch / getRowsNative,
    the batched natives INTEGRATION.md proposes) compiles against the stub jni.h, links against the static
    archive with no undefined smatrix_* symbol, and RUNS — together with the reference's unchanged
    src/smatrix_jni.c — under a toy JNIEnv (tests/stubs/fake_jvm.c) on the simulator library: the bulk
    natives agree with the reference's per-pair getRowNative and with a host-side tally."""
    glue = os.path.join(ROOT, "examples", "jni", "smatrix_jni_batch.c")
    from libsmatrix_b200 import build
    archive = os.path.join(os.path.dirname(build.build()), "smatrix-static.a")
    nm = _link(tmp_path, glue, archive, ["-Wl,--no-undefined"])
    for sym in ("incrBatch", "setBatch", "getBatch", "getRowsNative"):
        assert re.search(rf" T Java_com_paulasmuth_libsmatrix_SparseMatrix_{sym}\b", nm), sym
    assert re.search(r" [Tt] smatrix_getrow_batch\b", nm) and not re.search(r" U smatrix_", nm)
    from hostsim import build as sim_build
    sim = sim_build.build()
    exe = str(tmp_path / "fake_jvm")
    r = subprocess.run(["gcc", "-O1", "-w", f"-I{ROOT}/include", f"-I{ROOT}/tests/stubs", f"-I{REF}",
                        os.path.join(ROOT, "tests", "stubs", "fake_jvm.c"), os.path.join(REF, "smatrix_jni.c"), glue,
                        "-L", os.path.dirname(sim), "-l" + os.path.basename(sim)[3:-3],
                        f"-Wl,-rpath,{os.path.dirname(sim)}", "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300, env=dict(os.environ, SMATRIX_DIR_LOG2="6"))
    assert r.returncode == 0 and "fake_jvm: OK" in r.stdout, r.stdout + r.stderr
