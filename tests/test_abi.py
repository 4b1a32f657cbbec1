"""The C-ABI library builds here (nvcc cross-compiles), loads, and exports every symbol that
include/b200w.h declares; and the product path fails loudly — never falls back — without a GPU."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "b200w.h")).read()
    return sorted(set(re.findall(r"B200W_API[^;(]*?\b(b200w_\w+)\s*\(", src)))


def test_header_declares_the_expected_surface():
    syms = header_symbols()
    for must in ("b200w_create", "b200w_train_step", "b200w_comm_init", "b200w_op_gemm",
                 "b200w_op_attention_bwd", "b200w_load_tensor", "b200w_read_tensor"):
        assert must in syms
    assert len(syms) >= 30


def test_library_exports_every_declared_symbol(lib_path):
    lib = C.CDLL(lib_path)
    for s in header_symbols():
        assert hasattr(lib, s), f"libb200w.so does not export {s}"
    assert lib.b200w_abi_version() == 2


def test_python_prototypes_cover_the_header(lib_path):
    from runbooks_b200 import _lib
    assert sorted(_lib.PROTOTYPES) == header_symbols()
    _lib.load()


def test_library_is_sm100a_tcgen05_tma(lib_path):
    """SASS evidence that the hot kernels are Blackwell-native (B200_PROFILING.md table)."""
    sass = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "HMMA.16" not in sass  # no legacy mma.sync path


def test_no_torch_or_cpu_dependency_in_the_library(lib_path):
    needed = subprocess.run(["ldd", lib_path], capture_output=True, text=True).stdout
    assert "torch" not in needed and "libcuda.so" not in needed


def test_create_fails_loudly_without_a_gpu(lib_path):
    """Run in a child process with every device hidden, so that the failure mode is checked on a GPU machine too
    (this process may already hold a CUDA context)."""
    code = ("from runbooks_b200.engine import Engine\n"
            "from runbooks_b200._lib import B200WError\n"
            "try:\n"
            "    Engine(0)\n"
            "except B200WError as ex:\n"
            "    print(ex)\n"
            "else:\n"
            "    raise SystemExit('Engine(0) did not raise')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert "no CPU fallback" in r.stdout or "CUDA" in r.stdout, r.stdout


def test_product_code_never_touches_the_oracle():
    bad = []
    for root, _, files in os.walk(os.path.join(ROOT, "runbooks_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(root, f), errors="ignore").read()
                # imports, includes, dlopen / subprocess paths — a comment citing the oracle is fine
                if re.search(r"^\s*(from|import)\s+oracle\b|#include[^\n]*oracle|[\"']oracle[/.\"']|"
                             r"[\"'][^\"'\n]*oracle/_ref", txt, re.M):
                    bad.append(f)
    assert not bad, bad


def test_header_is_plain_c_and_the_integration_example_links(lib_path, tmp_path):
    """include/b200w.h is what a cgo / C host binds (INTEGRATION.md 2): it must compile as C99 (no C++-isms,
    no torch types) and a C program using it as that section shows must link against the library and get
    the documented loud failure on a machine without a B200."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    src = tmp_path / "host.c"
    src.write_text(r'''
#include <stdio.h>
#include <stdint.h>
#include "b200w.h"
int main(void) {
  b200w_ctx* ctx = NULL;
  int st = b200w_create(0, &ctx);
  if (st != B200W_OK) { printf("create failed as documented: %d %s\n", st, b200w_last_error(NULL)); return 3; }
  b200w_arch a = {.vocab_size = 32000, .hidden_size = 4096, .intermediate_size = 11008, .num_layers = 32,
                  .num_heads = 32, .num_kv_heads = 32, .head_dim = 128, .max_seq_len = 4096, .rms_norm_eps = 1e-5f,
                  .rope_theta = 10000.0f, .family = B200W_FAMILY_LLAMA,
                  .pad_token_id = 0 /* Llama-2-7b-hf config.json; -1 when the checkpoint has none */};
  st = b200w_model_init(ctx, &a, NULL, 1, 1);
  float loss = 0, gnorm = 0;
  int32_t ids[1] = {0};
  if (st == B200W_OK) st = b200w_train_step(ctx, ids, ids, 1, 5e-5f, &loss, &gnorm);
  b200w_destroy(ctx);
  return st == B200W_OK ? 0 : 4;
}
''')
    exe = tmp_path / "host"
    libdir = os.path.dirname(lib_path)
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
                        "-o", str(exe), "-L", libdir, "-lb200w", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert run.returncode == 3 and "no CPU fallback" in run.stdout, (run.returncode, run.stdout, run.stderr)
