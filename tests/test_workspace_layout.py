"""CPU: the workspace layout helper (ws_layout / ws_room / ws_append in csrc/common.cuh) sizes a buffer from the same code
that carves it, and turns a layout that takes more than was reserved into an error instead of an out-of-bounds slice.
Compiled host-only against a stand-in ws_reserve: no device memory is touched."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHECK = r"""
#include "common.cuh"
#include <stdarg.h>
static char g_err[512];
void dppo_set_error(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap); }
int ws_reserve(Workspace& w, size_t bytes, cudaStream_t) {      // grow-only, no slack: any extra take overflows
    if (bytes > w.cap) { w.base = (char*)(uintptr_t)0x100000; w.cap = bytes; }
    return 0;
}
#define EXPECT(c) do { if (!(c)) { printf("failed: %s (line %d)\n", #c, __LINE__); return 1; } } while (0)
int main() {
    Workspace w;
    float* a; int* b;
    // reserved = the high-water mark, including the room of a nested program; every slice 256-byte aligned
    EXPECT(ws_layout(w, 0, [&] { a = ws_take<float>(w, 1000); b = ws_take<int>(w, 3); ws_room(w, [&] { ws_take<char>(w, 5000); }); }) == 0);
    EXPECT(w.cap == 4096 + 256 + 5120 && w.used == 4096 + 256);
    EXPECT((uintptr_t)a % 256 == 0 && (char*)b - (char*)a == 4096);
    // the nested program appends what the room was made for
    const size_t mark = w.used;
    EXPECT(ws_append(w, [&] { ws_take<char>(w, 5000); }) == 0);
    w.used = mark;
    // one more slice than the caller made room for: an error
    EXPECT(ws_append(w, [&] { ws_take<char>(w, 5000); ws_take<float>(w, 1); }) == -7);
    EXPECT(strstr(g_err, "workspace layout takes 9728 bytes, 9472 reserved"));
    // a layout whose second pass takes more than its counting pass: an error before any pointer is handed out
    Workspace w2; int pass = 0;
    EXPECT(ws_layout(w2, 0, [&] { ws_take<float>(w2, 100); if (pass++) ws_take<float>(w2, 100); }) == -7);
    printf("ok\n");
    return 0;
}
"""


def test_layout_sizes_and_checks(tmp_path):
    src = tmp_path / "check.cu"
    src.write_text(CHECK)
    exe = tmp_path / "check"
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-I", os.path.join(ROOT, "diffusionpolicyoptimization_b200", "csrc"), "-o", str(exe), str(src)],
                   check=True, capture_output=True, text=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stdout + r.stderr
