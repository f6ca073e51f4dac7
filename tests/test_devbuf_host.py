"""The owners of device memory and captured graphs (DevBuf, GraphExec in gingr_b200/csrc/common.cuh) compiled FOR THE
HOST with g++, with cudaMalloc / cudaFree / cudaGraphExecDestroy replaced by stubs that log every allocation and free:
the shipped header, not a copy, checked for exactly one free per allocation at the moment it is due.  No GPU."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INC = "/usr/local/cuda/include"
pytestmark = pytest.mark.skipif(shutil.which("g++") is None or not os.path.isdir(CUDA_INC), reason="needs g++ and the CUDA headers")

# Log: "+k" = allocation k, "-k" = free of allocation k, "xk" = graph k destroyed, other words = markers of the scenario.
WRAPPER = r'''
#include <stdint.h>
#include <stdlib.h>
#include <string>
#include <type_traits>
#include <utility>
#include "common.cuh"

static_assert(!std::is_copy_constructible<DevBuf<double>>::value && !std::is_copy_assignable<DevBuf<double>>::value,
              "DevBuf must not be copied: two copies would free one block twice");
static_assert(std::is_nothrow_move_constructible<DevBuf<double>>::value && std::is_nothrow_move_assignable<DevBuf<double>>::value,
              "DevBuf moves");
static_assert(!std::is_copy_constructible<GraphExec>::value && !std::is_copy_assignable<GraphExec>::value,
              "GraphExec must not be copied");
static_assert(std::is_nothrow_move_constructible<GraphExec>::value && std::is_nothrow_move_assignable<GraphExec>::value,
              "GraphExec moves");

static std::string g_log;
static int g_next = 0;
static void mark(const char* w) { g_log += w; g_log += ' '; }

extern "C" {
cudaError_t cudaMalloc(void** p, size_t bytes) {
  int* b = (int*)malloc(bytes < sizeof(int) ? sizeof(int) : bytes);
  *b = ++g_next;
  *p = b;
  mark(("+" + std::to_string(*b)).c_str());
  return cudaSuccess;
}
cudaError_t cudaFree(void* p) {
  mark(("-" + std::to_string(*(int*)p)).c_str());
  free(p);
  return cudaSuccess;
}
cudaError_t cudaGraphExecDestroy(cudaGraphExec_t g) {
  mark(("x" + std::to_string((uintptr_t)g)).c_str());
  return cudaSuccess;
}

static cudaGraphExec_t fake_graph(uintptr_t k) { return reinterpret_cast<cudaGraphExec_t>(k); }

const char* scenario(int which) {
  g_log.clear();
  g_next = 0;
  if (which == 0) {          // leaving scope frees
    { DevBuf<double> a; a.alloc(4); mark("in"); }
    mark("out");
  } else if (which == 1) {   // alloc keeps a block that is big enough, else frees it before allocating the larger one
    DevBuf<double> a;
    a.alloc(8); a.alloc(8); a.alloc(3);
    mark(a.n == 8 ? "kept" : "lost");
    a.alloc(9);
    mark(a.n == 9 ? "grown" : "wrong");
  } else if (which == 2) {   // move construction transfers the block
    {
      DevBuf<double> a;
      a.alloc(4);
      {
        DevBuf<double> b(std::move(a));
        mark(a.p == nullptr && a.n == 0 && b.n == 4 ? "moved" : "not-moved");
      }
      mark("b-gone");
    }
    mark("a-gone");
  } else if (which == 3) {   // move assignment frees the target's block, then takes the source's
    {
      DevBuf<double> a, b;
      a.alloc(4); b.alloc(4);
      b = std::move(a);
      mark(a.p == nullptr && b.n == 4 ? "assigned" : "not-assigned");
    }
    mark("out");
  } else if (which == 4) {   // GraphExec: reset destroys once, a second reset and the destructor of an empty owner do nothing
    {
      GraphExec g;
      g.h = fake_graph(1);
      g.reset();
      mark(g.h == nullptr ? "reset" : "still-set");
      g.reset();
      mark("again");
      g.h = fake_graph(2);
    }
    mark("out");
  } else if (which == 5) {   // GraphExec moves
    {
      GraphExec a;
      a.h = fake_graph(3);
      GraphExec b(std::move(a));
      GraphExec c;
      c.h = fake_graph(4);
      c = std::move(b);
      mark(a.h == nullptr && b.h == nullptr ? "moved" : "not-moved");
    }
    mark("out");
  }
  return g_log.c_str();
}
}
'''


@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    d = tmp_path_factory.mktemp("hostdevbuf")
    src = d / "wrap.cpp"
    src.write_text(WRAPPER)
    so = str(d / "libhostdevbuf.so")
    # -Bsymbolic: the header's calls bind to the stubs above even when the real CUDA runtime is already loaded globally
    cmd = ["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wno-attributes", "-I" + CUDA_INC,
           "-I" + os.path.join(ROOT, "gingr_b200", "csrc"), str(src), "-o", so]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    lib = ctypes.CDLL(so)
    lib.scenario.restype = ctypes.c_char_p
    lib.scenario.argtypes = [ctypes.c_int]
    return lib


def _log(lib, which):
    return lib.scenario(which).decode().split()


def test_devbuf_leaving_scope_frees(hostlib):
    assert _log(hostlib, 0) == ["+1", "in", "-1", "out"]


def test_devbuf_alloc_grows_only_and_frees_before_it_allocates(hostlib):
    assert _log(hostlib, 1) == ["+1", "kept", "-1", "+2", "grown", "-2"]


def test_devbuf_move_construction_transfers_ownership(hostlib):
    assert _log(hostlib, 2) == ["+1", "moved", "-1", "b-gone", "a-gone"]


def test_devbuf_move_assignment_frees_the_old_block_once(hostlib):
    assert _log(hostlib, 3) == ["+1", "+2", "-2", "assigned", "-1", "out"]


def test_graph_exec_reset_and_destructor_destroy_once(hostlib):
    assert _log(hostlib, 4) == ["x1", "reset", "again", "x2", "out"]


def test_graph_exec_moves(hostlib):
    assert _log(hostlib, 5) == ["x4", "moved", "x3", "out"]
