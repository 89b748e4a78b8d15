"""The context's device-memory owner, s3d::DeviceBuffer and its group growth (csrc/scan3d_device_buffer.h), checked on
the CPU: tests/device_buffer_host.cpp is compiled against the real header and a stub CUDA runtime that prints every
cudaMalloc and cudaFree, hands out numbered fake pointers, keeps the live bytes and can fail the k-th allocation.
The rules: an ensure that is not larger makes no call, growth frees before it allocates, a failed allocation leaves
the buffer empty, moves and swaps transfer ownership without a call, the destructor frees exactly once, release is
idempotent, a group releases every member that is too small before it allocates any, and nothing is left live."""
import os
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

STUB = r"""
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#include <map>

typedef int cudaError_t;
constexpr cudaError_t cudaSuccess = 0;
constexpr cudaError_t cudaErrorMemoryAllocation = 2;

inline std::map<uintptr_t, size_t> g_live;   // allocation id -> bytes
inline int g_attempts = 0, g_fail_at = 0;     // g_fail_at: the attempt (1-based) that fails, 0 = none
inline uintptr_t g_next_id = 0;

inline cudaError_t cudaMalloc(void** p, size_t bytes)
{
    if (++g_attempts == g_fail_at) {
        *p = (void*)0xbad00;                   // the header must not keep what a failed call leaves here
        printf("fail %zu\n", bytes);
        return cudaErrorMemoryAllocation;
    }
    const uintptr_t id = ++g_next_id;
    g_live[id] = bytes;
    *p = (void*)(id * 256);
    printf("malloc %zu %zu\n", (size_t)id, bytes);
    return cudaSuccess;
}

inline cudaError_t cudaFree(void* p)
{
    const uintptr_t id = (uintptr_t)p / 256;
    printf(g_live.erase(id) ? "free %zu\n" : "free-unknown %zu\n", (size_t)id);
    return cudaSuccess;
}
"""


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    d = tmp_path_factory.mktemp("devbuf")
    inc = d / "include"
    inc.mkdir()
    (inc / "cuda_runtime.h").write_text(STUB)
    exe = str(d / "device_buffer_host")
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-Wall", "-I", str(inc), "-o", exe,
                           os.path.join(HERE, "device_buffer_host.cpp")])

    def run(scenario, fail_at=0):
        out = subprocess.run([exe, scenario, str(fail_at)], capture_output=True, text=True, check=True).stdout
        lines = out.splitlines()
        assert lines[-1] == "live 0", out                      # every scenario ends with nothing allocated
        assert not any(l.startswith("free-unknown") for l in lines), out
        sections, name = {"": []}, ""
        for l in lines[:-1]:
            if l.startswith("-- "):
                name = l[3:]
                sections[name] = []
            else:
                sections[name].append(l)
        return sections

    return run


def calls(lines):
    return [l for l in lines if l.split()[0] in ("malloc", "fail", "free")]


def test_ensure_allocates_only_when_larger_and_frees_first(driver):
    s = driver("ensure")
    assert s[""] == ["b 0 0", "ret 0"]                         # ensure(0) of an empty buffer: no call
    assert s["first"] == ["malloc 1 24", "ret 0", "b 3 1"]     # 3 doubles
    assert s["not larger"] == ["ret 0", "ret 0", "ret 0", "b 3 1"]
    assert s["larger"] == ["free 1", "malloc 2 40", "ret 0", "b 5 2"]
    assert s["end"] == ["free 2"]                              # the destructor, once


def test_failed_allocation_leaves_the_buffer_empty(driver):
    s = driver("fail", fail_at=2)
    assert s["failing growth"] == ["free 1", "fail 32", "ret 2", "b 0 0"]
    assert s["retry"] == ["malloc 2 8", "ret 0", "b 2 2"]
    assert s["end"] == ["free 2"]


def test_move_and_swap_transfer_ownership_without_a_call(driver):
    s = driver("move")
    assert s[""] == ["malloc 1 16", "malloc 2 24"]
    assert calls(s["move"]) == []
    assert s["move"] == ["a 0 0", "c 4 1", "b 4 1", "c 6 2", "c 0 0", "d 6 2"]
    assert sorted(s["end"]) == ["free 1", "free 2"]            # each owner frees once, the moved-from ones nothing


def test_release_is_idempotent(driver):
    s = driver("release")
    assert s["release"] == ["free 1", "b 0 0"]
    assert s["end"] == []


def test_group_releases_every_short_member_before_allocating(driver):
    s = driver("group")
    assert s["grow"] == ["free 1", "free 2", "free 4", "malloc 5 32", "malloc 6 64", "malloc 7 16", "ret 0",
                         "a 8 5", "b 8 6", "c 4 3", "d 8 7"]  # c holds enough and keeps its memory
    assert sorted(s["end"]) == ["free 3", "free 5", "free 6", "free 7"]


def test_group_stops_at_the_first_failed_allocation(driver):
    s = driver("group", fail_at=6)
    assert s["grow"] == ["free 1", "free 2", "free 4", "malloc 5 32", "fail 64", "ret 2",
                         "a 8 5", "b 0 0", "c 4 3", "d 0 0"]
    assert sorted(s["end"]) == ["free 3", "free 5"]
