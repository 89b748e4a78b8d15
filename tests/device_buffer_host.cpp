// device_buffer_host.cpp -- scenarios of s3d::DeviceBuffer and s3d::grow_group (3dscan_b200/csrc/scan3d_device_buffer.h)
// on the CPU.  tests/test_device_buffer_host.py compiles it against a stub cuda_runtime.h that prints every cudaMalloc
// ("malloc <id> <bytes>", "fail <bytes>") and cudaFree ("free <id>", "free-unknown <id>"); this file prints the
// buffers' state and section marks in between.  Usage: device_buffer_host <scenario> [k: the k-th cudaMalloc fails]
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <utility>

#include "../3dscan_b200/csrc/scan3d_device_buffer.h"

using s3d::DeviceBuffer;
using s3d::Grow;
using s3d::grow_group;

// "<name> <elements> <allocation id, 0 = null>"
template <class T>
static void show(const char* name, const DeviceBuffer<T>& b)
{
    printf("%s %zu %zu\n", name, b.size(), (size_t)((uintptr_t)b.get() / 256));
}
static void mark(const char* section) { printf("-- %s\n", section); }
static void ret(cudaError_t e) { printf("ret %d\n", (int)e); }

static void ensure_scenario()
{
    DeviceBuffer<double> b;
    show("b", b);
    ret(b.ensure(0));
    mark("first");
    ret(b.ensure(3));
    show("b", b);
    mark("not larger");
    ret(b.ensure(3));
    ret(b.ensure(1));
    ret(b.ensure(0));
    show("b", b);
    mark("larger");
    ret(b.ensure(5));
    show("b", b);
    mark("end");
}

static void fail_scenario()   // run with k = 2
{
    DeviceBuffer<float> b;
    ret(b.ensure(4));
    mark("failing growth");
    ret(b.ensure(8));
    show("b", b);
    mark("retry");
    ret(b.ensure(2));
    show("b", b);
    mark("end");
}

static void move_scenario()
{
    DeviceBuffer<int> a, b;
    a.ensure(4);
    b.ensure(6);
    mark("move");
    DeviceBuffer<int> c(std::move(a));
    show("a", a);
    show("c", c);
    std::swap(b, c);
    show("b", b);
    show("c", c);
    DeviceBuffer<int> d;
    d = std::move(c);
    show("c", c);
    show("d", d);
    mark("end");
}

static void release_scenario()
{
    DeviceBuffer<char> b;
    b.ensure(8);
    mark("release");
    b.release();
    b.release();
    show("b", b);
    mark("end");
}

static void group_scenario()   // also run with k = 6: the growth's second allocation fails
{
    DeviceBuffer<float> a;
    DeviceBuffer<double> b;
    DeviceBuffer<char> c;
    DeviceBuffer<uint16_t> d;
    ret(grow_group(Grow(a, 4), Grow(b, 4), Grow(c, 4), Grow(d, 4)));
    mark("grow");
    ret(grow_group(Grow(a, 8), Grow(b, 8), Grow(c, 2), Grow(d, 8)));
    show("a", a);
    show("b", b);
    show("c", c);
    show("d", d);
    mark("end");
}

int main(int argc, char** argv)
{
    if (argc < 2) return 2;
    if (argc > 2) g_fail_at = atoi(argv[2]);
    const char* s = argv[1];
    if (!strcmp(s, "ensure")) ensure_scenario();
    else if (!strcmp(s, "fail")) fail_scenario();
    else if (!strcmp(s, "move")) move_scenario();
    else if (!strcmp(s, "release")) release_scenario();
    else if (!strcmp(s, "group")) group_scenario();
    else return 2;
    size_t live = 0;
    for (const auto& kv : g_live) live += kv.second;
    printf("live %zu\n", live);
    return 0;
}
