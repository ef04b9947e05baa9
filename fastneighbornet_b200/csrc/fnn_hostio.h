// fnn_hostio.h — pieces shared by the host-only file loaders (fnn_phylip.cpp, fnn_align.cpp): a read-only mmap of the
// input, line splitting and a fixed pool of worker threads.
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <cstring>
#include <thread>
#include <vector>
#include "fastnn.h"
#include "fnn_common.h"

namespace fnn {

struct Mapped {
    const char* p = nullptr;
    size_t len = 0;
    int fd = -1;
    ~Mapped() {
        if (p && len) munmap((void*)p, len);
        if (fd >= 0) close(fd);
    }
    int open_(const char* path) {
        fd = open(path, O_RDONLY);
        if (fd < 0) { fnn::set_error("cannot open %s", path); return FNN_E_IO; }
        struct stat sb;
        if (fstat(fd, &sb) != 0) { fnn::set_error("cannot stat %s", path); return FNN_E_IO; }
        len = (size_t)sb.st_size;
        if (len == 0) { fnn::set_error("%s: empty file", path); return FNN_E_IO; }
        void* m = mmap(nullptr, len, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) { p = nullptr; fnn::set_error("cannot map %s", path); return FNN_E_IO; }
        p = (const char*)m;
        madvise(m, len, MADV_SEQUENTIAL);
        return FNN_OK;
    }
};

inline const char* line_end(const char* s, const char* end) {
    const char* e = (const char*)memchr(s, '\n', (size_t)(end - s));
    return e ? e : end;
}

// threads <= 0: all host cores, at most 32
inline int pick_threads(int threads) {
    if (threads > 0) return std::min(threads, 256);
    const unsigned hc = std::thread::hardware_concurrency();
    return (int)std::min<unsigned>(hc ? hc : 1, 32);
}

template <class F>
void run_pool(int threads, F&& body) {
    if (threads <= 1) { body(0); return; }
    std::vector<std::thread> pool;
    pool.reserve((size_t)threads);
    for (int t = 0; t < threads; ++t) pool.emplace_back([&body, t] { body(t); });
    for (auto& th : pool) th.join();
}

}  // namespace fnn
