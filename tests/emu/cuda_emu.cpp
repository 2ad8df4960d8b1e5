// cuda_emu.cpp -- TEST INFRASTRUCTURE ONLY (see cuda_emu.h).
// Fiber scheduler: one CTA = blockDim.x ucontext fibers on one OS thread.
#include "cuda_emu.h"

#include <sys/mman.h>

#include <mutex>

namespace cuemu {

thread_local Idx t_threadIdx, t_blockIdx, t_blockDim, t_gridDim;
thread_local Cta *t_cta = nullptr;

static void fiber_entry() {
    Cta *c = t_cta;
    (*c->body)();
    Fiber &f = c->fib[c->cur];
    f.done = true;
    c->live -= 1;
    swapcontext(&f.ctx, &c->sched);
}

void yield_until(const long *counter, long target) {
    if (*counter >= target) return;
    Cta *c = t_cta;
    Fiber &f = c->fib[c->cur];
    f.wait_counter = counter;
    f.wait_target = target;
    swapcontext(&f.ctx, &c->sched);
}

static void run_cta(Cta &c, Idx bidx, dim3 block, dim3 grid) {
    t_cta = &c;
    t_blockIdx = bidx;
    t_blockDim = Idx{block.x, block.y, block.z};
    t_gridDim = Idx{grid.x, grid.y, grid.z};
    c.bar_arrived = 0;
    for (auto &g : c.bar_gen) g = 0;
    for (auto &w : c.warps) { w.arrived = 0; memset(w.gen, 0, sizeof(w.gen)); }
    c.live = c.nthreads;
    for (int t = 0; t < c.nthreads; ++t) {
        Fiber &f = c.fib[t];
        f.done = false;
        f.wait_counter = nullptr;
        getcontext(&f.ctx);
        f.ctx.uc_stack.ss_sp = f.stack;
        f.ctx.uc_stack.ss_size = kStack;
        f.ctx.uc_link = nullptr;
        makecontext(&f.ctx, (void (*)())fiber_entry, 0);
    }
    while (c.live > 0) {
        bool progressed = false;
        for (int t = 0; t < c.nthreads; ++t) {
            Fiber &f = c.fib[t];
            if (f.done) continue;
            if (f.wait_counter) {
                if (*f.wait_counter < f.wait_target) continue;
                f.wait_counter = nullptr;
            }
            c.cur = t;
            t_threadIdx = Idx{(unsigned)t % block.x, ((unsigned)t / block.x) % block.y,
                              (unsigned)t / (block.x * block.y)};
            swapcontext(&c.sched, &f.ctx);
            progressed = true;
        }
        if (!progressed) {
            fprintf(stderr, "cuda_emu: deadlock in CTA (%u,%u,%u): %d fibers blocked\n", bidx.x,
                    bidx.y, bidx.z, c.live);
            abort();
        }
    }
}

void run_grid(const std::function<void()> &body, dim3 grid, dim3 block, size_t smem) {
    const int nthreads = (int)(block.x * block.y * block.z);
    const long nblocks = (long)grid.x * grid.y * grid.z;
    if (nthreads <= 0 || nblocks <= 0) return;
    int nworkers = (int)std::thread::hardware_concurrency();
    if (nworkers < 1) nworkers = 1;
    if (nworkers > 16) nworkers = 16;
    if (nworkers > nblocks) nworkers = (int)nblocks;
    std::atomic<long> next{0};
    auto worker = [&]() {
        Cta c;
        c.nthreads = nthreads;
        c.fib.resize(nthreads);
        c.bar_gen.assign(nthreads, 0);
        c.warps.resize((nthreads + 31) / 32);
        c.body = &body;
        char *stacks = (char *)mmap(nullptr, kStack * (size_t)nthreads, PROT_READ | PROT_WRITE,
                                    MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
        if (stacks == (char *)MAP_FAILED) { perror("cuda_emu mmap"); abort(); }
        for (int t = 0; t < nthreads; ++t) c.fib[t].stack = stacks + kStack * (size_t)t;
        c.smem = (unsigned char *)aligned_alloc(128, ((smem + 127) / 128 + 1) * 128);
        for (;;) {
            const long b = next.fetch_add(1);
            if (b >= nblocks) break;
            Idx bidx{(unsigned)(b % grid.x), (unsigned)((b / grid.x) % grid.y),
                     (unsigned)(b / ((long)grid.x * grid.y))};
            run_cta(c, bidx, block, grid);
        }
        free(c.smem);
        munmap(stacks, kStack * (size_t)nthreads);
    };
    if (nworkers == 1) {
        worker();
    } else {
        std::vector<std::thread> pool;
        for (int i = 0; i < nworkers; ++i) pool.emplace_back(worker);
        for (auto &th : pool) th.join();
    }
}

}  // namespace cuemu
