// simt.cpp — fibers, scheduler and collectives of the SIMT emulator (tests only, see simt.h).
#include <cstdlib>
#include "simt.h"

#include <deque>
#include <unordered_map>

#include <signal.h>
#include <sys/mman.h>
#include <unistd.h>

namespace simt {

static State g_state;
State& state() { return g_state; }

// ---- context switch (x86-64 System V): callee-saved registers + stack pointer -----------------------
extern "C" void simt_switch(void** save_sp, void* load_sp);
asm(R"(
    .text
    .globl simt_switch
    .type simt_switch,@function
simt_switch:
    pushq %rbp
    pushq %rbx
    pushq %r12
    pushq %r13
    pushq %r14
    pushq %r15
    movq %rsp, (%rdi)
    movq %rsi, %rsp
    popq %r15
    popq %r14
    popq %r13
    popq %r12
    popq %rbx
    popq %rbp
    ret
    .size simt_switch,.-simt_switch
)");

constexpr size_t kStackBytes = 256 * 1024;

static void fiber_main() {
    State& S = g_state;
    Fiber* f = S.cur;
    (*S.body)();
    f->done = true;
    S.warps[f->warp].exited |= 1u << f->lane;
    ++S.progress;
    simt_switch(&f->sp, S.sched_sp);
    abort();      // a finished fiber is never resumed
}

void yield() {
    State& S = g_state;
    Fiber* f = S.cur;
    simt_switch(&f->sp, S.sched_sp);
}

static void prepare(Fiber& f) {
    if (!f.stack) f.stack = static_cast<unsigned char*>(aligned_alloc(64, kStackBytes));
    uintptr_t top = (reinterpret_cast<uintptr_t>(f.stack) + kStackBytes) & ~(uintptr_t)15;
    void** sp = reinterpret_cast<void**>(top);
    *--sp = nullptr;                                     // fake return address of fiber_main (keeps rsp = 8 mod 16 at entry)
    *--sp = reinterpret_cast<void*>(&fiber_main);        // `ret` of the first switch jumps here
    for (int i = 0; i < 6; ++i) *--sp = nullptr;         // rbp rbx r12 r13 r14 r15
    f.sp = sp;
    f.done = false;
}

// warp state lives in deques so that references stay valid while lanes wait
static std::vector<std::deque<Pending>> g_pending;

static void die(const char* what) {
    State& S = g_state;
    fprintf(stderr, "[simt] %s (block %u, thread %u)\n", what, S.bid.x, S.cur ? S.cur->tid.x : 0u);
    abort();
}

uint64_t collective(int op, uint32_t mask, uint64_t value, int arg, const char* file, int line) {
    State& S = g_state;
    Fiber* f = S.cur;
    const int lane = f->lane;
    if (!((mask >> lane) & 1u)) die("collective called by a lane that is not in its mask");
    std::deque<Pending>& list = g_pending[f->warp];
    Pending* p = nullptr;
    for (Pending& q : list)
        if (q.mask == mask) { p = &q; break; }
    if (!p) {
        list.emplace_back();
        p = &list.back();
        p->mask = mask;
    }
    if (p->arrived == 0) {
        p->op = op;
        p->file = file;
        p->line = line;
    } else if (p->op != op || p->line != line || strcmp(p->file, file) != 0) {
        // a divergent warp: some lanes took a branch the others did not, and both sides reached a collective
        fprintf(stderr, "[simt] lanes of one warp wait in different collectives with mask %08x: %s:%d (lanes %08x) vs %s:%d (lane %d)\n",
                mask, p->file, p->line, p->arrived, file, line, lane);
        die("divergent collective");
    }
    if ((p->arrived >> lane) & 1u) die("a lane re-entered a collective that has not completed");
    p->val[lane] = value;
    p->arg[lane] = arg;
    p->arrived |= 1u << lane;
    const uint32_t my_gen = p->gen;
    if (p->arrived == mask) {
        uint64_t all = 0;
        switch (op) {
            case OP_BALLOT:
                for (int l = 0; l < kWarp; ++l) if (((mask >> l) & 1u) && p->val[l]) all |= 1ull << l;
                break;
            case OP_RED_ADD:
                for (int l = 0; l < kWarp; ++l) if ((mask >> l) & 1u) all = (uint32_t)(all + p->val[l]);
                break;
            case OP_RED_MAX:
                for (int l = 0; l < kWarp; ++l) if ((mask >> l) & 1u) all = std::max<uint64_t>(all, (uint32_t)p->val[l]);
                break;
            case OP_RED_OR:
                for (int l = 0; l < kWarp; ++l) if ((mask >> l) & 1u) all |= (uint32_t)p->val[l];
                break;
            default: break;
        }
        for (int l = 0; l < kWarp; ++l) {
            if (!((mask >> l) & 1u)) continue;
            uint64_t r = 0;
            switch (op) {
                case OP_SYNC: break;
                case OP_SHFL: { const int src = p->arg[l] & 31; r = ((mask >> src) & 1u) ? p->val[src] : p->val[l]; break; }
                case OP_SHFL_UP: { const int src = l - p->arg[l]; r = (src >= 0 && ((mask >> src) & 1u)) ? p->val[src] : p->val[l]; break; }
                case OP_SHFL_XOR: { const int src = (l ^ p->arg[l]) & 31; r = ((mask >> src) & 1u) ? p->val[src] : p->val[l]; break; }
                case OP_MATCH:
                    for (int m = 0; m < kWarp; ++m) if (((mask >> m) & 1u) && p->val[m] == p->val[l]) r |= 1ull << m;
                    break;
                default: r = all; break;
            }
            p->res[l] = r;
        }
        p->arrived = 0;
        ++p->gen;
        ++S.progress;
    } else {
        while (p->gen == my_gen) yield();
    }
    return p->res[lane];
}

void block_barrier() {
    State& S = g_state;
    const uint32_t n = S.bdim.x;
    const uint32_t my_gen = S.block_gen;
    if (++S.block_arrived == n) {
        S.block_arrived = 0;
        ++S.block_gen;
        ++S.progress;
    } else {
        while (S.block_gen == my_gen) yield();
    }
}

// ---- LT_SIMT_MEMCHECK=1: device buffers and the dynamic shared memory of a launch end at a guard page ----------
// (what compute-sanitizer's memcheck finds on the device, for accesses past the END of a buffer: the buffer is
// placed so that its last 16-byte unit touches an inaccessible page, and the page before the mapping is
// inaccessible as well; the fault is reported with the block and thread that made the access)
static bool memcheck() {
    static const bool on = [] { const char* e = getenv("LT_SIMT_MEMCHECK"); return e && e[0] == '1'; }();
    return on;
}
// LT_SIMT_FILL=<byte>: what fresh device buffers and a block's shared memory hold before the kernels write them
// (default 0xCD / 0xA5).  On the GPU that is whatever the previous owner left: a result that changes with the
// fill depends on uninitialised memory (compute-sanitizer's initcheck, by differential runs).
static int fill_byte(int dflt) {
    static const int v = [] { const char* e = getenv("LT_SIMT_FILL"); return e ? (int)strtol(e, nullptr, 0) & 0xFF : -1; }();
    return v < 0 ? dflt : v;
}
struct Guarded { void* base; size_t len; };
static std::unordered_map<void*, Guarded> g_guarded;

static void on_fault(int, siginfo_t* info, void*) {
    State& S = g_state;
    char msg[200];
    const int n = snprintf(msg, sizeof msg, "[simt] memcheck: invalid access at %p (block %u, thread %u)\n", info->si_addr, S.bid.x,
                           S.cur ? S.cur->tid.x : 0u);
    if (n > 0 && write(2, msg, (size_t)n) < 0) {}
    abort();
}

static void* guarded_alloc(size_t n, int fill) {
    static const bool installed = [] {
        struct sigaction sa;
        memset(&sa, 0, sizeof sa);
        sa.sa_sigaction = on_fault;
        sa.sa_flags = SA_SIGINFO;
        sigaction(SIGSEGV, &sa, nullptr);
        return true;
    }();
    (void)installed;
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    const size_t body = (n + 15) & ~(size_t)15;
    const size_t pages = (body + page - 1) / page + 2;               // guard | data ... | guard
    unsigned char* base = static_cast<unsigned char*>(mmap(nullptr, pages * page, PROT_NONE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0));
    if (base == MAP_FAILED) return nullptr;
    if (mprotect(base + page, (pages - 2) * page, PROT_READ | PROT_WRITE) != 0) { munmap(base, pages * page); return nullptr; }
    unsigned char* p = base + (pages - 1) * page - body;
    memset(p, fill, body);
    g_guarded[p] = Guarded{base, pages * page};
    return p;
}
static void guarded_free(void* p) {
    auto it = g_guarded.find(p);
    if (it == g_guarded.end()) { fprintf(stderr, "[simt] memcheck: free of %p, which is no live device buffer\n", p); abort(); }
    munmap(it->second.base, it->second.len);
    g_guarded.erase(it);
}
// the device buffers live under LT_SIMT_MEMCHECK=1: a leak check compares the count before and after
extern "C" size_t simt_live_buffers() { return g_guarded.size(); }

void* dev_alloc(size_t n) {
    if (memcheck()) return guarded_alloc(n ? n : 1, fill_byte(0xCD));
    void* p = aligned_alloc(256, (n + 255) & ~(size_t)255);
    if (p) memset(p, fill_byte(0xCD), n);
    return p;
}
void dev_free(void* p) {
    if (!p) return;
    if (memcheck()) guarded_free(p); else free(p);
}

static std::vector<unsigned char> g_smem;

void launch(dim3 grid, dim3 block, size_t smem_bytes, const std::function<void()>& body) {
    State& S = g_state;
    if (S.cur) die("nested launch");
    const unsigned nthreads = block.x;
    if (nthreads == 0 || grid.x == 0) return;
    void* guarded_smem = nullptr;
    if (memcheck()) {
        guarded_smem = guarded_alloc(smem_bytes ? smem_bytes : 1, fill_byte(0xA5));
        if (!guarded_smem) die("memcheck: no memory for the shared-memory mapping");
        S.smem = static_cast<unsigned char*>(guarded_smem);
    } else {
        if (g_smem.size() < smem_bytes + 64) g_smem.resize(smem_bytes + 64);
        S.smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(g_smem.data()) + 63) & ~(uintptr_t)63);
    }
    S.bdim = block;
    S.gdim = grid;
    S.body = &body;
    if (S.fibers.size() < nthreads) S.fibers.resize(nthreads);
    const unsigned nwarps = (nthreads + kWarp - 1) / kWarp;
    // Blocks run one after another; LT_SIMT_BLOCK_ORDER=reverse runs them last to first, so that a kernel whose
    // result depends on which of two CTAs writes last (a race on the GPU) fails one of the two orders.
    const char* order_env = getenv("LT_SIMT_BLOCK_ORDER");
    const bool reverse = order_env && order_env[0] == 'r';
    for (unsigned bi = 0; bi < grid.x; ++bi) {
        const unsigned b = reverse ? grid.x - 1 - bi : bi;
        S.bid = uint3{b, 0, 0};
        // poison shared memory: a kernel that relies on stale contents fails the same way everywhere
        memset(S.smem, fill_byte(0xA5), smem_bytes);
        S.warps.assign(nwarps, Warp());
        g_pending.assign(nwarps, std::deque<Pending>());
        S.block_arrived = 0;
        for (unsigned t = 0; t < nthreads; ++t) {
            Fiber& f = S.fibers[t];
            prepare(f);
            f.tid = uint3{t, 0, 0};
            f.lane = (int)(t % kWarp);
            f.warp = (int)(t / kWarp);
        }
        // a partial last warp: the missing lanes never arrive, so kernels must not use full masks there
        unsigned live = nthreads;
        while (live > 0) {
            const uint64_t before = S.progress;
            for (unsigned t = 0; t < nthreads; ++t) {
                Fiber& f = S.fibers[t];
                if (f.done) continue;
                S.cur = &f;
                simt_switch(&S.sched_sp, f.sp);
                if (f.done) --live;
            }
            S.cur = nullptr;
            if (live > 0 && S.progress == before) {
                fprintf(stderr, "[simt] deadlock in block %u: %u fibers wait for lanes that never arrive\n", b, live);
                for (unsigned w = 0; w < nwarps; ++w)
                    for (const Pending& p : g_pending[w])
                        if (p.arrived) fprintf(stderr, "  warp %u: op %d mask %08x arrived %08x\n", w, p.op, p.mask, p.arrived);
                abort();
            }
        }
    }
    S.cur = nullptr;
    S.body = nullptr;
    if (guarded_smem) guarded_free(guarded_smem);
}

}  // namespace simt
