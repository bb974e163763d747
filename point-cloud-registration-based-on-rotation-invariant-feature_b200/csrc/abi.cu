// abi.cu — ABI bookkeeping for libri_b200.so (include/ri_b200.h).
#include "ri_common.cuh"

#include <string.h>

extern "C" int ri_abi_version(void) { return 11; }

// ---- environment knobs (DESIGN.md §11): read once per process, here
namespace {
int env_int(const char* name, int unset)
{
    const char* ev = getenv(name);
    return ev ? atoi(ev) : unset;
}
RiEnv& env_instance()
{
    static RiEnv env = [] {
        RiEnv e;
        e.carveout_pct = env_int("RI_CARVEOUT_PCT", 100);
        if (e.carveout_pct < 1 || e.carveout_pct > 100) e.carveout_pct = 100;
        e.devox_stream = env_int("RI_DEVOX_STREAM", -1);
        e.devox_tile_kb = env_int("RI_DEVOX_TILE_KB", -1);
        e.devox_ring_kb = env_int("RI_DEVOX_RING_KB", -1);
        e.devox_pad_kb = env_int("RI_DEVOX_PAD_KB", -1);
        e.devox_dbg_skip = getenv("RI_DEVOX_DBG_SKIP") != nullptr;
        e.fill_ring = env_int("RI_FILL_RING", -1);
        e.fill_ctas = env_int("RI_FILL_CTAS", -1);
        e.fill_pad_kb = env_int("RI_FILL_PAD_KB", -1);
        e.fill_group = env_int("RI_FILL_GROUP", -1);
        e.fill_warps = env_int("RI_FILL_WARPS", -1);
        e.fill_listcap = env_int("RI_FILL_LISTCAP", -1);
        e.fill_tile_cells = env_int("RI_FILL_TILE", -1);
        e.vox_atomic = getenv("RI_VOX_ATOMIC") != nullptr;
        e.ppf_maxl1 = env_int("RI_PPF_MAXL1", 0) == 1;
        e.match_pair = env_int("RI_MATCH_PAIR", -1);
        e.match_dbg = getenv("RI_MATCH_DBG") != nullptr;
        e.match_tma = env_int("RI_MATCH_TMA", -1);
        return e;
    }();
    return env;
}
}  // namespace

const RiEnv& ri_env() { return env_instance(); }

// Tests and tools: set one knob of the already-initialised environment by its variable name ("RI_DEVOX_STREAM", ...).
// Returns RI_ERR_BAD_ARG for a name that cannot be changed at run time.
extern "C" int ri_debug_set_knob(const char* name, int value)
{
    RiEnv& e = env_instance();
    if (name == nullptr) return RI_ERR_BAD_ARG;
    if (!strcmp(name, "RI_DEVOX_STREAM")) e.devox_stream = value;
    else if (!strcmp(name, "RI_MATCH_PAIR")) e.match_pair = value;
    else if (!strcmp(name, "RI_DEVOX_DBG_SKIP")) e.devox_dbg_skip = value;
    else if (!strcmp(name, "RI_MATCH_DBG")) e.match_dbg = value;
    else if (!strcmp(name, "RI_MATCH_TMA")) e.match_tma = value;
    else if (!strcmp(name, "RI_VOX_ATOMIC")) e.vox_atomic = value;
    else if (!strcmp(name, "RI_FILL_WARPS")) e.fill_warps = value;
    else if (!strcmp(name, "RI_FILL_LISTCAP")) e.fill_listcap = value;
    else if (!strcmp(name, "RI_FILL_RING")) e.fill_ring = value;
    else if (!strcmp(name, "RI_FILL_GROUP")) e.fill_group = value;
    else return RI_ERR_BAD_ARG;
    return RI_OK;
}

// Debug aid for tools/timeline.py: one thread stores the GPU's nanosecond timer; enqueued between the kernels of a
// step it yields the start/end of every kernel on every stream (a profiler cannot show concurrent branches).
namespace {
__global__ void stamp_kernel(unsigned long long* slot)
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    *slot = t;
}
}  // namespace

extern "C" int ri_debug_stamp(unsigned long long* slot, void* stream)
{
    stamp_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(slot);
    RI_LAUNCH_CHECK();
    return RI_OK;
}
