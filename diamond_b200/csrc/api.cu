// libdiamond_b200.so — C ABI (include/diamond_b200.h) over the sm_100a kernels.
#include <cstdlib>
#include <memory>
#include <mutex>
#include <map>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/diamond_b200.h"
#include "aux_kernels.cuh"
#include "conv_tc.cuh"
#include "conv_fused.cuh"
#include "wgrad_tc.cuh"
#include "bwd_kernels.cuh"

using namespace dmd;

// ---------------------------------------------------------------------------------------------- errors / counters
static thread_local std::string g_err;
static thread_local long long g_launches = 0;

static int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
#define DMD_CHECK(cond, ...) \
  do {                       \
    if (!(cond)) return fail(__VA_ARGS__); \
  } while (0)
#define DMD_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess) { (void)cudaGetLastError(); return fail("%s failed: %s", #expr, cudaGetErrorString(e__)); } \
  } while (0)
#define DMD_LAUNCH_OK()                                                                 \
  do {                                                                                  \
    ++g_launches;                                                                       \
    cudaError_t e__ = cudaGetLastError();                                               \
    if (e__ != cudaSuccess) return fail("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

extern "C" int dmd_version(void) { return DMD_VERSION; }
extern "C" const char* dmd_last_error(void) { return g_err.c_str(); }
extern "C" long long dmd_launch_count(int reset) {
  long long v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

// ---- kernel trace (diagnostics; scripts/ktrace.py): launches issued between dmd_ktrace_begin and dmd_ktrace_end get one slot
// each in a device buffer and stamp the GPU nanosecond timer when their inputs are ready
static long long* g_kt_buf = nullptr;
static int g_kt_cap = 0, g_kt_n = 0;
static bool g_kt_on = false;
static std::vector<std::string> g_kt_names;
static long long* kt_slot(const char* kind, int grid, int aux) {
  if (!g_kt_on || g_kt_n >= g_kt_cap) return nullptr;
  char buf[96];
  snprintf(buf, sizeof(buf), "%s grid=%d aux=%d", kind, grid, aux);
  g_kt_names.push_back(buf);
  return g_kt_buf + g_kt_n++;
}
extern "C" int dmd_ktrace_begin(int capacity) {
  if (g_kt_cap < capacity) {
    if (g_kt_buf) cudaFree(g_kt_buf);
    if (cudaMalloc(&g_kt_buf, (size_t)capacity * 8) != cudaSuccess) { g_kt_buf = nullptr; g_kt_cap = 0; g_err = "ktrace: cudaMalloc failed"; return 1; }
    g_kt_cap = capacity;
  }
  cudaMemset(g_kt_buf, 0, (size_t)g_kt_cap * 8);
  g_kt_n = 0; g_kt_names.clear(); g_kt_on = true;
  return 0;
}
// stops assigning slots; copies the stamps (ns) to `stamps` and returns the number of traced launches (call after a device sync)
extern "C" int dmd_ktrace_end(long long* stamps, int capacity) {
  g_kt_on = false;
  const int n = g_kt_n < capacity ? g_kt_n : capacity;
  if (n > 0 && stamps) cudaMemcpy(stamps, g_kt_buf, (size_t)n * 8, cudaMemcpyDeviceToHost);
  return n;
}
extern "C" const char* dmd_ktrace_name(int i) { return (i >= 0 && i < (int)g_kt_names.size()) ? g_kt_names[i].c_str() : ""; }

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline int gn_group_size(int C) {  // blocks.py:12,27: num_groups = max(1, C // 32)
  int G = C / 32 > 1 ? C / 32 : 1;
  return C / G;
}

// ---------------------------------------------------------------------------------------------- conv launcher
static size_t plc16_bytes(int B, int H, int W, int C) {
  const Plc g = plc_geometry(B, H, W);
  return (size_t)(round_up(C, 16) / 8) * g.Qalloc * 16;
}
extern "C" size_t dmd_plc16_bytes(int B, int H, int W, int C) { return plc16_bytes(B, H, W, C); }

// Tuning knobs (read once per name): integers from the environment, for sweeps on the GPU box without a rebuild.
static int tune_int(const char* name, int dflt) {
  static std::mutex mu;
  static std::map<std::string, int> cache;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(name);
  if (it != cache.end()) return it->second;
  const char* v = getenv(name);
  const int r = (v && *v) ? atoi(v) : dflt;
  cache[name] = r;
  return r;
}

static int conv_fill(const dmd_conv_desc* d, ConvParams* p, size_t* smem, int* tmem_cols) {
  DMD_CHECK(d->src0 && d->out && d->wpk, "conv: null src0/out/wpk");
  DMD_CHECK(d->taps == 9 || d->taps == 1, "conv: taps must be 1 or 9 (got %d)", d->taps);
  DMD_CHECK(d->stride == 1 || d->stride == 2, "conv: stride must be 1 or 2");
  DMD_CHECK(d->C0 > 0 && d->C0 % 16 == 0 && d->C1 % 16 == 0 && d->C0 + d->C1 <= kMaxCin, "conv: operand channels must be multiples of 16, total <= %d (C0=%d C1=%d)", kMaxCin, d->C0, d->C1);
  DMD_CHECK((d->C1 == 0) == (d->src1 == nullptr), "conv: src1/C1 mismatch");
  if (d->precise) DMD_CHECK(d->src0_lo && ((d->C1 == 0) == (d->src1_lo == nullptr)), "conv: precise mode needs the low operand parts");
  DMD_CHECK(d->CoutPad % 16 == 0 && d->CoutPad >= 16 && d->CoutPad <= 128 && d->Cout <= d->CoutPad && d->Cout > 0, "conv: bad Cout=%d CoutPad=%d", d->Cout, d->CoutPad);
  memset(p, 0, sizeof(*p));
  {
    const uint8_t* hi[2] = {(const uint8_t*)d->src0, (const uint8_t*)d->src1};
    const uint8_t* lo[2] = {(const uint8_t*)d->src0_lo, (const uint8_t*)d->src1_lo};
    const int cs[2] = {d->C0, d->C1};
    const int nsrc = d->C1 ? 2 : 1;
    int n = 0;
    for (int rep = 0; rep < (d->precise ? 3 : 1); ++rep)  // [hi | lo | hi] against weights [W_hi | W_hi | W_lo]
      for (int k = 0; k < nsrc; ++k) { p->seg_base[n] = (rep == 1) ? lo[k] : hi[k]; p->seg_slabs[n] = cs[k] / 16; ++n; }
    p->Cin = (d->C0 + d->C1) * (d->precise ? 3 : 1);
    p->Cextra = 0;
    if (d->wpk_x) {  // fused split-fp16 1x1 projection: [x_hi | x_lo | x_hi] against [W_hi | W_hi | W_lo], centre tap only
      DMD_CHECK(d->xsrc0 && d->xsrc0_lo && d->xC0 > 0 && d->xC0 % 16 == 0 && d->xC1 % 16 == 0 && d->xC0 + d->xC1 <= kMaxCin, "conv: bad fused projection operands");
      DMD_CHECK((d->xC1 == 0) == (d->xsrc1 == nullptr) && (d->xC1 == 0) == (d->xsrc1_lo == nullptr), "conv: fused projection src1 mismatch");
      const uint8_t* xh[2] = {(const uint8_t*)d->xsrc0, (const uint8_t*)d->xsrc1};
      const uint8_t* xl[2] = {(const uint8_t*)d->xsrc0_lo, (const uint8_t*)d->xsrc1_lo};
      const int xc[2] = {d->xC0, d->xC1};
      // the hi parts are loaded ONCE and multiplied by both W_hi and W_lo (two MMAs per slab), the lo parts by W_hi: 2/3 of the
      // slabs of the naive [x_hi | x_lo | x_hi] K order, and each slab holds only the tile's own 128 rows (centre tap: no halo)
      for (int rep = 0; rep < 2; ++rep)
        for (int k = 0; k < (d->xC1 ? 2 : 1); ++k) {
          DMD_CHECK(n < kMaxSegs, "conv: too many operand segments");
          p->seg_base[n] = (rep == 1) ? xl[k] : xh[k]; p->seg_slabs[n] = xc[k] / 16; ++n;
        }
      p->Cextra = 3 * (d->xC0 + d->xC1);
      p->xslabs = 2 * (d->xC0 + d->xC1) / 16;
      p->wpk_extra = reinterpret_cast<const __half*>(d->wpk_x);
      p->bias_extra = d->bias_x;
    }
    p->nseg = n;
  }
  p->B = d->B; p->H = d->H; p->W = d->W; p->taps = d->taps; p->stride = d->stride;
  if (d->stride == 2) DMD_CHECK(p->H % 2 == 0 && p->W % 2 == 0, "conv: stride 2 needs even H,W");
  p->wpk = reinterpret_cast<const __half*>(d->wpk); p->bias = d->bias; p->Cout = d->Cout; p->CoutPad = d->CoutPad;
  p->resid = d->residual; p->out = d->out; p->ostats = d->out_stats; p->ogs = d->out_gs > 0 ? d->out_gs : d->Cout;
  p->dbg = d->debug; p->dbg_buf = (long long*)d->debug_buf;
  const Plc g = plc_geometry(d->B, d->H, d->W);
  p->PW = g.PW; p->PH = g.PH; p->Q = g.Q; p->G = g.G; p->plane_bytes = (unsigned long long)g.Qalloc * 16;
  DMD_CHECK((long long)g.Q * (g.PW > g.PH ? g.PW : g.PH) < (1ll << 32), "conv: problem too large for 32-bit position math");
  // tap-row-stacked mode (TrsEpilogue, conv_tc.cuh): weights packed with dmd_pack_conv_weight(precise = 3)
  p->trs = d->wpk_layout == 1 ? 1 : 0;
  if (p->trs) DMD_CHECK(d->taps == 9 && !d->precise && 3 * d->CoutPad <= 256, "conv: row-stacked weights need a 3x3, non-split conv with CoutPad <= 80");
  p->tile_stride = p->trs ? 126 : kTileM;
  const int halo = p->trs ? g.PW : (d->taps == 9 ? g.PW + 1 : 0);
  p->P = kTileM + 2 * halo; p->Palloc = p->P | 1;
  if (tune_int("DMD_CONV_PALLOC8", 0)) p->Palloc = round_up(p->P, 8);   // experiment: 128-byte aligned slab / chunk bases
  if (d->out_stats) {
    const int L4 = d->Cout / 4;
    DMD_CHECK(g.PH * g.PW >= 64, "conv: image too small for the statistics epilogue (a tile may touch at most %d images)", kStatSlots);
    DMD_CHECK(d->Cout % 4 == 0 && (L4 == 4 || L4 == 8 || L4 == 16 || L4 == 32), "conv: out_stats needs Cout in {16,32,64,128} (got %d)", d->Cout);
    DMD_CHECK(d->out_gs == 16 || d->out_gs == 32 || d->out_gs == 64 || d->out_gs == 128, "conv: out_gs must be 16/32/64/128");
    DMD_CHECK(d->Cout % d->out_gs == 0 && d->Cout / d->out_gs <= kMaxOutGroups, "conv: bad output groups");
  }
  p->dPW.init(g.PW); p->dPH.init(g.PH);
  p->num_tiles = (g.Q + p->tile_stride - 1) / p->tile_stride;
  // slab ring: everything that fits next to the resident weights, at most four tiles' worth.  Two epilogue groups (each with
  // its own staging tile) when the ring still gets >= 4 slabs and a CTA sees at least two tiles; else one group.
  const int kslabs = p->Cin / 16 + p->xslabs;
  const uint32_t w_bytes = conv_weight_bytes(p->taps, p->Cin, p->Cextra, p->CoutPad);
  // epilogue organisation: direct (0) unless switched off (DMD_CONV_EPI=0) or a warp's columns would span several GroupNorm groups
  const bool direct = tune_int("DMD_CONV_EPI", 1) != 0 && (!d->out_stats || d->CoutPad <= 64);
  if (p->trs) DMD_CHECK(!d->out_stats || d->CoutPad <= 64, "conv: row-stacked mode computes statistics for CoutPad <= 64");
  int groups = p->trs ? 3 : (direct ? 0 : (tune_int("DMD_CONV_GROUPS", 2) >= 2 ? 2 : 1));
  int stages = 0;
  for (;; groups = 1) {
    const ConvSmemLayout L0 = conv_smem_layout(w_bytes, p->CoutPad, p->Palloc, 0, groups);
    const long long budget = 227ll * 1024 - (long long)L0.total;
    stages = budget > 0 ? (int)(budget / (long long)L0.slab_bytes) : 0;
    if (groups <= 1 || groups == 3 || stages >= (kslabs < 4 ? kslabs + 1 : 4)) break;
  }
  if (stages > 4 * kslabs) stages = 4 * kslabs;
  if (stages > kMaxStages) stages = kMaxStages;
  { const int cap = tune_int("DMD_CONV_MAX_STAGES", kMaxStages); if (cap >= 2 && stages > cap) stages = cap; }
  DMD_CHECK(stages >= 2, "conv: shared memory too small for W=%d Cin=%d CoutPad=%d", p->W, p->Cin, p->CoutPad);
  p->stages = stages;
  p->egroups = groups;
  // row-stacked mode: two epilogue groups on alternate tiles once a CTA sees more than one tile
  p->trs_groups = (p->trs && tune_int("DMD_TRS_GROUPS", 2) == 2 && p->num_tiles > 148) ? 2 : 1;
  *smem = conv_smem_layout(w_bytes, p->CoutPad, p->Palloc, stages, groups).total;
  *tmem_cols = d->CoutPad <= 32 ? 32 : (d->CoutPad <= 64 ? 64 : 128);
  if (p->trs) *tmem_cols = 3 * d->CoutPad <= 64 ? 64 : (3 * d->CoutPad <= 128 ? 128 : 256);   // accumulator = three column blocks
  return 0;
}

// Per-device state: SM count, the >48 KB dynamic shared memory opt-ins (function attributes are per device) and a small
// all-zero buffer (source of the zero row groups of the wgrad kernel).  Initialised on first use of each device, never
// during stream capture.
struct DevState { int num_sms = 0; void* zeros = nullptr; };
static thread_local int g_num_sms = 0;
static thread_local const uint8_t* g_zeros = nullptr;
static int init_kernels() {
  static std::mutex mu;
  static std::map<int, DevState> states;
  int dev = 0;
  DMD_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  auto it = states.find(dev);
  if (it == states.end()) {
    DevState st;
    DMD_CUDA(cudaDeviceGetAttribute(&st.num_sms, cudaDevAttrMultiProcessorCount, dev));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<128, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<256, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<32, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<128, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<32, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<128, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<32, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<64, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_tc_kernel<128, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_fused_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_fused_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(conv_fused_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_cluster_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(linear_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(linear_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    DMD_CUDA(cudaFuncSetAttribute(linear_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    DMD_CUDA(cudaMalloc(&st.zeros, 4096));
    DMD_CUDA(cudaMemset(st.zeros, 0, 4096));
    it = states.emplace(dev, st).first;
  }
  g_num_sms = it->second.num_sms;
  g_zeros = (const uint8_t*)it->second.zeros;
  return 0;
}

// Launch with programmatic stream serialization: the kernel may become resident while its predecessor drains and runs
// its prologue up to griddepcontrol.wait.  Captured into CUDA graphs as a programmatic dependency edge.
template <typename Kernel, typename Params>
static int launch_pdl(Kernel kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Params& p) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = tune_int("DMD_NO_PDL", 0) ? 0 : 1;   // bring-up switch: plain stream-ordered launches
  DMD_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
  DMD_LAUNCH_OK();
  return 0;
}

template <int kCols>
static int conv_launch_t(const ConvParams& p0, size_t smem, cudaStream_t st) {
  if (init_kernels()) return 1;
  const int grid = p0.num_tiles < g_num_sms ? p0.num_tiles : g_num_sms;  // persistent: one CTA per SM
  ConvParams p = p0;
  p.ktrace = kt_slot(p.taps == 9 ? "conv3x3" : "conv1x1", p.num_tiles, (p.Cin + p.Cextra) * 1000 + p.W);
  if (p.egroups == 0) return launch_pdl(conv_tc_kernel<kCols, 0>, dim3(grid), dim3(kConvThreads), smem, st, p);
  if (p.egroups == 2) return launch_pdl(conv_tc_kernel<kCols, 2>, dim3(grid), dim3(kConvThreads), smem, st, p);
  return launch_pdl(conv_tc_kernel<kCols, 1>, dim3(grid), dim3(kConvThreads), smem, st, p);
}

// ---- prep (GroupNorm / AdaGroupNorm / SiLU / upsample -> PLC16 operand)
static int prep_fill(const dmd_prep_desc* d, PrepParams* p, int* nsrc) {
  DMD_CHECK(d->src0 && d->dst0, "prep: null src0/dst0");
  DMD_CHECK(d->C0 % 8 == 0 && d->C1 % 8 == 0 && d->C0 > 0 && d->C0 <= kMaxCin && d->C1 <= kMaxCin, "prep: channels must be multiples of 8 (C0=%d C1=%d)", d->C0, d->C1);
  DMD_CHECK((d->C1 == 0) == (d->src1 == nullptr) && (d->C1 == 0) == (d->dst1 == nullptr), "prep: src1/dst1/C1 mismatch");
  DMD_CHECK(d->mode >= 0 && d->mode <= 2, "prep: bad mode");
  for (int c : {d->C0, d->C1 ? d->C1 : 16}) {
    const int cp = round_up(c, 16);
    DMD_CHECK(cp == 16 || cp == 32 || cp == 64 || cp == 128, "prep: a source must have <= 16/32/64/128 channels after padding (got %d)", c);
  }
  memset(p, 0, sizeof(*p));
  p->s[0].src = d->src0; p->s[0].C = d->C0; p->s[0].Cpad = round_up(d->C0, 16); p->s[0].stats = d->stats0; p->s[0].gs = d->gs0 > 0 ? d->gs0 : 8;
  p->s[0].c_offset = 0; p->s[0].dst = (uint8_t*)d->dst0; p->s[0].dst_raw = (uint8_t*)d->dst_raw0;
  p->s[0].dst_lo = (uint8_t*)d->dst_lo0; p->s[0].dst_raw_lo = (uint8_t*)d->dst_raw_lo0;
  p->s[1].dst_lo = (uint8_t*)d->dst_lo1; p->s[1].dst_raw_lo = (uint8_t*)d->dst_raw_lo1;
  DMD_CHECK(!(d->dst_raw_lo0 && !d->dst_raw0) && !(d->dst_raw_lo1 && !d->dst_raw1), "prep: raw low part needs the raw operand too");
  p->s[1].src = d->src1; p->s[1].C = d->C1; p->s[1].Cpad = round_up(d->C1 > 0 ? d->C1 : 16, 16); p->s[1].stats = d->stats1; p->s[1].gs = d->gs1 > 0 ? d->gs1 : 8;
  p->s[1].c_offset = d->C0; p->s[1].dst = (uint8_t*)d->dst1; p->s[1].dst_raw = (uint8_t*)d->dst_raw1;
  if (d->mode) {
    DMD_CHECK(d->stats0 && d->gs0 > 0 && d->C0 % d->gs0 == 0, "prep: norm mode needs stats0/gs0");
    if (d->C1) DMD_CHECK(d->stats1 && d->gs1 > 0 && d->C1 % d->gs1 == 0, "prep: norm mode needs stats1/gs1");
    if (d->mode == 1) DMD_CHECK(d->film != nullptr, "prep: AdaGroupNorm needs film");
    if (d->mode == 2) DMD_CHECK(d->gamma && d->beta, "prep: GroupNorm needs gamma/beta");
    DMD_CHECK(d->upsample == 0, "prep: norm + upsample unsupported");
  }
  p->B = d->B; p->Hs = d->Hs; p->Ws = d->Ws; p->ups = d->upsample;   // 1 nearest-2x, 2 zero insertion (stride-2 adjoint)
  DMD_CHECK(d->upsample >= 0 && d->upsample <= 2, "prep: upsample must be 0, 1 (nearest 2x) or 2 (zero insertion)");
  DMD_CHECK(d->upsample != 2 || (d->mode == 0 && !d->silu && d->C1 == 0 && !d->dst_raw0 && !d->dst_lo0), "prep: zero insertion is a raw single-source operand");
  p->H = d->upsample ? 2 * d->Hs : d->Hs; p->W = d->upsample ? 2 * d->Ws : d->Ws;
  p->mode = d->mode; p->act = d->silu ? 1 : 0;
  p->film = d->film; p->film_stride = d->film_stride; p->film_off = d->film_off; p->film_ctot = d->C0 + d->C1;
  p->gamma = d->gamma; p->beta = d->beta; p->eps = d->eps;
  const Plc g = plc_geometry(d->B, p->H, p->W);
  DMD_CHECK(g.PH * g.PW >= 32, "prep: image too small");
  // a block touches at most 2 images; low-resolution levels get smaller blocks so that the grid still covers the SMs
  int ppb = g.PH * g.PW >= 256 ? 256 : (g.PH * g.PW / 32) * 32;
  while (ppb > 64 && (g.Qalloc + ppb - 1) / ppb < tune_int("DMD_PREP_MIN_BLOCKS", 2 * 148)) ppb >>= 1;
  ppb = (ppb / 32) * 32;
  p->pos_per_block = ppb;
  DMD_CHECK(d->C0 / (d->gs0 > 0 ? d->gs0 : 8) <= 4 || d->mode == 0, "prep: at most 4 groups per source");
  DMD_CHECK((long long)g.Q * (g.PW > g.PH ? g.PW : g.PH) < (1ll << 32), "prep: problem too large for 32-bit position math");
  p->PW = g.PW; p->PH = g.PH; p->Q = g.Q; p->G = g.G; p->Qalloc = g.Qalloc; p->plane_bytes = (unsigned long long)g.Qalloc * 16;
  p->dPW.init(g.PW); p->dPH.init(g.PH);
  *nsrc = d->C1 ? 2 : 1;
  return 0;
}
static int prep_launch(const PrepParams& p0, int nsrc, cudaStream_t st) {
  PrepParams p = p0;
  p.ktrace = kt_slot("prep", (p.Qalloc + p.pos_per_block - 1) / p.pos_per_block * nsrc, p.mode * 1000 + p.W);
  if (p.ups == 2) {  // zero insertion: its own kernel (single source, raw mode)
    const long long total = (long long)p.Qalloc * (p.s[0].Cpad >> 3);
    return launch_pdl(zero_insert_prep_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, p);
  }
  const dim3 grid((p.Qalloc + p.pos_per_block - 1) / p.pos_per_block, 1, nsrc);
  // the hot cases (norm + SiLU, no upsample, no low part of the normalised operand; raw + raw-low on every source or on none)
  // run on the lean kernel; everything else on the generic one
  bool fast = tune_int("DMD_PREP_FAST", 1) != 0 && p.mode != 0 && p.act && p.ups == 0;
  const bool raw = p.s[0].dst_raw != nullptr;
  for (int k = 0; k < nsrc && fast; ++k) {
    const PrepSrc& S = p.s[k];
    if (S.dst_lo != nullptr || (S.dst_raw != nullptr) != raw || (S.dst_raw_lo != nullptr) != raw || S.Cpad != p.s[0].Cpad || S.C % 8 != 0) fast = false;
  }
  if (fast && (long long)p.B * p.Hs * p.Ws * (p.s[0].C > p.s[nsrc - 1].C ? p.s[0].C : p.s[nsrc - 1].C) >= (1ll << 31)) fast = false;   // 32-bit source indices
  if (fast) {
    const int nch = p.s[0].Cpad >> 3;
    if (nch == 8) return raw ? launch_pdl(prep_fast_kernel<8, true>, grid, dim3(kPrepThreads), 0, st, p) : launch_pdl(prep_fast_kernel<8, false>, grid, dim3(kPrepThreads), 0, st, p);
    if (nch == 4) return raw ? launch_pdl(prep_fast_kernel<4, true>, grid, dim3(kPrepThreads), 0, st, p) : launch_pdl(prep_fast_kernel<4, false>, grid, dim3(kPrepThreads), 0, st, p);
  }
  return launch_pdl(prep_act_kernel, grid, dim3(kPrepThreads), 0, st, p);
}
extern "C" int dmd_prep_plan(const dmd_prep_desc* d, int* blocks, int* pos_per_block, int* sources) {
  DMD_CHECK(d && blocks && pos_per_block && sources, "prep_plan: null argument");
  PrepParams p; int nsrc;
  if (prep_fill(d, &p, &nsrc)) return 1;
  *blocks = (p.Qalloc + p.pos_per_block - 1) / p.pos_per_block; *pos_per_block = p.pos_per_block; *sources = nsrc;
  return 0;
}
extern "C" int dmd_conv_plan(const dmd_conv_desc* d, dmd_conv_plan_info* out) {
  DMD_CHECK(d && out, "conv_plan: null argument");
  ConvParams p; size_t smem; int cols;
  if (conv_fill(d, &p, &smem, &cols)) return 1;
  out->tiles = p.num_tiles; out->kslabs = p.Cin / 16 + p.xslabs; out->stages = p.stages; out->tmem_cols = cols;
  out->smem_bytes = smem; out->weight_bytes = conv_weight_bytes(p.taps, p.Cin, p.Cextra, p.CoutPad);
  return 0;
}
extern "C" int dmd_prep_act(const dmd_prep_desc* d, void* stream) {
  PrepParams p; int nsrc;
  if (prep_fill(d, &p, &nsrc)) return 1;
  return prep_launch(p, nsrc, (cudaStream_t)stream);
}

static int conv_launch_trs(const ConvParams& p0, size_t smem, int tmem_cols, cudaStream_t st) {
  if (init_kernels()) return 1;
  const int grid = p0.num_tiles < g_num_sms ? p0.num_tiles : g_num_sms;
  ConvParams p = p0;
  p.ktrace = kt_slot("conv3x3rs", p.num_tiles, (p.Cin + p.Cextra) * 1000 + p.W);
  switch (tmem_cols) {
    case 64: return launch_pdl(conv_tc_kernel<64, 3>, dim3(grid), dim3(kConvThreads), smem, st, p);
    case 128: return launch_pdl(conv_tc_kernel<128, 3>, dim3(grid), dim3(kConvThreads), smem, st, p);
    default: return launch_pdl(conv_tc_kernel<256, 3>, dim3(grid), dim3(kConvThreads), smem, st, p);
  }
}

static int conv_launch(const ConvParams& p, size_t smem, int tmem_cols, cudaStream_t st) {
  if (p.trs) return conv_launch_trs(p, smem, tmem_cols, st);
  switch (tmem_cols) {
    case 32: return conv_launch_t<32>(p, smem, st);
    case 64: return conv_launch_t<64>(p, smem, st);
    default: return conv_launch_t<128>(p, smem, st);
  }
}

static int fused_launch(const FusedParams& f0, size_t smem, int tmem_cols, cudaStream_t st) {
  if (init_kernels()) return 1;
  FusedParams f = f0;
  f.c.ktrace = kt_slot(f.c.taps == 9 ? "fused3x3" : "fused1x1", f.c.num_tiles, (f.c.Cin + f.c.Cextra) * 1000 + f.c.W);
  const dim3 grid(f.c.num_tiles), block(kConvThreads);
  switch (tmem_cols) {
    case 32: return launch_pdl(conv_fused_kernel<32>, grid, block, smem, st, f);
    case 64: return launch_pdl(conv_fused_kernel<64>, grid, block, smem, st, f);
    default: return launch_pdl(conv_fused_kernel<128>, grid, block, smem, st, f);
  }
}

extern "C" int dmd_conv2d_fprop(const dmd_conv_desc* d, void* stream) {
  ConvParams p; size_t smem; int cols;
  if (conv_fill(d, &p, &smem, &cols)) return 1;
  return conv_launch(p, smem, cols, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------- wgrad launcher
// Fills the tcgen05 weight-gradient launch for one (gradient operand, activation operand) pair.  grad: PLC16, Cg stored
// channels (<= 64); act: PLC16, Ca stored channels (16 / 32 / 64), both over B images of H x W (conv INPUT size; a
// stride-2 conv passes its zero-inserted gradient).
struct WgradLaunch { WgradParams wp; WgradReduceParams rp; size_t smem; int grid; };
static size_t wgrad_partial_bytes(int num_sms) { return (size_t)num_sms * kWgMaxMma * kTileM * 64 * sizeof(float); }

static int wgrad_fill(const void* grad, int Cg, const void* act, int Ca, int B, int H, int W, int taps, float* partial,
                      int Cout, int Cin, int CinTot, int ci_off, const float* inv_scale, int accumulate, int debug, WgradLaunch* L) {
  DMD_CHECK(grad && act && partial, "wgrad: null operand / partial buffer");
  DMD_CHECK(taps == 9 || taps == 1, "wgrad: taps must be 1 or 9");
  DMD_CHECK(Cg % 8 == 0 && Cg > 0 && Cg <= 64, "wgrad: gradient operand channels must be a multiple of 8, <= 64 (got %d)", Cg);
  DMD_CHECK(Ca == 16 || Ca == 32 || Ca == 64, "wgrad: activation operand channels must be 16, 32 or 64 (got %d)", Ca);
  DMD_CHECK(Cout > 0 && Cout <= Cg && Cin > 0 && Cin <= Ca && ci_off >= 0 && ci_off + Cin <= CinTot, "wgrad: bad channel counts");
  if (init_kernels()) return 1;
  memset(L, 0, sizeof(*L));
  const Plc g = plc_geometry(B, H, W);
  const size_t plane = (size_t)g.Qalloc * 16;
  WgradParams& wp = L->wp;
  const int ng = Cg / 8;
  for (int k = 0; k < 16; ++k) {
    const int j = k & 7;
    const bool second = k >= 8;
    wp.a_plane[k] = (j < ng && !(second && taps == 1)) ? (const uint8_t*)grad + (size_t)j * plane : nullptr;
    wp.a_shift[k] = second ? -g.PW : 0;
  }
  wp.zeros = g_zeros;
  wp.nB = Ca / 8;
  for (int j = 0; j < wp.nB; ++j) wp.b_plane[j] = (const uint8_t*)act + (size_t)j * plane;
  WgradReduceParams& rp = L->rp;
  for (int i = 0; i < kWgMaxMma; ++i) rp.tap_of[i][0] = rp.tap_of[i][1] = -1;
  if (taps == 9) {
    wp.n_mma = 6; wp.halo = g.PW + 1;
    for (int i = 0; i < 3; ++i) {
      wp.b_shift[i] = -g.PW - 1 + i;      // rows 0-63: tap (ky = 0, kx = i); rows 64-127 (window shifted by -PW): tap (1, i)
      rp.tap_of[i][0] = i; rp.tap_of[i][1] = 3 + i;
      wp.b_shift[3 + i] = g.PW - 1 + i;   // rows 0-63: tap (2, i); rows 64-127 unused
      rp.tap_of[3 + i][0] = 6 + i;
    }
  } else {
    wp.n_mma = 1; wp.halo = 0; wp.b_shift[0] = 0; rp.tap_of[0][0] = 0;
  }
  wp.G = g.G; wp.num_tiles = (g.Q + kTileM - 1) / kTileM; wp.Pb = kTileM + 2 * wp.halo;
  const WgradSmem one = wgrad_smem(wp.nB, wp.halo, 1);
  int stages = (int)((227ll * 1024 - 512) / (long long)(one.a_bytes + one.b_bytes));
  if (stages > kWgStagesMax) stages = kWgStagesMax;
  DMD_CHECK(stages >= 2, "wgrad: image too wide for the shared-memory stage (W=%d)", W);
  wp.stages = stages;
  wp.partial = partial; wp.dbg = debug;
  L->smem = wgrad_smem(wp.nB, wp.halo, stages).total;
  L->grid = wp.num_tiles < g_num_sms ? wp.num_tiles : g_num_sms;
  rp.partial = partial; rp.nparts = L->grid; rp.n_mma = wp.n_mma; rp.N = Ca;
  rp.Cout = Cout; rp.Cin = Cin; rp.CinTot = CinTot; rp.ci_off = ci_off; rp.taps = taps;
  rp.inv_scale = inv_scale; rp.accumulate = accumulate;
  return 0;
}
static int wgrad_launch(const WgradLaunch& L, float* dW, cudaStream_t st) {
  if (launch_pdl(wgrad_tc_kernel, dim3(L.grid), dim3(kWgThreads), L.smem, st, L.wp)) return 1;
  WgradReduceParams rp = L.rp;
  rp.dW = dW;
  const int total = rp.n_mma * 2 * 64 * rp.N;
  wgrad_reduce_kernel<<<(total + 63) / 64, 256, 0, st>>>(rp);
  DMD_LAUNCH_OK();
  return 0;
}

extern "C" size_t dmd_wgrad_partial_bytes(void) {
  if (init_kernels()) return 0;
  return wgrad_partial_bytes(g_num_sms);
}
extern "C" int dmd_conv2d_wgrad(const dmd_wgrad_desc* d, void* stream) {
  DMD_CHECK(d && d->dW, "wgrad: null descriptor / dW");
  if (init_kernels()) return 1;
  DMD_CHECK(d->partial_bytes >= wgrad_partial_bytes(g_num_sms), "wgrad: partial buffer too small (%zu < %zu)", d->partial_bytes, wgrad_partial_bytes(g_num_sms));
  WgradLaunch L;
  if (wgrad_fill(d->grad, d->Cg, d->act, d->Ca, d->B, d->H, d->W, d->taps, (float*)d->partial, d->Cout, d->Cin, d->CinTot, d->ci_off,
                 d->inv_scale, d->accumulate, d->debug, &L)) return 1;
  return wgrad_launch(L, d->dW, (cudaStream_t)stream);
}
extern "C" int dmd_pack_conv_weight_dgrad(const float* w, void* wpk, int CoutF, int CinTotF, int ci_off, int CinK, int taps, void* stream) {
  DMD_CHECK(w && wpk, "pack_T: null pointer");
  const int CinP = round_up(CoutF, 16), CoutP = round_up(CinK, 16);
  const int total = taps * CinP * CoutP;
  pack_conv_weight_T_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, (__half*)wpk, CoutF, CinTotF, ci_off, CinK, CinP, CoutP, taps);
  DMD_LAUNCH_OK();
  return 0;
}

extern "C" int dmd_pack_conv_weight(const float* w, void* wpk, int Cout, int CoutPad, int CinReal, int Cin, int taps,
                                    int c0_real, int c0_store, int precise, void* stream) {
  DMD_CHECK(w && wpk, "pack: null pointer");
  if (precise == 3) {   // tap-row-stacked layout [dy][Cin/8][3 * CoutPad][8]: column dx * CoutPad + co of kernel row dy
    DMD_CHECK(taps == 9, "pack: the row-stacked layout is for 3x3 kernels");
    const int total3 = 9 * Cin * CoutPad;
    pack_conv_weight_trs_kernel<<<(total3 + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, (__half*)wpk, Cout, CoutPad, CinReal, Cin, c0_real, c0_store);
    DMD_LAUNCH_OK();
    return 0;
  }
  DMD_CHECK(precise >= 0 && precise <= 2, "pack: precise must be 0, 1 (split [W_hi | W_hi | W_lo]), 2 (low parts only) or 3 (row-stacked)");
  const int total = taps * Cin * CoutPad * (precise == 1 ? 3 : 1);
  pack_conv_weight_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, (__half*)wpk, Cout, CoutPad, CinReal, Cin, taps, c0_real, c0_store, precise);
  DMD_LAUNCH_OK();
  return 0;
}

extern "C" int dmd_gn_stats(const float* x, double* stats, int B, int HW, int C, int gs, void* stream) {
  DMD_CHECK(x && stats && gs > 0 && C % gs == 0, "gn_stats: bad arguments");
  long long per = (long long)HW * C;
  int chunks = (int)((per + 256 * 64 - 1) / (256 * 64));
  if (chunks < 1) chunks = 1;
  if (chunks > 64) chunks = 64;
  gn_stats_kernel<<<dim3(chunks, B), 256, 0, (cudaStream_t)stream>>>(x, stats, HW, C, gs);
  DMD_LAUNCH_OK();
  return 0;
}

static int attn_launch(const AttnParams& p, int B, cudaStream_t st) {
  DMD_CHECK((p.C == 64 || p.C == 32) && p.L == kAttnL && p.C % p.gs == 0 && p.gs % 8 == 0,
            "attn: unsupported shape L=%d C=%d gs=%d (built for 8x8 = 64 tokens, C in {32, 64})", p.L, p.C, p.gs);
  if (init_kernels()) return 1;
  const size_t smem = sizeof(float) * ((size_t)p.L * (p.C + 1) * 2 + (size_t)p.L * (3 * p.C + 4));
  AttnParams pt = p;
  pt.ktrace = kt_slot("attn", B, p.C);
  if (tune_int("DMD_ATTN_CLUSTER", 1) != 0 && p.gs % (p.C / 4) == 0) {
    // four CTAs per image (thread-block cluster), distributed shared memory for the head outputs
    const int CH = p.C / 4;
    const size_t csmem = sizeof(float) * ((size_t)p.L * (p.C + 1) * 2 + (size_t)p.L * (3 * CH + 4) + (size_t)p.L * CH + (size_t)4 * CH * p.C);
    if (p.C == 64) attn_cluster_kernel<64><<<4 * B, kAttnCThreads, csmem, st>>>(pt);
    else attn_cluster_kernel<32><<<4 * B, kAttnCThreads, csmem, st>>>(pt);
    DMD_LAUNCH_OK();
    return 0;
  }
  if (p.C == 64) attn_kernel<64><<<B, kAttnThreads, smem, st>>>(pt);
  else attn_kernel<32><<<B, kAttnThreads, smem, st>>>(pt);
  DMD_LAUNCH_OK();
  return 0;
}

static int linear_launch(const float* in, const float* W, const float* bias, float* out, int B, int K, int F, int silu, cudaStream_t st,
                         int accumulate = 0, int hw_perm = 0) {
  DMD_CHECK(K % 4 == 0, "linear: K=%d must be a multiple of 4", K);
  DMD_CHECK(hw_perm == 0 || K % hw_perm == 0, "linear: bad hw_perm");
  if (init_kernels()) return 1;
  // enough blocks to cover the SMs: 8, 16 or 32 output features per block
  const int by = (B + 31) / 32;
  const int forceJ = tune_int("DMD_LINEAR_J", 0);
  if (forceJ == 4 || (forceJ == 0 && (long long)((F + 31) / 32) * by >= 296))
    linear_kernel<4><<<dim3((F + 31) / 32, by), 256, (size_t)(32 + 32) * kLinChunk * sizeof(float), st>>>(in, W, bias, out, B, K, F, silu, accumulate, hw_perm);
  else if (forceJ == 2 || (forceJ == 0 && (long long)((F + 15) / 16) * by >= 148))
    linear_kernel<2><<<dim3((F + 15) / 16, by), 256, (size_t)(16 + 32) * kLinChunk * sizeof(float), st>>>(in, W, bias, out, B, K, F, silu, accumulate, hw_perm);
  else
    linear_kernel<1><<<dim3((F + 7) / 8, by), 256, (size_t)(8 + 32) * kLinChunk * sizeof(float), st>>>(in, W, bias, out, B, K, F, silu, accumulate, hw_perm);
  DMD_LAUNCH_OK();
  return 0;
}

extern "C" int dmd_attn_fwd(const float* x, const double* stats_in, const float* gamma, const float* beta,
                            const float* wqkv, const float* bqkv, const float* wout, const float* bout, float* out,
                            double* out_stats, int B, int L, int C, int gs, float eps, void* stream) {
  AttnParams p{x, stats_in, gamma, beta, wqkv, bqkv, wout, bout, out, out_stats, L, C, gs, eps};
  return attn_launch(p, B, (cudaStream_t)stream);
}

extern "C" int dmd_nchw_to_nhwc(const float* in, float* out, int B, int C, int CP, int HW, void* stream) {
  nchw_to_nhwc_kernel<<<dim3((HW + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(in, out, C, CP, HW);
  DMD_LAUNCH_OK();
  return 0;
}
extern "C" int dmd_nhwc_to_nchw(const float* in, float* out, int B, int C, int CP, int HW, void* stream) {
  nhwc_to_nchw_kernel<<<dim3((HW + 255) / 256, B), 256, 0, (cudaStream_t)stream>>>(in, out, C, CP, HW);
  DMD_LAUNCH_OK();
  return 0;
}

// ---------------------------------------------------------------------------------------------- denoiser executor
// zero-pad / crop copy of an NHWC tensor, then the GroupNorm partial sums of the result (the consumer's prologue reads them)
static int resize_launch(const ResizeParams& p, cudaStream_t st) {
  const long long total = (long long)p.B * p.Hd * p.Wd * (p.C / 4);
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  resize_nhwc_kernel<<<(int)blocks, 256, 0, st>>>(p);
  DMD_LAUNCH_OK();
  if (p.stats) return dmd_gn_stats(p.dst, p.stats, p.B, p.Hd * p.Wd, p.C, p.gs, st);
  return 0;
}

namespace {

constexpr float kGnEps = 1e-5f;  // blocks.py:13

struct ConvW {          // one nn.Conv2d
  int w_idx, b_idx;     // indices into the state_dict pointer list
  int Cout, CoutPad, CinReal, Cin, taps, c0_real, c0_store;
  int precise = 0;      // split-fp16: K = 3 * Cin
  int trs = 0;          // forward weights in the tap-row-stacked layout (3x3, non-split)
  int three_pass = 0;   // split-fp16 as three launches (A_hi W_hi, A_lo W_hi, A_hi W_lo) when 3 * Cin weights exceed shared memory
  size_t pk_off;        // byte offset into the packed-weight buffer
  size_t pk_lo_off = 0; // three_pass: the low-part pack
  // backward-data packs (transposed, tap-flipped; one per source of a channel concat), training only
  int nsrcT = 0; int srcC[2] = {0, 0}; int srcOff[2] = {0, 0}; size_t pkT_off[2] = {0, 0};
};
struct FilmW { int w_idx, b_idx, C, off; };  // AdaGroupNorm.linear ; off = row offset into the batched FiLM GEMM
struct ResBlockW {
  int cin, cout;
  int has_proj; ConvW proj;
  FilmW n1, n2; ConvW c1, c2;
  int has_attn; int an_w, an_b, qkv_w, qkv_b, op_w, op_b;
};

struct Tens { float* data; double* stats; int C, H, W, gs; float* grad = nullptr; int gid = -1; };

enum OpKind { OP_CONV = 0, OP_ATTN = 1, OP_PREP = 2, OP_FUSED = 3, OP_RESIZE = 4 };
struct Op { int kind; ConvParams conv; size_t smem; int cols; AttnParams attn; PrepParams prep; int prep_nsrc; FusedParams fused; ResizeParams rs; };
constexpr int kScratchSlots = 10;  // round-robin pool of PLC16 operand buffers (each lives from its prep to the next conv)

// PLC16 operands produced by one prep launch (op = index of that launch in Plan::ops, replayed by the backward pass)
struct Operand {
  uint8_t *n0 = nullptr, *n1 = nullptr, *r0 = nullptr, *r1 = nullptr, *nl0 = nullptr, *rl0 = nullptr, *rl1 = nullptr; int C0 = 0, C1 = 0, H = 0, W = 0, op = -1;
  // description of the transform (always filled).  lazy: no prep launch has been emitted -- the consumer either runs the
  // transform inside its own kernel (conv_fused_kernel, small problems) or materialises the operand first
  bool lazy = false;
  Tens a{}, b{}; bool has_b = false;
  int upsample = 0, mode = 0; const FilmW* film = nullptr; int gamma_idx = 0, beta_idx = 0; bool silu = false, also_raw = false, split = false;
  bool split_main = false;   // the low part of the main operand as well as of the raw one (a split-fp16 conv reads it)
};

// backward op list (training).  Parameter-gradient destinations are OFFSETS into the caller's flat gradient buffer.
enum BKind { B_PREP = 0, B_CONV, B_WGRAD, B_COLSUM, B_NORM1, B_NORM2, B_AFFINE, B_POOL, B_ADD, B_ATTN, B_MEMSET, B_SGEMM, B_FILMW,
             B_LINEAR, B_DSILU, B_EMB };
struct BOp {
  int kind = 0;
  PrepParams prep; int prep_nsrc = 1;
  ConvParams conv; size_t smem = 0; int cols = 0;
  WgradLaunch wg;
  long long goff = -1, goff2 = -1;            // flat-gradient offsets (floats)
  NormBwdParams nb; int ppb = 0, chunks = 0;
  const float* src = nullptr; float* dst = nullptr; long long rows = 0; int C = 0, Creal = 0, H = 0, W = 0, acc = 0; long long total4 = 0;
  AttnBwdParams ab; long long goffs[6] = {-1, -1, -1, -1, -1, -1};
  void* ms_ptr = nullptr; size_t ms_bytes = 0;
  // sgemm: C = alpha * op(A) op(B); c_goff >= 0 -> C lives in the gradient buffer
  const float *ga = nullptr, *gb = nullptr; float* gc = nullptr; long long sam = 0, sak = 0, sbk = 0, sbn = 0, ldc = 0, c_goff = -1;
  int M = 0, N = 0, K = 0, use_inv = 0;
  // linear recompute
  const float *lin_in = nullptr, *lin_w = nullptr, *lin_b = nullptr; float* lin_out = nullptr; int lin_K = 0, lin_F = 0;
};

enum RecKind { R_CONVIN = 0, R_DOWN, R_UP, R_RES, R_OUT };
struct Rec {
  int kind = 0;
  const ConvW* cw = nullptr; const ResBlockW* rb = nullptr;
  Tens x, skip, t, o, a; bool has_skip = false;
  Operand in1, in2;
};

// The RewEnd encoder (rew_end_model.py:93-132): U-Net blocks driven by PlanBuilder::build_rew_end.  A training plan built with
// one of these records the encoder's tape instead of the InnerModel's, and its backward ends in the action-embedding gradient.
struct EncoderDef {
  const std::vector<std::vector<ResBlockW>>* blocks; const std::vector<ConvW>* downs; const ConvW* conv_in; int i_actemb;
};

struct Plan {
  int B = 0, H = 0, W = 0;
  uint8_t* base = nullptr;
  size_t bytes = 0;
  float *xin = nullptr, *cs = nullptr, *cemb = nullptr, *chid = nullptr, *cond = nullptr, *film = nullptr, *fout = nullptr;
  double* stats = nullptr; size_t stats_bytes = 0;
  int CP_in = 0, CF = 0;
  std::vector<Op> ops;
  uint8_t* scratch[kScratchSlots] = {nullptr};
  int scratch_next = 0;
  // training (dmd_inner_model_forward_train / dmd_denoiser_backward): gradient buffers and the backward op list
  bool train = false;
  int n_grad_tensors = 0;
  std::vector<BOp> bops;
  std::vector<Rec> tape;
  const int64_t* t_act = nullptr;                         // the forward's action tensor (embedding gradient)
  float *tA = nullptr, *tB = nullptr, *tC = nullptr;      // fp32 NHWC temporaries (largest activation)
  uint8_t *gyA = nullptr, *gyB = nullptr;                 // PLC16 gradient operands
  float *gF = nullptr;                                    // scaled dL/d(model output), NHWC with 8 channels
  float *dfilm = nullptr, *nsum = nullptr, *partial = nullptr, *scale = nullptr;
  float *dcond = nullptr, *dh = nullptr, *cpre = nullptr, *dpre = nullptr, *de = nullptr;
  unsigned int* amax = nullptr;
  long long *film_woff = nullptr, *film_boff = nullptr;   // device tables: flat-gradient offset of every FiLM row
  std::vector<long long> film_woff_h, film_boff_h;
  uint8_t* zero_begin = nullptr; size_t zero_bytes = 0;   // region cleared at the start of every backward (dfilm, sums, amax)
  Tens enc_out{};                                         // RewEnd encoder output (its .grad receives the LSTM's input gradient)
  int seq_b = 0, seq_t = 0;                               // RewEnd: (b, t) of the last training forward on this workspace
  // sampler state (NCHW fp32): temporaries only -- the frame stack, the actions and the trajectory are used IN PLACE
  float *s_xc = nullptr, *s_x2 = nullptr, *s_d = nullptr;
  float *sig_all = nullptr, *cemb_all = nullptr, *chid_all = nullptr, *cond_all = nullptr, *film_all = nullptr;  // hoisted conditioning
};

constexpr int kMaxSamplerEvals = 24;   // U-Net evaluations per sample() whose conditioning is hoisted (12 Heun / 24 Euler steps)
struct SamplerGraph {
  bool valid = false;
  int B = 0, H = 0, W = 0; void* ws = nullptr; int order = 0; bool has_eps = false;
  const void *obs = nullptr, *act = nullptr, *traj = nullptr, *eps = nullptr, *out = nullptr; StackView sv{};   // graphs bake pointers in
  unsigned long long stamp = 0;
  std::vector<float> sigmas; float churn[4] = {0, 0, 0, 0};
  long long kernels = 0;  // kernel nodes per replay
  cudaGraphExec_t exec = nullptr;
};

}  // namespace

struct dmd_denoiser {
  dmd_denoiser_config cfg;
  int n_tensors = 0;
  // state_dict indices
  int i_fourier = 0, i_actemb = 0, i_cp0w = 0, i_cp0b = 0, i_cp2w = 0, i_cp2b = 0, i_normout_w = 0, i_normout_b = 0;
  ConvW conv_in, conv_out;
  std::vector<std::vector<ResBlockW>> d_blocks, u_blocks;
  std::vector<ResBlockW> mid;
  std::vector<ConvW> downs, ups;  // index 0 unused (Identity)
  int film_rows = 0;
  size_t packed_bytes = 0, film_w_off = 0, film_b_off = 0;
  std::vector<const float*> ptrs;
  uint8_t* packed = nullptr;
  std::vector<long long> numel, goff;   // per state_dict tensor: element count and offset into the flat gradient buffer
  long long grad_total = 0;
  Plan plan;
  std::vector<SamplerGraph> graphs;     // one per distinct (buffers, ring head): a WorldModelEnv replays T of them round-robin
  unsigned long long graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  // training plans, one per live training workspace (an autoregressive Denoiser.forward holds several forwards before
  // their backwards run); kept apart from `plan` so that imagination and training can alternate
  std::vector<std::unique_ptr<Plan>> tplans;
  int need_B = 0, need_H = 0, need_W = 0; size_t need_bytes = 0;
};

namespace {

struct Walker {  // assigns state_dict indices in module registration order and packed-buffer offsets
  dmd_denoiser* h; int idx = 0; size_t pk = 0;
  int next(long long n) { h->numel.push_back(n); return idx++; }
  ConvW conv(int cout, int cin_real, int taps, int c0_real, int c0_store, int c1, int precise = 0, bool dgrad = true) {
    ConvW c; c.w_idx = next((long long)cout * cin_real * taps); c.b_idx = next(cout);
    c.Cout = cout; c.CoutPad = round_up(cout, 16); c.CinReal = cin_real; c.taps = taps;
    c.c0_real = c0_real; c.c0_store = c0_store; c.Cin = round_up(c0_store + c1, 16); c.precise = precise;
    // tap-row-stacked layout: opt-in (DMD_CONV_TRS=1).  Correct (tests/test_gpu_conv.py runs it), but measured slower on the B200:
    // 25 us vs 20 us for the 64->64 conv at 64x64 -- see DESIGN.md section 4
    c.trs = (taps == 9 && !precise && 3 * c.CoutPad <= 256 && tune_int("DMD_CONV_TRS", 0) != 0) ? 1 : 0;
    c.pk_off = pk; pk += (size_t)taps * c.Cin * c.CoutPad * 2 * (precise ? 3 : 1); pk = (pk + 255) & ~(size_t)255;
    if (dgrad) {
      c.nsrcT = c1 ? 2 : 1;
      c.srcC[0] = c0_real; c.srcC[1] = c1; c.srcOff[0] = 0; c.srcOff[1] = c0_real;
      for (int k = 0; k < c.nsrcT; ++k) {
        c.pkT_off[k] = pk;
        pk += (size_t)taps * round_up(cout, 16) * round_up(c.srcC[k], 16) * 2; pk = (pk + 255) & ~(size_t)255;
      }
    }
    return c;
  }
  FilmW film(int C) {
    FilmW f; f.w_idx = next((long long)2 * C * h->cfg.cond_channels); f.b_idx = next(2 * C);
    f.C = C; f.off = h->film_rows; h->film_rows += 2 * C; return f;
  }
  // c0/c1: channels of the two concatenated inputs (c1 = 0: single input)
  ResBlockW resblock(int c0, int c1, int cout, bool attn) {
    ResBlockW r; r.cin = c0 + c1; r.cout = cout;
    r.has_proj = (r.cin != cout);
    if (r.has_proj) r.proj = conv(cout, r.cin, 1, c0, c0, c1, 1);  // raw residual stream -> split-fp16
    r.n1 = film(r.cin);
    r.c1 = conv(cout, r.cin, 9, c0, c0, c1);
    r.n2 = film(cout);
    r.c2 = conv(cout, cout, 9, cout, cout, 0);
    r.has_attn = attn;
    if (attn) {
      r.an_w = next(cout); r.an_b = next(cout); r.qkv_w = next((long long)3 * cout * cout); r.qkv_b = next(3 * cout);
      r.op_w = next((long long)cout * cout); r.op_b = next(cout);
    }
    return r;
  }
};

int build_structure(dmd_denoiser* h) {
  const dmd_denoiser_config& c = h->cfg;
  const int L = c.num_levels;
  Walker w{h};
  // InnerModel.__init__ registration order (inner_model.py:24-42): noise_emb, act_emb, cond_proj, conv_in, unet,
  // norm_out, conv_out.  UNet (blocks.py:183-220): d_blocks, u_blocks, mid_blocks, downsamples, upsamples.
  const long long CC = c.cond_channels;
  h->numel.clear();
  h->i_fourier = w.next(CC / 2); h->i_actemb = w.next((long long)c.num_actions * (CC / c.num_steps_conditioning));
  h->i_cp0w = w.next(CC * CC); h->i_cp0b = w.next(CC); h->i_cp2w = w.next(CC * CC); h->i_cp2b = w.next(CC);
  const int cin_real = (c.num_steps_conditioning + 1) * c.img_channels;
  const int cin_store = round_up(cin_real, 16);
  h->conv_in = w.conv(c.channels[0], cin_real, 9, cin_real, cin_store, 0, 1, false);  // its input needs no gradient
  h->d_blocks.resize(L);
  for (int i = 0; i < L; ++i) {
    const int c1 = c.channels[i > 0 ? i - 1 : 0], c2 = c.channels[i];
    for (int k = 0; k < c.depths[i]; ++k) h->d_blocks[i].push_back(w.resblock(k == 0 ? c1 : c2, 0, c2, c.attn_depths[i] != 0));
  }
  // u_blocks were built per level i then reversed (blocks.py:199-207,209): module order = level L-1 ... 0
  h->u_blocks.resize(L);
  for (int m = 0; m < L; ++m) {
    const int i = L - 1 - m;
    const int c1 = c.channels[i > 0 ? i - 1 : 0], c2 = c.channels[i];
    const int n = c.depths[i];
    // list_in_channels = [2*c2]*n + [c1+c2] ; list_out = [c2]*n + [c1]; the concat is (x, skip) with x first.
    // x has c2 channels for every block (block n's x is the previous block's output, c2); skips carry c2 except the
    // last one (the level's x_down, c1 channels).
    for (int k = 0; k <= n; ++k) h->u_blocks[m].push_back(w.resblock(c2, k < n ? c2 : c1, k < n ? c2 : c1, c.attn_depths[i] != 0));
  }
  for (int k = 0; k < 2; ++k) h->mid.push_back(w.resblock(c.channels[L - 1], 0, c.channels[L - 1], true));
  h->downs.resize(L); h->ups.resize(L);
  for (int i = 1; i < L; ++i) h->downs[i] = w.conv(c.channels[i - 1], c.channels[i - 1], 9, c.channels[i - 1], c.channels[i - 1], 0);
  for (int m = 1; m < L; ++m) { const int ch = c.channels[L - 1 - m]; h->ups[m] = w.conv(ch, ch, 9, ch, ch, 0); }
  h->i_normout_w = w.next(c.channels[0]); h->i_normout_b = w.next(c.channels[0]);
  h->conv_out = w.conv(c.img_channels, c.channels[0], 9, c.channels[0], c.channels[0], 0, 0);  // split-fp16 here costs 3x on an N=16 conv for 3.2e-4
  h->n_tensors = w.idx;
  h->goff.assign(h->n_tensors, 0);
  h->grad_total = 0;
  for (int i = 0; i < h->n_tensors; ++i) { h->goff[i] = h->grad_total; h->grad_total += (h->numel[i] + 3) & ~3ll; }  // 16-byte aligned slices
  size_t pk = w.pk;
  h->film_w_off = pk; pk += (size_t)h->film_rows * c.cond_channels * 4; pk = (pk + 255) & ~(size_t)255;
  h->film_b_off = pk; pk += (size_t)h->film_rows * 4; pk = (pk + 255) & ~(size_t)255;
  h->packed_bytes = pk;
  return 0;
}

struct Bump {
  uint8_t* base; size_t off = 0;
  void* take(size_t bytes) { off = (off + 255) & ~(size_t)255; void* p = base ? base + off : nullptr; off += bytes; return p; }
};

// -- plan construction: mirrors InnerModel.forward / UNet.forward / ResBlock.forward
struct PlanBuilder {
  dmd_denoiser* h; Plan* pl; Bump* bump; Bump* sbump; int err = 0;

  Tens tensor(int C, int H, int W, bool with_stats, bool with_grad = true) {
    Tens t; t.C = C; t.H = H; t.W = W; t.gs = gn_group_size(C);
    t.data = (float*)bump->take((size_t)pl->B * H * W * C * 4);
    t.stats = with_stats ? (double*)sbump->take((size_t)pl->B * (C / t.gs) * 2 * 8) : nullptr;
    if (pl->train && with_grad) { t.grad = (float*)bump->take((size_t)pl->B * H * W * C * 4); t.gid = pl->n_grad_tensors++; }
    return t;
  }
  void record(const Rec& r) { if (pl->train) pl->tape.push_back(r); }
  const float* P(int idx) const { return h->ptrs.empty() ? nullptr : h->ptrs[idx]; }

  uint8_t* scratch() {
    uint8_t* p = pl->scratch[pl->scratch_next];
    pl->scratch_next = (pl->scratch_next + 1) % kScratchSlots;
    return p ? p : (uint8_t*)1;
  }

  // mode 0 raw / 1 AdaGroupNorm(film) / 2 GroupNorm(gamma,beta); also_raw: additionally emit the raw operand (skip projection)
  // split: also emit the low fp16 part of the operand that a precise conv will read (raw if also_raw, else the main one)
  Operand prep(const Tens& a, const Tens* b, int upsample, int mode, const FilmW* film, int gamma_idx, int beta_idx, bool silu, bool also_raw,
               bool split = false, bool split_main = false) {
    Operand o;
    o.a = a; o.has_b = b != nullptr; if (b) o.b = *b;
    o.upsample = upsample; o.mode = mode; o.film = film; o.gamma_idx = gamma_idx; o.beta_idx = beta_idx; o.silu = silu; o.also_raw = also_raw; o.split = split;
    o.split_main = split_main;
    o.C0 = round_up(a.C, 16); o.C1 = b ? round_up(b->C, 16) : 0;
    o.H = upsample ? 2 * a.H : a.H; o.W = upsample ? 2 * a.W : a.W;
    // small problems (at most one tile per SM) may leave the transform to the consuming conv (conv_fused_kernel, DMD_FUSE_SMALL=1;
    // measured in the CUDA graph at B=32: one 8.7 us launch instead of 4.0 + 4.6 us -- no gain yet, so it is opt-in); never in
    // training plans, whose backward replays the prep launches
    const Plc g = plc_geometry(pl->B, o.H, o.W);
    const int tiles = (g.Q + kTileM - 1) / kTileM;
    o.lazy = !pl->train && g_num_sms > 0 && tiles <= g_num_sms && tune_int("DMD_FUSE_SMALL", 0) != 0 && upsample != 2 &&
             a.C % 16 == 0 && (!b || b->C % 16 == 0);
    if (!o.lazy) materialize(o);
    return o;
  }
  void materialize(Operand& o) {
    if (!o.lazy && o.n0) return;
    o.lazy = false;
    const Tens& a = o.a; const Tens* b = o.has_b ? &o.b : nullptr;
    dmd_prep_desc d; memset(&d, 0, sizeof(d));
    d.src0 = a.data ? a.data : (const float*)1; d.C0 = a.C; d.src1 = b ? (b->data ? b->data : (const float*)1) : nullptr; d.C1 = b ? b->C : 0;
    d.B = pl->B; d.Hs = a.H; d.Ws = a.W; d.upsample = o.upsample; d.mode = o.mode; d.silu = o.silu;
    if (o.mode) {
      d.stats0 = a.stats ? a.stats : (const double*)1; d.gs0 = a.gs;
      if (b) { d.stats1 = b->stats ? b->stats : (const double*)1; d.gs1 = b->gs; }
    }
    if (o.mode == 1) { d.film = pl->film ? pl->film : (const float*)1; d.film_stride = h->film_rows; d.film_off = o.film->off; }
    if (o.mode == 2) { d.gamma = P(o.gamma_idx) ? P(o.gamma_idx) : (const float*)1; d.beta = P(o.beta_idx) ? P(o.beta_idx) : (const float*)1; }
    d.eps = kGnEps;
    o.n0 = scratch(); d.dst0 = o.n0;
    if (b) { o.n1 = scratch(); d.dst1 = o.n1; }
    if (o.also_raw) { o.r0 = scratch(); d.dst_raw0 = o.r0; if (b) { o.r1 = scratch(); d.dst_raw1 = o.r1; } }
    if (o.split && o.also_raw) { o.rl0 = scratch(); d.dst_raw_lo0 = o.rl0; if (b) { o.rl1 = scratch(); d.dst_raw_lo1 = o.rl1; } }
    if ((o.split && !o.also_raw) || o.split_main) { o.nl0 = scratch(); d.dst_lo0 = o.nl0; }
    Op op; op.kind = OP_PREP;
    if (prep_fill(&d, &op.prep, &op.prep_nsrc)) { err = 1; return; }
    o.op = (int)pl->ops.size();
    pl->ops.push_back(op);
  }

  // the conv with its input transform inside the kernel (conv_fused.cuh); false: not applicable (the caller materialises)
  bool try_fused(const ConvW& cw, Operand& in, int stride, const Tens* resid, Tens& out, bool out_stats, const ConvW* xproj, Operand* xin) {
    if (!in.lazy || cw.precise || cw.trs || (xproj && !(xin && xin->lazy))) return false;   // (the fused kernel reads tap-major weights)
    if (in.mode != 0 && (in.a.C / in.a.gs > 4 || (in.has_b && in.b.C / in.b.gs > 4))) return false;   // coefficient table: 4 groups per source
    Op op; op.kind = OP_FUSED;
    FusedParams& f = op.fused; memset(&f, 0, sizeof(f));
    ConvParams& c = f.c;
    const int Cmain = in.C0 + in.C1, Cx = xproj ? xin->C0 + xin->C1 : 0;
    if (Cmain != cw.Cin || Cmain > kMaxCin || Cx > kMaxCin) return false;
    c.Cin = Cmain; c.Cextra = 3 * Cx;
    c.B = pl->B; c.H = in.H; c.W = in.W; c.taps = cw.taps; c.stride = stride;
    if (stride == 2 && (c.H % 2 || c.W % 2)) return false;
    c.wpk = reinterpret_cast<const __half*>(h->packed ? h->packed + cw.pk_off : (const uint8_t*)1); c.bias = P(cw.b_idx);
    c.Cout = cw.Cout; c.CoutPad = cw.CoutPad;
    if (xproj) { c.wpk_extra = reinterpret_cast<const __half*>(h->packed ? h->packed + xproj->pk_off : (const uint8_t*)1); c.bias_extra = P(xproj->b_idx); }
    c.resid = resid ? (resid->data ? resid->data : (const float*)1) : nullptr; c.out = out.data ? out.data : (float*)1;
    c.ostats = out_stats ? (out.stats ? out.stats : (double*)1) : nullptr; c.ogs = out.gs > 0 ? out.gs : cw.Cout;
    if (out_stats && (cw.CoutPad > 64 || (cw.Cout != 16 && cw.Cout != 32 && cw.Cout != 64) || cw.Cout % c.ogs)) return false;
    const Plc g = plc_geometry(pl->B, in.H, in.W);
    c.PW = g.PW; c.PH = g.PH; c.Q = g.Q; c.G = g.G;
    const int halo = cw.taps == 9 ? g.PW + 1 : 0;
    c.P = kTileM + 2 * halo; c.Palloc = c.P | 1;
    c.dPW.init(g.PW); c.dPH.init(g.PH);
    c.num_tiles = (g.Q + kTileM - 1) / kTileM;
    if (out_stats && g.PH * g.PW < 64) return false;                              // epilogue: a tile touches at most 3 images
    if ((c.P - 1) / (g.PH * g.PW) + 2 > kFusedCoefSlots) return false;          // the halo window touches at most 4 images
    const uint32_t w_bytes = conv_weight_bytes(cw.taps, c.Cin, c.Cextra, c.CoutPad);
    const FusedSmem L = fused_smem_layout(w_bytes, Cmain, Cx, c.Palloc);
    if (L.total > 227u * 1024u) return false;
    f.coef_off = L.coef_off; f.a_off = L.a_off; f.xa_off = L.xa_off; f.w_off = L.w_off; f.slab_bytes = L.slab_bytes; f.xslab_bytes = L.xslab_bytes;
    f.Cmain = Cmain; f.Cx = Cx;
    auto src = [&](const Tens& t, int c_off, bool with_stats) {
      FusedSrc q; q.src = t.data ? t.data : (const float*)1; q.C = t.C; q.stats = with_stats ? (t.stats ? t.stats : (const double*)1) : nullptr;
      q.gs = t.gs > 0 ? t.gs : 8; q.c_offset = c_off; return q;
    };
    f.m[0] = src(in.a, 0, in.mode != 0); f.nm = 1;
    if (in.has_b) { f.m[1] = src(in.b, in.a.C, in.mode != 0); f.nm = 2; }
    f.mode = in.mode; f.act = in.silu ? 1 : 0; f.ups = in.upsample; f.Hs = in.a.H; f.Ws = in.a.W;
    if (in.mode == 1) { f.film = pl->film ? pl->film : (const float*)1; f.film_stride = h->film_rows; f.film_off = in.film->off; f.film_ctot = in.a.C + (in.has_b ? in.b.C : 0); }
    if (in.mode == 2) { f.gamma = P(in.gamma_idx) ? P(in.gamma_idx) : (const float*)1; f.beta = P(in.beta_idx) ? P(in.beta_idx) : (const float*)1; }
    f.eps = kGnEps;
    if (xproj) {
      if (xin->upsample || xin->H != in.H || xin->W != in.W) return false;
      f.x[0] = src(xin->a, 0, false); f.nx = 1;
      if (xin->has_b) { f.x[1] = src(xin->b, xin->a.C, false); f.nx = 2; }
    }
    op.smem = L.total;
    op.cols = cw.CoutPad <= 32 ? 32 : (cw.CoutPad <= 64 ? 64 : 128);
    pl->ops.push_back(op);
    return true;
  }

  void conv(const ConvW& cw, Operand& in, bool raw, int stride, const Tens* resid, Tens& out, bool out_stats,
            const ConvW* xproj = nullptr, Operand* xin = nullptr) {
    if (!raw && try_fused(cw, in, stride, resid, out, out_stats, xproj, xin)) return;
    materialize(in);
    if (xin) materialize(*xin);
    if (err) return;
    dmd_conv_desc d; memset(&d, 0, sizeof(d));
    if (xproj) {  // skip projection of the block input, accumulated into this conv's output tile
      d.xsrc0 = xin->r0; d.xsrc0_lo = xin->rl0; d.xC0 = xin->C0;
      if (xin->C1) { d.xsrc1 = xin->r1; d.xsrc1_lo = xin->rl1; d.xC1 = xin->C1; }
      d.wpk_x = h->packed ? h->packed + xproj->pk_off : (const void*)1; d.bias_x = P(xproj->b_idx);
    }
    d.src0 = raw ? in.r0 : in.n0; d.src1 = in.C1 ? (raw ? in.r1 : in.n1) : nullptr;
    d.precise = cw.precise; d.wpk_layout = cw.trs;
    if (cw.precise) { d.src0_lo = raw ? in.rl0 : in.nl0; d.src1_lo = in.C1 ? in.rl1 : nullptr; }
    d.C0 = in.C0; d.C1 = in.C1; d.B = pl->B; d.H = in.H; d.W = in.W; d.taps = cw.taps; d.stride = stride;
    d.wpk = h->packed ? h->packed + cw.pk_off : (const void*)1; d.bias = P(cw.b_idx);
    d.Cout = cw.Cout; d.CoutPad = cw.CoutPad;
    d.residual = resid ? (resid->data ? resid->data : (const float*)1) : nullptr; d.out = out.data ? out.data : (float*)1;
    d.out_stats = out_stats ? (out.stats ? out.stats : (double*)1) : nullptr; d.out_gs = out.gs;
    if (cw.precise && (!d.src0_lo || (in.C1 && !d.src1_lo))) { fail("plan: precise conv without low operand parts"); err = 1; return; }
    if (cw.precise && !raw && in.C1) { fail("plan: a split-fp16 conv of a normalised concat is not built"); err = 1; return; }
    if (in.C0 + in.C1 != cw.Cin) { fail("plan: operand channels %d+%d do not match the packed weights (%d)", in.C0, in.C1, cw.Cin); err = 1; return; }
    Op op; op.kind = OP_CONV;
    if (conv_fill(&d, &op.conv, &op.smem, &op.cols)) { err = 1; return; }
    pl->ops.push_back(op);
  }

  // ResBlock.forward (blocks.py:141-147)
  Tens resblock(const ResBlockW& rb, const Tens& x, const Tens* skip) {
    const int H = x.H, W = x.W;
    Operand in1 = prep(x, skip, 0, 1, &rb.n1, 0, 0, true, rb.has_proj != 0, rb.has_proj != 0, rb.c1.precise != 0);
    Tens t = tensor(rb.cout, H, W, true, false);   // its gradient lives in a temporary
    conv(rb.c1, in1, false, 1, nullptr, t, true);
    Operand in2 = prep(t, nullptr, 0, 1, &rb.n2, 0, 0, true, false, rb.c2.precise != 0);
    Tens o = tensor(rb.cout, H, W, true);
    // x + r: r is the block input itself, or proj(input) fused into conv2's accumulator (no r tensor, no extra launch)
    if (rb.has_proj) conv(rb.c2, in2, false, 1, nullptr, o, true, &rb.proj, &in1);
    else conv(rb.c2, in2, false, 1, &x, o, true);
    Rec rec; rec.kind = R_RES; rec.rb = &rb; rec.x = x; rec.has_skip = skip != nullptr; if (skip) rec.skip = *skip;
    rec.t = t; rec.o = o; rec.in1 = in1; rec.in2 = in2;
    if (!rb.has_attn) { record(rec); return o; }
    Tens a = tensor(rb.cout, H, W, true);
    Op op; op.kind = OP_ATTN;
    op.attn = AttnParams{o.data, o.stats, P(rb.an_w), P(rb.an_b), P(rb.qkv_w), P(rb.qkv_b), P(rb.op_w), P(rb.op_b), a.data, a.stats, H * W, rb.cout, o.gs, kGnEps};
    pl->ops.push_back(op);
    rec.a = a;
    record(rec);
    return a;
  }

  // RewEndEncoder.forward (rew_end_model.py:127-132): conv_in, then per level [Downsample] + ResBlocks, then two attention
  // ResBlocks; the same blocks as the U-Net, conditioned on the action embedding.  Output: pl->feat (NHWC, last level).
  int build_rew_end(const std::vector<std::vector<ResBlockW>>& blocks, const std::vector<ConvW>& downs, const ConvW& conv_in, Tens* feat) {
    const dmd_denoiser_config& c = h->cfg;
    const int L = c.num_levels, B = pl->B, H = pl->H, W = pl->W;
    if (H % (1 << (L - 1)) || W % (1 << (L - 1))) return fail("rew_end: H=%d W=%d must be multiples of %d", H, W, 1 << (L - 1));
    int cmax = 16;
    for (int i = 0; i < L; ++i) cmax = c.channels[i] > cmax ? c.channels[i] : cmax;
    const size_t slot_bytes = (plc16_bytes(B, H, W, cmax) + 255) & ~(size_t)255;
    for (int i = 0; i < kScratchSlots; ++i) pl->scratch[i] = (uint8_t*)bump->take(slot_bytes);
    pl->scratch_next = 0;
    pl->CP_in = conv_in.c0_store;
    pl->xin = (float*)bump->take((size_t)B * H * W * pl->CP_in * 4);
    pl->cond = (float*)bump->take((size_t)B * c.cond_channels * 4);
    pl->film = (float*)bump->take((size_t)B * h->film_rows * 4);
    Tens xin{pl->xin, nullptr, pl->CP_in, H, W, 8};
    Tens x = tensor(c.channels[0], H, W, true);
    {
      Operand in0 = prep(xin, nullptr, 0, 0, nullptr, 0, 0, false, false, true);
      conv(conv_in, in0, false, 1, nullptr, x, true);
      Rec rec; rec.kind = R_CONVIN; rec.cw = &conv_in; rec.x = xin; rec.o = x; rec.in1 = in0; record(rec);
    }
    for (int i = 0; i <= L; ++i) {
      if (i > 0 && i < L) {
        Tens xd = tensor(c.channels[i - 1], x.H / 2, x.W / 2, true);
        Operand ind = prep(x, nullptr, 0, 0, nullptr, 0, 0, false, false, downs[i].precise != 0);
        conv(downs[i], ind, false, 2, nullptr, xd, true);
        Rec rec; rec.kind = R_DOWN; rec.cw = &downs[i]; rec.x = x; rec.o = xd; rec.in1 = ind; record(rec);
        x = xd;
      }
      for (auto& rb : blocks[i]) x = resblock(rb, x, nullptr);
    }
    *feat = x;
    return err;
  }

  void resize(const Tens& src, const Tens& dst) {
    Op op; op.kind = OP_RESIZE;
    op.rs = ResizeParams{src.data ? src.data : (const float*)1, dst.data ? dst.data : (float*)1, pl->B, src.H, src.W, dst.H, dst.W, src.C,
                         dst.stats ? dst.stats : (double*)1, dst.gs};
    pl->ops.push_back(op);
  }

  int build() {
    const dmd_denoiser_config& c = h->cfg;
    const int L = c.num_levels, B = pl->B, H = pl->H, W = pl->W;
    const int div = 1 << (L - 1);
    // UNet.forward pads its input (the conv_in output) at the bottom / right to multiples of 2^(levels-1) and crops its output
    // back (blocks.py:225-229,245): conv_in and norm_out / conv_out run at H x W, everything between at Hp x Wp
    const int Hp = (H + div - 1) / div * div, Wp = (W + div - 1) / div * div;
    const bool padded = Hp != H || Wp != W;
    if (padded && pl->train) return fail("denoiser: training at H=%d W=%d (not multiples of %d) needs the pad / crop adjoints, which are not built", H, W, div);
    // operand scratch pool: sized for the largest operand of the network (level 0, widest channel count)
    int cmax = 16;
    for (int i = 0; i < L; ++i) cmax = c.channels[i] > cmax ? c.channels[i] : cmax;
    const size_t slot_bytes = (plc16_bytes(B, Hp, Wp, cmax) + 255) & ~(size_t)255;
    for (int i = 0; i < kScratchSlots; ++i) pl->scratch[i] = (uint8_t*)bump->take(slot_bytes);
    pl->scratch_next = 0;
    pl->CP_in = h->conv_in.c0_store;
    pl->xin = (float*)bump->take((size_t)B * H * W * pl->CP_in * 4);
    pl->cs = (float*)bump->take((size_t)(B + 1) * 4 * 4);  // +1: scalar sigma slot used by the sampler
    pl->cemb = (float*)bump->take((size_t)B * c.cond_channels * 4);
    pl->chid = (float*)bump->take((size_t)B * c.cond_channels * 4);
    pl->cond = (float*)bump->take((size_t)B * c.cond_channels * 4);
    pl->film = (float*)bump->take((size_t)B * h->film_rows * 4);
    Tens xin{pl->xin, nullptr, pl->CP_in, H, W, 8};
    Tens x = tensor(c.channels[0], H, W, !padded);
    {
      Operand in = prep(xin, nullptr, 0, 0, nullptr, 0, 0, false, false, true);
      conv(h->conv_in, in, false, 1, nullptr, x, !padded);
      Rec rec; rec.kind = R_CONVIN; rec.cw = &h->conv_in; rec.x = xin; rec.o = x; rec.in1 = in; record(rec);
    }
    if (padded) {
      Tens xp = tensor(c.channels[0], Hp, Wp, true);
      resize(x, xp);
      x = xp;
    }
    std::vector<std::vector<Tens>> d_outputs;
    for (int i = 0; i < L; ++i) {
      Tens xd = x;
      if (i > 0) {  // Downsample (blocks.py:93-100): raw input, stride 2
        xd = tensor(c.channels[i - 1], x.H / 2, x.W / 2, true);
        Operand in = prep(x, nullptr, 0, 0, nullptr, 0, 0, false, false);
        conv(h->downs[i], in, false, 2, nullptr, xd, true);
        Rec rec; rec.kind = R_DOWN; rec.cw = &h->downs[i]; rec.x = x; rec.o = xd; rec.in1 = in; record(rec);
      }
      std::vector<Tens> outs{xd};
      x = xd;
      for (auto& rb : h->d_blocks[i]) { x = resblock(rb, x, nullptr); outs.push_back(x); }
      d_outputs.push_back(outs);
    }
    for (auto& rb : h->mid) x = resblock(rb, x, nullptr);
    for (int m = 0; m < L; ++m) {
      Tens xu = x;
      if (m > 0) {  // Upsample (blocks.py:103-110): nearest x2 folded into the operand, then conv
        xu = tensor(x.C, x.H * 2, x.W * 2, true);
        Operand in = prep(x, nullptr, 1, 0, nullptr, 0, 0, false, false);
        conv(h->ups[m], in, false, 1, nullptr, xu, true);
        Rec rec; rec.kind = R_UP; rec.cw = &h->ups[m]; rec.x = x; rec.o = xu; rec.in1 = in; record(rec);
      }
      x = xu;
      const std::vector<Tens>& skip = d_outputs[L - 1 - m];  // reversed(d_outputs); block k uses skip[::-1][k]
      const int ns = (int)skip.size();
      for (size_t k = 0; k < h->u_blocks[m].size(); ++k) x = resblock(h->u_blocks[m][k], x, &skip[ns - 1 - (int)k]);
    }
    if (padded) {   // x[..., :h, :w]
      Tens xc = tensor(x.C, H, W, true);
      resize(x, xc);
      x = xc;
    }
    pl->CF = c.img_channels;
    pl->fout = (float*)bump->take((size_t)B * H * W * pl->CF * 4);
    Tens f{pl->fout, nullptr, pl->CF, H, W, pl->CF};
    // conv_out(silu(norm_out(x)))  (inner_model.py:48)
    {
      Operand in = prep(x, nullptr, 0, 2, nullptr, h->i_normout_w, h->i_normout_b, true, false, false);
      conv(h->conv_out, in, false, 1, nullptr, f, false);
      Rec rec; rec.kind = R_OUT; rec.cw = &h->conv_out; rec.x = x; rec.in1 = in; record(rec);
    }
    // sampler temporaries + hoisted conditioning of up to kMaxSamplerEvals evaluations
    const size_t img = (size_t)B * c.img_channels * H * W * 4;
    pl->s_xc = (float*)bump->take(img); pl->s_x2 = (float*)bump->take(img); pl->s_d = (float*)bump->take(img);
    if (!pl->train) {
      const size_t K = kMaxSamplerEvals;
      pl->sig_all = (float*)bump->take(K * 4);
      pl->cemb_all = (float*)bump->take(K * B * c.cond_channels * 4); pl->chid_all = (float*)bump->take(K * B * c.cond_channels * 4);
      pl->cond_all = (float*)bump->take(K * B * c.cond_channels * 4); pl->film_all = (float*)bump->take(K * B * h->film_rows * 4);
    }
    return err;
  }
};

int make_plan(dmd_denoiser* h, Plan* pl, int B, int H, int W, uint8_t* base, size_t* total) {
  pl->B = B; pl->H = H; pl->W = W; pl->ops.clear();
  // pass 1: stats region size (tiny) — run the builder on null bases
  Bump b0{nullptr}, s0{nullptr};
  { Plan tmp; tmp.B = B; tmp.H = H; tmp.W = W; PlanBuilder pb{h, &tmp, &b0, &s0}; if (pb.build()) return 1; }
  const size_t stats_bytes = (s0.off + 255) & ~(size_t)255;
  if (total) *total = stats_bytes + b0.off + 256;
  if (!base) return 0;
  Bump sb{base}, bb{base + stats_bytes};
  pl->base = base; pl->stats = (double*)base; pl->stats_bytes = stats_bytes;
  PlanBuilder pb{h, pl, &bb, &sb};
  if (pb.build()) return 1;
  pl->bytes = stats_bytes + bb.off;
  return 0;
}

// ---------------------------------------------------------------------------------------------- backward plan (training)
// Walks the forward tape in reverse and emits the backward op list.  Every gradient tensor is fp32 NHWC and carries the
// loss scale; "first writer assigns, later writers accumulate" is decided here at plan time (ginit), so no gradient
// buffer needs a memset.  Forward conv inputs (the PLC16 operands) are not kept: the forward prep launch is replayed.
struct BwdBuilder {
  dmd_denoiser* h; Plan* pl; Bump* bump; const EncoderDef* enc = nullptr; int err = 0;
  std::vector<char> ginit;

  const float* P(int idx) const { return h->ptrs.empty() ? nullptr : h->ptrs[idx]; }
  bool was_init(const Tens& t) { const bool w = ginit[t.gid] != 0; ginit[t.gid] = 1; return w; }
  void push(const BOp& b) { pl->bops.push_back(b); }

  void replay(const Operand& o) { BOp b; b.kind = B_PREP; b.prep = pl->ops[o.op].prep; b.prep_nsrc = pl->ops[o.op].prep_nsrc; push(b); }
  // NHWC fp32 gradient [B][Hs][Ws][C] -> PLC16 operand (ups = 2: zero insertion, the adjoint of a stride-2 conv)
  void gprep(const float* g, int C, int Hs, int Ws, int ups, uint8_t* dst) {
    dmd_prep_desc d; memset(&d, 0, sizeof(d));
    d.src0 = g ? g : (const float*)1; d.C0 = C; d.B = pl->B; d.Hs = Hs; d.Ws = Ws; d.upsample = ups; d.dst0 = dst ? dst : (void*)1; d.eps = kGnEps;
    BOp b; b.kind = B_PREP;
    if (prep_fill(&d, &b.prep, &b.prep_nsrc)) { err = 1; return; }
    push(b);
  }
  void colsum(const float* g, long long rows, int C, int Creal, int idx, int idx2 = -1) {
    BOp b; b.kind = B_COLSUM; b.src = g; b.rows = rows; b.C = C; b.Creal = Creal; b.goff = h->goff[idx]; b.goff2 = idx2 >= 0 ? h->goff[idx2] : -1;
    push(b);
  }
  // backward-data for source k of conv cw: out (+)= conv(gy, W_k^T flipped)
  void dgrad(const ConvW& cw, int k, const uint8_t* gy, int H, int W, float* out, bool accumulate) {
    dmd_conv_desc d; memset(&d, 0, sizeof(d));
    d.src0 = gy ? gy : (const void*)1; d.C0 = round_up(cw.Cout, 16); d.B = pl->B; d.H = H; d.W = W; d.taps = cw.taps; d.stride = 1;
    d.wpk = h->packed ? h->packed + cw.pkT_off[k] : (const void*)1;
    d.Cout = cw.srcC[k]; d.CoutPad = round_up(cw.srcC[k], 16);
    d.out = out ? out : (float*)1; d.residual = accumulate ? d.out : nullptr;
    BOp b; b.kind = B_CONV;
    if (conv_fill(&d, &b.conv, &b.smem, &b.cols)) { err = 1; return; }
    push(b);
  }
  void wgrad(const ConvW& cw, const uint8_t* gy, const uint8_t* act, int Ca, int Cin, int ci_off, int H, int W) {
    BOp b; b.kind = B_WGRAD; b.goff = h->goff[cw.w_idx];
    if (wgrad_fill(gy ? gy : (const void*)1, round_up(cw.Cout, 16), act ? act : (const void*)1, Ca, pl->B, H, W, cw.taps,
                   pl->partial ? pl->partial : (float*)1, cw.Cout, Cin, cw.CinReal, ci_off, pl->scale ? pl->scale + 1 : (const float*)1, 1, 0, &b.wg)) { err = 1; return; }
    push(b);
  }
  void norm_bwd(const Tens& x, const float* gy, int mode, const FilmW* film, int c_off, int ctot, int gamma_idx, int beta_idx,
                float* gx, const float* addend, bool accumulate) {
    NormBwdParams nb; memset(&nb, 0, sizeof(nb));
    nb.x = x.data; nb.gy = gy; nb.stats = x.stats; nb.B = pl->B; nb.HW = x.H * x.W; nb.C = x.C; nb.gs = x.gs; nb.mode = mode; nb.act = 1;
    nb.eps = kGnEps; nb.c_off = c_off;
    BOp b1; b1.kind = B_NORM1;
    if (mode == 1) {
      nb.film = pl->film; nb.film_stride = h->film_rows; nb.film_off = film->off; nb.film_ctot = ctot;
      nb.sumB = pl->dfilm ? pl->dfilm + film->off + c_off : nullptr;            // d scale
      nb.sumA = pl->dfilm ? pl->dfilm + film->off + ctot + c_off : nullptr;     // d shift
      nb.sum_stride = h->film_rows;
    } else {
      nb.gamma = P(gamma_idx); nb.beta = P(beta_idx);
      nb.sumA = pl->nsum; nb.sumB = pl->nsum ? pl->nsum + (size_t)pl->B * kMaxCin : nullptr; nb.sum_stride = kMaxCin;
      BOp m; m.kind = B_MEMSET; m.ms_ptr = pl->nsum; m.ms_bytes = (size_t)2 * pl->B * kMaxCin * 4; push(m);
    }
    nb.gx = gx; nb.addend = addend; nb.accumulate = accumulate ? 1 : 0;
    // pixels per block: enough blocks to cover the SMs, at least 32 pixels each
    int ppb = nb.HW;
    while (ppb > 32 && (long long)pl->B * ((nb.HW + ppb - 1) / ppb) < 2 * 148) ppb >>= 1;
    b1.nb = nb; b1.ppb = ppb; b1.chunks = (nb.HW + ppb - 1) / ppb;
    push(b1);
    if (mode == 2) {
      BOp a; a.kind = B_AFFINE; a.nb = nb; a.goff = h->goff[gamma_idx]; a.goff2 = h->goff[beta_idx]; push(a);
    }
    BOp b2 = b1; b2.kind = B_NORM2; push(b2);
  }

  // ResBlock.forward (blocks.py:141-147) backward
  void resblock(const Rec& r) {
    const ResBlockW& rb = *r.rb;
    const int H = r.o.H, W = r.o.W, B = pl->B;
    const long long pix = (long long)B * H * W;
    Tens o = r.o;
    if (rb.has_attn) {  // attention consumes o alone: its backward ASSIGNS o's gradient
      BOp b; b.kind = B_ATTN;
      b.ab = AttnBwdParams{o.data, o.stats, P(rb.an_w), P(rb.an_b), P(rb.qkv_w), P(rb.qkv_b), P(rb.op_w), r.a.grad, o.grad,
                           nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, pl->scale ? pl->scale + 1 : nullptr, H * W, rb.cout, o.gs, kGnEps};
      const int ids[6] = {rb.an_w, rb.an_b, rb.qkv_w, rb.qkv_b, rb.op_w, rb.op_b};
      for (int i = 0; i < 6; ++i) b.goffs[i] = h->goff[ids[i]];
      push(b);
      ginit[o.gid] = 1;
    }
    const Tens* src[2] = {&r.x, r.has_skip ? &r.skip : nullptr};
    const int nsrc = r.has_skip ? 2 : 1;
    // ---- conv2 (+ fused projection): gradient operand of o
    gprep(o.grad, rb.cout, H, W, 0, pl->gyA);
    colsum(o.grad, pix, rb.cout, rb.cout, rb.c2.b_idx, rb.has_proj ? rb.proj.b_idx : -1);
    replay(r.in2);
    wgrad(rb.c2, pl->gyA, r.in2.n0, round_up(rb.cout, 16), rb.cout, 0, H, W);
    dgrad(rb.c2, 0, pl->gyA, H, W, pl->tA, false);
    // ---- norm2 + SiLU
    norm_bwd(r.t, pl->tA, 1, &rb.n2, 0, rb.cout, 0, 0, pl->tB, nullptr, false);
    // ---- conv1
    gprep(pl->tB, rb.cout, H, W, 0, pl->gyB);
    colsum(pl->tB, pix, rb.cout, rb.cout, rb.c1.b_idx);
    replay(r.in1);
    for (int k = 0; k < nsrc; ++k) {
      const uint8_t* act = k == 0 ? r.in1.n0 : r.in1.n1;
      wgrad(rb.c1, pl->gyB, act, round_up(src[k]->C, 16), src[k]->C, rb.c1.srcOff[k], H, W);
      float* ga = k == 0 ? pl->tA : pl->tC;
      dgrad(rb.c1, k, pl->gyB, H, W, ga, false);
      // ---- norm1 + SiLU ; the identity residual (no projection) rides along as the addend of source 0
      const float* addend = (!rb.has_proj && k == 0) ? o.grad : nullptr;
      const bool acc = was_init(*src[k]);
      norm_bwd(*src[k], ga, 1, &rb.n1, rb.c1.srcOff[k], rb.cin, 0, 0, src[k]->grad, addend, acc);
    }
    if (rb.has_proj) {  // r = proj(cat(x, skip)) (blocks.py:142): 1x1 on the raw operand
      for (int k = 0; k < nsrc; ++k) {
        const uint8_t* raw = k == 0 ? r.in1.r0 : r.in1.r1;
        wgrad(rb.proj, pl->gyA, raw, round_up(src[k]->C, 16), src[k]->C, rb.proj.srcOff[k], H, W);
        dgrad(rb.proj, k, pl->gyA, H, W, src[k]->grad, true);
      }
    }
  }

  int build() {
    const int B = pl->B;
    ginit.assign(pl->n_grad_tensors, 0);
    pl->bops.clear();
    for (int i = (int)pl->tape.size() - 1; i >= 0; --i) {
      const Rec& r = pl->tape[i];
      if (r.kind == R_OUT) {
        // conv_out(silu(norm_out(x))) (inner_model.py:48): gF is the scaled gradient of the model output, NHWC x 8 channels
        const ConvW& cw = *r.cw;
        const int H = r.x.H, W = r.x.W;
        gprep(pl->gF, 8, H, W, 0, pl->gyA);
        colsum(pl->gF, (long long)B * H * W, 8, cw.Cout, cw.b_idx);
        replay(r.in1);
        wgrad(cw, pl->gyA, r.in1.n0, round_up(r.x.C, 16), r.x.C, 0, H, W);
        dgrad(cw, 0, pl->gyA, H, W, pl->tA, false);
        norm_bwd(r.x, pl->tA, 2, nullptr, 0, r.x.C, h->i_normout_w, h->i_normout_b, r.x.grad, nullptr, was_init(r.x));
      } else if (r.kind == R_RES) {
        resblock(r);
      } else if (r.kind == R_UP) {   // Upsample (blocks.py:103-110): nearest x2 then conv
        const ConvW& cw = *r.cw;
        const int H = r.o.H, W = r.o.W;
        gprep(r.o.grad, cw.Cout, H, W, 0, pl->gyA);
        colsum(r.o.grad, (long long)B * H * W, cw.Cout, cw.Cout, cw.b_idx);
        replay(r.in1);
        wgrad(cw, pl->gyA, r.in1.n0, round_up(r.x.C, 16), r.x.C, 0, H, W);
        dgrad(cw, 0, pl->gyA, H, W, pl->tA, false);
        BOp b; b.kind = B_POOL; b.src = pl->tA; b.dst = r.x.grad; b.H = r.x.H; b.W = r.x.W; b.C = r.x.C; b.acc = was_init(r.x) ? 1 : 0;
        b.total4 = (long long)B * r.x.H * r.x.W * r.x.C / 4;
        push(b);
      } else if (r.kind == R_DOWN) {  // Downsample (blocks.py:93-100): stride-2 conv == stride-1 conv sampled at even pixels
        const ConvW& cw = *r.cw;
        const int H = r.x.H, W = r.x.W;
        gprep(r.o.grad, cw.Cout, r.o.H, r.o.W, 2, pl->gyA);
        colsum(r.o.grad, (long long)B * r.o.H * r.o.W, cw.Cout, cw.Cout, cw.b_idx);
        replay(r.in1);
        wgrad(cw, pl->gyA, r.in1.n0, round_up(r.x.C, 16), r.x.C, 0, H, W);
        dgrad(cw, 0, pl->gyA, H, W, r.x.grad, was_init(r.x));
      } else {  // R_CONVIN: weight / bias gradients only (the network input needs none)
        const ConvW& cw = *r.cw;
        const int H = r.o.H, W = r.o.W;
        gprep(r.o.grad, cw.Cout, H, W, 0, pl->gyA);
        colsum(r.o.grad, (long long)B * H * W, cw.Cout, cw.Cout, cw.b_idx);
        replay(r.in1);
        wgrad(cw, pl->gyA, r.in1.n0, cw.c0_store, cw.c0_real, 0, H, W);
      }
      if (err) return 1;
    }
    // ---- conditioning path (inner_model.py:45; blocks.py:39): FiLM linears, then cond_proj MLP and action embedding
    const dmd_denoiser_config& c = h->cfg;
    const int CC = c.cond_channels, R = h->film_rows;
    { BOp b; b.kind = B_FILMW; push(b); }
    auto sgemm = [&](const float* A, long long sam, long long sak, const float* Bm, long long sbk, long long sbn, float* C, long long c_goff,
                     long long ldc, int M, int N, int K, int use_inv, int acc) {
      BOp b; b.kind = B_SGEMM; b.ga = A; b.sam = sam; b.sak = sak; b.gb = Bm; b.sbk = sbk; b.sbn = sbn; b.gc = C; b.c_goff = c_goff; b.ldc = ldc;
      b.M = M; b.N = N; b.K = K; b.use_inv = use_inv; b.acc = acc; push(b);
    };
    const float* Wf = h->packed ? (const float*)(h->packed + h->film_w_off) : nullptr;
    sgemm(pl->dfilm, R, 1, Wf, CC, 1, pl->dcond, -1, CC, B, CC, R, 0, 0);                       // dcond = dfilm Wf
    {   // K = R (7168 rows for the default net) over a handful of 64 x 64 output tiles: split K across the SMs
      int cmax = 16;
      for (int i = 0; i < c.num_levels; ++i) cmax = c.channels[i] > cmax ? c.channels[i] : cmax;
      long long fit = (long long)pl->H * pl->W * cmax / CC;   // partials live in tA (B * H * W * cmax floats)
      int splits = R / 256; if (splits > 32) splits = 32; if (splits > fit) splits = (int)fit;
      if (splits > 1) pl->bops.back().chunks = splits;
    }
    if (enc) {   // RewEnd: cond = act_emb(act) (rew_end_model.py:51), one embedding row per encoder row
      BOp b; b.kind = B_EMB; b.src = pl->dcond; b.goff = h->goff[enc->i_actemb]; push(b);
      return err;
    }
    sgemm(pl->dcond, 1, CC, pl->chid, CC, 1, nullptr, h->goff[h->i_cp2w], CC, CC, CC, B, 1, 1);  // dW2 += dcond^T h
    colsum(pl->dcond, B, CC, CC, h->i_cp2b);
    sgemm(pl->dcond, CC, 1, P(h->i_cp2w), CC, 1, pl->dh, -1, CC, B, CC, CC, 0, 0);               // dh = dcond W2
    { BOp b; b.kind = B_LINEAR; b.lin_in = pl->cemb; b.lin_w = P(h->i_cp0w); b.lin_b = P(h->i_cp0b); b.lin_out = pl->cpre; b.lin_K = CC; b.lin_F = CC; push(b); }
    { BOp b; b.kind = B_DSILU; b.src = pl->cpre; b.ga = pl->dh; b.dst = pl->dpre; b.rows = (long long)B * CC; push(b); }
    sgemm(pl->dpre, 1, CC, pl->cemb, CC, 1, nullptr, h->goff[h->i_cp0w], CC, CC, CC, B, 1, 1);   // dW0 += dpre^T e
    colsum(pl->dpre, B, CC, CC, h->i_cp0b);
    sgemm(pl->dpre, CC, 1, P(h->i_cp0w), CC, 1, pl->de, -1, CC, B, CC, CC, 0, 0);                // de = dpre W0
    { BOp b; b.kind = B_EMB; b.src = pl->de; b.goff = h->goff[h->i_actemb]; push(b); }
    return err;
  }
};

// training workspace = forward plan (with gradient buffers) + backward temporaries.  enc: the RewEnd encoder instead of
// the InnerModel (its forward records the encoder's tape and its backward ends in the action embedding)
int make_train_plan(dmd_denoiser* h, Plan* pl, int B, int H, int W, uint8_t* base, size_t* total, const EncoderDef* enc = nullptr) {
  pl->train = true; pl->n_grad_tensors = 0; pl->tape.clear();
  pl->B = B; pl->H = H; pl->W = W; pl->ops.clear(); pl->bops.clear();
  auto build_fwd = [&](PlanBuilder& pb, Plan* p) {
    return enc ? pb.build_rew_end(*enc->blocks, *enc->downs, *enc->conv_in, &p->enc_out) : pb.build();
  };
  Bump b0{nullptr}, s0{nullptr};
  { Plan tmp; tmp.train = true; tmp.B = B; tmp.H = H; tmp.W = W; PlanBuilder pb{h, &tmp, &b0, &s0}; if (build_fwd(pb, &tmp)) return 1; }
  const size_t stats_bytes = (s0.off + 255) & ~(size_t)255;
  Bump sb{base}, bb{base ? base + stats_bytes : nullptr};
  if (base) { pl->base = base; pl->stats = (double*)base; pl->stats_bytes = stats_bytes; }
  if (base) { PlanBuilder pb{h, pl, &bb, &sb}; if (build_fwd(pb, pl)) return 1; } else bb.off = b0.off;
  // backward temporaries
  const dmd_denoiser_config& c = h->cfg;
  int cmax = 16;
  for (int i = 0; i < c.num_levels; ++i) cmax = c.channels[i] > cmax ? c.channels[i] : cmax;
  const size_t act_bytes = (size_t)B * H * W * cmax * 4;
  pl->tA = (float*)bb.take(act_bytes); pl->tB = (float*)bb.take(act_bytes); pl->tC = (float*)bb.take(act_bytes);
  const size_t op_bytes = plc16_bytes(B, H, W, cmax);
  pl->gyA = (uint8_t*)bb.take(op_bytes); pl->gyB = (uint8_t*)bb.take(op_bytes);
  if (!enc) pl->gF = (float*)bb.take((size_t)B * H * W * 8 * 4);
  if (init_kernels()) return 1;
  pl->partial = (float*)bb.take(wgrad_partial_bytes(g_num_sms));
  const int CC = c.cond_channels;
  pl->dcond = (float*)bb.take((size_t)B * CC * 4); pl->dh = (float*)bb.take((size_t)B * CC * 4); pl->cpre = (float*)bb.take((size_t)B * CC * 4);
  pl->dpre = (float*)bb.take((size_t)B * CC * 4); pl->de = (float*)bb.take((size_t)B * CC * 4);
  pl->film_woff = (long long*)bb.take((size_t)h->film_rows * 8); pl->film_boff = (long long*)bb.take((size_t)h->film_rows * 8);
  pl->scale = (float*)bb.take(256);
  // zeroed at the start of every backward: dfilm, affine-norm sums, amax
  uint8_t* z0 = (uint8_t*)bb.take(0);
  pl->dfilm = (float*)bb.take((size_t)B * h->film_rows * 4);
  pl->nsum = (float*)bb.take((size_t)2 * B * kMaxCin * 4);
  pl->amax = (unsigned int*)bb.take(256);
  pl->zero_begin = z0; pl->zero_bytes = base ? (size_t)((uint8_t*)pl->amax + 256 - z0) : 0;
  if (total) *total = stats_bytes + bb.off + 512;
  if (!base) return 0;
  pl->bytes = stats_bytes + bb.off;
  BwdBuilder bw{h, pl, &bb, enc};
  if (bw.build()) return 1;
  // flat-gradient offsets of every FiLM row (weights) / element (biases)
  pl->film_woff_h.assign(h->film_rows, 0); pl->film_boff_h.assign(h->film_rows, 0);
  auto fill_film = [&](const FilmW& f) {
    for (int r = 0; r < 2 * f.C; ++r) { pl->film_woff_h[f.off + r] = h->goff[f.w_idx] + (long long)r * CC; pl->film_boff_h[f.off + r] = h->goff[f.b_idx] + r; }
  };
  auto fill_rb = [&](const ResBlockW& r) { fill_film(r.n1); fill_film(r.n2); };
  if (enc) {
    for (auto& lv : *enc->blocks) for (auto& r : lv) fill_rb(r);
    return 0;
  }
  for (auto& lv : h->d_blocks) for (auto& r : lv) fill_rb(r);
  for (auto& lv : h->u_blocks) for (auto& r : lv) fill_rb(r);
  for (auto& r : h->mid) fill_rb(r);
  return 0;
}

// cond_k >= 0: the conditioning of this evaluation was computed up front by sampler_conditioning (FiLM rows at film_all + k)
int run_forward(dmd_denoiser* h, Plan& pl, const float* noisy, const float* sigma, int sigma_is_scalar, const float* obs,
                const int64_t* act, cudaStream_t st, int prescaled = 0, StackView sv = StackView{}, int cond_k = -1) {
  const dmd_denoiser_config& c = h->cfg;
  const int HW = pl.H * pl.W;
  DMD_CUDA(cudaMemsetAsync(pl.stats, 0, pl.stats_bytes, st));
  pack_denoiser_input_kernel<<<dim3((HW + 255) / 256, pl.B), 256, 0, st>>>(
      noisy, obs, sigma, sigma_is_scalar, pl.xin, pl.cs, c.num_steps_conditioning * c.img_channels, c.img_channels,
      pl.CP_in, HW, c.sigma_data, c.sigma_offset_noise, prescaled, sv);
  DMD_LAUNCH_OK();
  const float* film = pl.film;
  if (cond_k >= 0) {
    film = pl.film_all + (size_t)cond_k * pl.B * h->film_rows;
  } else {
    const int total = pl.B * c.cond_channels;
    cond_embed_kernel<<<(total + 255) / 256, 256, 0, st>>>(pl.cs, nullptr, c.sigma_data, c.sigma_offset_noise, act, h->ptrs[h->i_fourier],
                                                           h->ptrs[h->i_actemb], pl.cemb, pl.B, pl.B, c.cond_channels, c.num_steps_conditioning,
                                                           c.num_actions, sv);
    DMD_LAUNCH_OK();
    if (linear_launch(pl.cemb, h->ptrs[h->i_cp0w], h->ptrs[h->i_cp0b], pl.chid, pl.B, c.cond_channels, c.cond_channels, 1, st)) return 1;
    if (linear_launch(pl.chid, h->ptrs[h->i_cp2w], h->ptrs[h->i_cp2b], pl.cond, pl.B, c.cond_channels, c.cond_channels, 0, st)) return 1;
    if (linear_launch(pl.cond, (const float*)(h->packed + h->film_w_off), (const float*)(h->packed + h->film_b_off), pl.film,
                      pl.B, c.cond_channels, h->film_rows, 0, st)) return 1;
  }
  for (const Op& op : pl.ops) {
    if (op.kind == OP_CONV) { if (conv_launch(op.conv, op.smem, op.cols, st)) return 1; }
    else if (op.kind == OP_PREP) {
      if (op.prep.film != nullptr && op.prep.film != film) { PrepParams pp = op.prep; pp.film = film; if (prep_launch(pp, op.prep_nsrc, st)) return 1; }
      else if (prep_launch(op.prep, op.prep_nsrc, st)) return 1;
    }
    else if (op.kind == OP_FUSED) {
      if (op.fused.film != nullptr && op.fused.film != film) { FusedParams fp = op.fused; fp.film = film; if (fused_launch(fp, op.smem, op.cols, st)) return 1; }
      else if (fused_launch(op.fused, op.smem, op.cols, st)) return 1;
    }
    else if (op.kind == OP_RESIZE) { if (resize_launch(op.rs, st)) return 1; }
    else { if (attn_launch(op.attn, pl.B, st)) return 1; }
  }
  return 0;
}

int run_wrap(dmd_denoiser* h, Plan& pl, const float* x, float* model_out, float* denoised, float* x_out, float* d_out,
             const float* d_prev, const float* x0, int mode, float sigma_hat, float dt, cudaStream_t st) {
  const int HW = pl.H * pl.W, total = pl.B * h->cfg.img_channels * HW;
  wrap_update_kernel<<<(total + 255) / 256, 256, 0, st>>>(pl.fout, x, pl.cs, model_out, denoised, x_out, d_out, d_prev, x0,
                                                         mode, sigma_hat, dt, h->cfg.img_channels, pl.CF, HW, total, kt_slot("wrap", (total + 255) / 256, mode));
  DMD_LAUNCH_OK();
  return 0;
}

int ensure_plan(dmd_denoiser* h, int B, int H, int W, void* ws, size_t ws_bytes) {
  DMD_CHECK(!h->ptrs.empty() && h->packed, "denoiser: call dmd_denoiser_set_weights first");
  Plan& pl = h->plan;
  if (pl.B == B && pl.H == H && pl.W == W && pl.base == (uint8_t*)ws) return 0;
  // size and validate on a scratch plan: the cached plan is replaced only after every check has passed, and is
  // invalidated (never left half-written) if the real build fails
  size_t need = 0;
  { Plan tmp; if (make_plan(h, &tmp, B, H, W, nullptr, &need)) return 1; }
  DMD_CHECK(ws && ws_bytes >= need, "denoiser: workspace too small (%zu < %zu)", ws_bytes, need);
  DMD_CHECK(((uintptr_t)ws & 255) == 0, "denoiser: workspace must be 256-byte aligned");
  for (auto& g : h->graphs) g.valid = false;
  if (make_plan(h, &pl, B, H, W, (uint8_t*)ws, nullptr)) { pl.B = 0; pl.base = nullptr; pl.ops.clear(); return 1; }
  return 0;
}

}  // namespace

extern "C" dmd_denoiser* dmd_denoiser_create(const dmd_denoiser_config* cfg) {
  if (!cfg || cfg->num_levels < 1 || cfg->num_levels > DMD_MAX_LEVELS) { fail("denoiser_create: bad config"); return nullptr; }
  if (cfg->cond_channels % 32 || cfg->cond_channels > 256 || cfg->cond_channels % cfg->num_steps_conditioning) { fail("denoiser_create: cond_channels must be a multiple of 32 (<= 256) and of num_steps_conditioning"); return nullptr; }
  for (int i = 0; i < cfg->num_levels; ++i)
    if (cfg->channels[i] % 32 || cfg->channels[i] > 64) { fail("denoiser_create: channels must be 32 or 64 per level (got %d)", cfg->channels[i]); return nullptr; }
  if (init_kernels()) return nullptr;
  dmd_denoiser* h = new dmd_denoiser();
  h->cfg = *cfg;
  build_structure(h);
  return h;
}
extern "C" void dmd_denoiser_destroy(dmd_denoiser* h) {
  if (!h) return;
  for (auto& g : h->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  delete h;
}
extern "C" int dmd_denoiser_num_tensors(const dmd_denoiser* h) { return h->n_tensors; }
extern "C" size_t dmd_denoiser_packed_bytes(const dmd_denoiser* h) { return h->packed_bytes; }

static int pack_one(dmd_denoiser* h, const ConvW& c, cudaStream_t st) {
  if (dmd_pack_conv_weight(h->ptrs[c.w_idx], h->packed + c.pk_off, c.Cout, c.CoutPad, c.CinReal, c.Cin, c.taps, c.c0_real, c.c0_store, c.trs ? 3 : c.precise, st)) return 1;
  for (int k = 0; k < c.nsrcT; ++k)  // backward-data packs (transposed, flipped), one per concat source
    if (dmd_pack_conv_weight_dgrad(h->ptrs[c.w_idx], h->packed + c.pkT_off[k], c.Cout, c.CinReal, c.srcOff[k], c.srcC[k], c.taps, st)) return 1;
  return 0;
}
static int pack_rb(dmd_denoiser* h, const ResBlockW& r, cudaStream_t st) {
  const int CC = h->cfg.cond_channels;
  if (r.has_proj && pack_one(h, r.proj, st)) return 1;
  if (pack_one(h, r.c1, st) || pack_one(h, r.c2, st)) return 1;
  for (const FilmW* f : {&r.n1, &r.n2}) {
    DMD_CUDA(cudaMemcpyAsync(h->packed + h->film_w_off + (size_t)f->off * CC * 4, h->ptrs[f->w_idx], (size_t)2 * f->C * CC * 4, cudaMemcpyDeviceToDevice, st));
    DMD_CUDA(cudaMemcpyAsync(h->packed + h->film_b_off + (size_t)f->off * 4, h->ptrs[f->b_idx], (size_t)2 * f->C * 4, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

extern "C" int dmd_denoiser_set_weights(dmd_denoiser* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream) {
  DMD_CHECK(h && ptrs_host && packed, "set_weights: null argument");
  DMD_CHECK(n_ptrs == h->n_tensors, "set_weights: expected %d tensors (InnerModel.state_dict order), got %d", h->n_tensors, n_ptrs);
  cudaStream_t st = (cudaStream_t)stream;
  const bool moved = h->packed != (uint8_t*)packed || h->ptrs.empty() || memcmp(h->ptrs.data(), ptrs_host, sizeof(float*) * n_ptrs) != 0;
  h->ptrs.assign(ptrs_host, ptrs_host + n_ptrs);
  h->packed = (uint8_t*)packed;
  if (moved) { h->plan.B = 0; h->tplans.clear(); for (auto& g : h->graphs) g.valid = false; }
  if (pack_one(h, h->conv_in, st) || pack_one(h, h->conv_out, st)) return 1;
  for (auto& lv : h->d_blocks) for (auto& r : lv) if (pack_rb(h, r, st)) return 1;
  for (auto& lv : h->u_blocks) for (auto& r : lv) if (pack_rb(h, r, st)) return 1;
  for (auto& r : h->mid) if (pack_rb(h, r, st)) return 1;
  for (int i = 1; i < h->cfg.num_levels; ++i) if (pack_one(h, h->downs[i], st) || pack_one(h, h->ups[i], st)) return 1;
  return 0;
}

extern "C" size_t dmd_denoiser_workspace_bytes(const dmd_denoiser* h, int B, int H, int W) {
  Plan tmp; size_t need = 0;
  if (make_plan(const_cast<dmd_denoiser*>(h), &tmp, B, H, W, nullptr, &need)) return 0;
  return need;
}

extern "C" int dmd_denoiser_forward(dmd_denoiser* h, int B, int H, int W, const float* noisy, const float* sigma,
                                    int sigma_is_scalar, const float* obs, const int64_t* act, float* out_model,
                                    float* out_denoised, void* workspace, size_t workspace_bytes, void* stream) {
  DMD_CHECK(h && noisy && sigma && obs && act, "denoiser_forward: null argument");
  if (ensure_plan(h, B, H, W, workspace, workspace_bytes)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (run_forward(h, h->plan, noisy, sigma, sigma_is_scalar, obs, act, st)) return 1;
  return run_wrap(h, h->plan, noisy, out_model, out_denoised, nullptr, nullptr, nullptr, nullptr, 0, 1.f, 0.f, st);
}

extern "C" int dmd_inner_model_forward(dmd_denoiser* h, int B, int H, int W, const float* noisy_rescaled,
                                       const float* c_noise, int c_noise_is_scalar, const float* obs_rescaled,
                                       const int64_t* act, float* out, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  DMD_CHECK(h && noisy_rescaled && c_noise && obs_rescaled && act && out, "inner_model_forward: null argument");
  if (ensure_plan(h, B, H, W, workspace, workspace_bytes)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (run_forward(h, h->plan, noisy_rescaled, c_noise, c_noise_is_scalar, obs_rescaled, act, st, 1)) return 1;
  return run_wrap(h, h->plan, noisy_rescaled, out, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 1.f, 0.f, st);
}

// ---------------------------------------------------------------------------------------------- training entry points
namespace {

Plan* find_train_plan(dmd_denoiser* h, int B, int H, int W, void* ws) {
  for (auto& p : h->tplans)
    if (p->B == B && p->H == H && p->W == W && p->base == (uint8_t*)ws) return p.get();
  return nullptr;
}

int ensure_train_plan(dmd_denoiser* h, int B, int H, int W, void* ws, size_t ws_bytes, cudaStream_t st, Plan** out,
                      const EncoderDef* enc = nullptr) {
  DMD_CHECK(!h->ptrs.empty() && h->packed, "denoiser: call dmd_denoiser_set_weights first");
  if ((*out = find_train_plan(h, B, H, W, ws)) != nullptr) return 0;
  size_t need = 0;
  { Plan tmp; if (make_train_plan(h, &tmp, B, H, W, nullptr, &need, enc)) return 1; }
  DMD_CHECK(ws && ws_bytes >= need, "denoiser: training workspace too small (%zu < %zu)", ws_bytes, need);
  DMD_CHECK(((uintptr_t)ws & 255) == 0, "denoiser: workspace must be 256-byte aligned");
  // a plan bound to the same workspace with another shape is stale; keep at most 8 plans
  for (size_t i = 0; i < h->tplans.size();)
    if (h->tplans[i]->base == (uint8_t*)ws) h->tplans.erase(h->tplans.begin() + i); else ++i;
  if (h->tplans.size() >= 8) h->tplans.erase(h->tplans.begin());
  std::unique_ptr<Plan> pl(new Plan());
  if (make_train_plan(h, pl.get(), B, H, W, (uint8_t*)ws, nullptr, enc)) return 1;
  DMD_CUDA(cudaMemcpyAsync(pl->film_woff, pl->film_woff_h.data(), pl->film_woff_h.size() * 8, cudaMemcpyHostToDevice, st));
  DMD_CUDA(cudaMemcpyAsync(pl->film_boff, pl->film_boff_h.data(), pl->film_boff_h.size() * 8, cudaMemcpyHostToDevice, st));
  *out = pl.get();
  h->tplans.push_back(std::move(pl));
  return 0;
}

// the backward op list of a training plan; the caller has cleared the zeroed region and set the loss scale in pl.scale
int run_bops(dmd_denoiser* h, Plan& pl, float* grads, cudaStream_t st) {
  const dmd_denoiser_config& c = h->cfg;
  const int B = pl.B, CC = c.cond_channels;
  const float* inv = pl.scale + 1;
  for (const BOp& b : pl.bops) {
    switch (b.kind) {
      case B_PREP: if (prep_launch(b.prep, b.prep_nsrc, st)) return 1; break;
      case B_CONV: if (conv_launch(b.conv, b.smem, b.cols, st)) return 1; break;
      case B_WGRAD: if (wgrad_launch(b.wg, grads + b.goff, st)) return 1; break;
      case B_COLSUM: {
        const int L4 = (b.C < 256 ? b.C : 256) >> 2, lanes = 256 / L4;
        long long blocks = (b.rows + (long long)lanes * 8 - 1) / ((long long)lanes * 8);
        if (blocks > 592) blocks = 592;
        if (blocks < 1) blocks = 1;
        colsum_kernel<<<dim3((unsigned)blocks, (b.C + 255) / 256), 256, 0, st>>>(b.src, grads + b.goff, b.goff2 >= 0 ? grads + b.goff2 : nullptr, inv, b.rows, b.C, b.Creal);
        DMD_LAUNCH_OK();
        break;
      }
      case B_NORM1: norm_bwd_pass1_kernel<<<dim3(b.chunks, B), kNormThreads, 0, st>>>(b.nb, b.ppb); DMD_LAUNCH_OK(); break;
      case B_NORM2: norm_bwd_pass2_kernel<<<dim3(b.chunks, B), kNormThreads, 0, st>>>(b.nb, b.ppb); DMD_LAUNCH_OK(); break;
      case B_AFFINE:
        affine_param_grad_kernel<<<(b.nb.C + 127) / 128, 128, 0, st>>>(b.nb.sumA, b.nb.sumB, B, b.nb.C, b.nb.sum_stride, grads + b.goff, grads + b.goff2, inv);
        DMD_LAUNCH_OK();
        break;
      case B_POOL: sumpool2_kernel<<<(unsigned)((b.total4 + 255) / 256), 256, 0, st>>>(b.src, b.dst, b.H, b.W, b.C, b.acc, b.total4); DMD_LAUNCH_OK(); break;
      case B_ADD: add_kernel<<<(unsigned)((b.total4 + 255) / 256), 256, 0, st>>>(b.src, b.dst, b.acc, b.total4); DMD_LAUNCH_OK(); break;
      case B_ATTN: {
        AttnBwdParams ab = b.ab;
        ab.dgamma = grads + b.goffs[0]; ab.dbeta = grads + b.goffs[1]; ab.dwqkv = grads + b.goffs[2]; ab.dbqkv = grads + b.goffs[3];
        ab.dwout = grads + b.goffs[4]; ab.dbout = grads + b.goffs[5];
        DMD_CHECK((ab.C == 64 || ab.C == 32) && ab.L == kAttnL, "attention backward: unsupported shape L=%d C=%d", ab.L, ab.C);
        const size_t smem = sizeof(float) * ((size_t)ab.L * (ab.C + 1) * 4 + (size_t)ab.L * (3 * ab.C + 4) * 2 + (size_t)(ab.C / 8) * ab.L * 3);
        if (ab.C == 64) attn_bwd_kernel<64><<<B, kAttnThreads, smem, st>>>(ab);
        else attn_bwd_kernel<32><<<B, kAttnThreads, smem, st>>>(ab);
        DMD_LAUNCH_OK();
        break;
      }
      case B_MEMSET: DMD_CUDA(cudaMemsetAsync(b.ms_ptr, 0, b.ms_bytes, st)); break;
      case B_SGEMM: {
        float* C = b.c_goff >= 0 ? grads + b.c_goff : b.gc;
        if (b.chunks > 1) {   // long-K product (dcond = dfilm Wf, K = all FiLM rows): split-K partials in tA, fixed-order reduce
          const int kchunk = ((b.K + b.chunks - 1) / b.chunks + 15) / 16 * 16;
          const int splits = (b.K + kchunk - 1) / kchunk;
          const long long count = (long long)b.M * b.N;
          sgemm_kernel<<<dim3((b.N + 63) / 64, (b.M + 63) / 64, splits), 256, 0, st>>>(b.ga, b.sam, b.sak, b.gb, b.sbk, b.sbn, pl.tA, b.N, b.M, b.N, b.K, nullptr, 0, kchunk, count);
          DMD_LAUNCH_OK();
          if (b.ldc != b.N) return fail("backward: split-K sgemm needs a dense result");
          splitk_reduce_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(pl.tA, splits, count, C, b.use_inv ? inv : nullptr, b.acc);
          DMD_LAUNCH_OK();
          break;
        }
        sgemm_kernel<<<dim3((b.N + 63) / 64, (b.M + 63) / 64), 256, 0, st>>>(b.ga, b.sam, b.sak, b.gb, b.sbk, b.sbn, C, b.ldc, b.M, b.N, b.K, b.use_inv ? inv : nullptr, b.acc);
        DMD_LAUNCH_OK();
        break;
      }
      case B_FILMW:
        film_wgrad_kernel<<<(h->film_rows + 7) / 8, 256, 0, st>>>(pl.dfilm, pl.cond, grads, pl.film_woff, pl.film_boff, B, h->film_rows, CC, inv);
        DMD_LAUNCH_OK();
        break;
      case B_LINEAR: if (linear_launch(b.lin_in, b.lin_w, b.lin_b, b.lin_out, B, b.lin_K, b.lin_F, 0, st)) return 1; break;
      case B_DSILU: dsilu_mul_kernel<<<(unsigned)((b.rows + 255) / 256), 256, 0, st>>>(b.src, b.ga, b.dst, b.rows); DMD_LAUNCH_OK(); break;
      case B_EMB:
        embedding_bwd_kernel<<<(B * CC + 255) / 256, 256, 0, st>>>(b.src, pl.t_act, grads + b.goff, B, CC, c.num_steps_conditioning, c.num_actions, inv);
        DMD_LAUNCH_OK();
        break;
      default: return fail("backward: unknown op kind %d", b.kind);
    }
  }
  return 0;
}

int run_backward(dmd_denoiser* h, Plan& pl, const float* grad_out, float* grads, cudaStream_t st) {
  const dmd_denoiser_config& c = h->cfg;
  const int B = pl.B, HW = pl.H * pl.W;
  DMD_CUDA(cudaMemsetAsync(grads, 0, (size_t)h->grad_total * 4, st));
  DMD_CUDA(cudaMemsetAsync(pl.zero_begin, 0, pl.zero_bytes, st));
  // loss scale from the incoming gradient, then the scaled NHWC gradient of the model output
  const long long n_out = (long long)B * c.img_channels * HW;
  absmax_kernel<<<(int)std::min<long long>((n_out + 255) / 256, 1184), 256, 0, st>>>(grad_out, pl.amax, n_out);
  DMD_LAUNCH_OK();
  loss_scale_kernel<<<1, 1, 0, st>>>(pl.amax, pl.scale);
  DMD_LAUNCH_OK();
  nchw_to_nhwc_scaled_kernel<<<dim3((HW + 255) / 256, B), 256, 0, st>>>(grad_out, pl.gF, pl.scale, c.img_channels, 8, HW);
  DMD_LAUNCH_OK();
  return run_bops(h, pl, grads, st);
}

}  // namespace

extern "C" size_t dmd_denoiser_train_workspace_bytes(const dmd_denoiser* h, int B, int H, int W) {
  Plan tmp; size_t need = 0;
  if (make_train_plan(const_cast<dmd_denoiser*>(h), &tmp, B, H, W, nullptr, &need)) return 0;
  return need;
}
extern "C" long long dmd_denoiser_grad_layout(const dmd_denoiser* h, long long* offsets, long long* numels, int n) {
  if (!h || n != h->n_tensors) { fail("grad_layout: expected %d entries", h ? h->n_tensors : 0); return -1; }
  for (int i = 0; i < n; ++i) { if (offsets) offsets[i] = h->goff[i]; if (numels) numels[i] = h->numel[i]; }
  return h->grad_total;
}

extern "C" int dmd_inner_model_forward_train(dmd_denoiser* h, int B, int H, int W, const float* noisy_rescaled, const float* c_noise,
                                             int c_noise_is_scalar, const float* obs_rescaled, const int64_t* act, float* out,
                                             void* workspace, size_t workspace_bytes, void* stream) {
  DMD_CHECK(h && noisy_rescaled && c_noise && obs_rescaled && act && out, "inner_model_forward_train: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  Plan* pl = nullptr;
  if (ensure_train_plan(h, B, H, W, workspace, workspace_bytes, st, &pl)) return 1;
  pl->t_act = act;
  if (run_forward(h, *pl, noisy_rescaled, c_noise, c_noise_is_scalar, obs_rescaled, act, st, 1)) return 1;
  return run_wrap(h, *pl, noisy_rescaled, out, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 1.f, 0.f, st);
}

extern "C" int dmd_denoiser_backward(dmd_denoiser* h, int B, int H, int W, const float* grad_out, float* grads, long long grads_numel,
                                     void* workspace, void* stream) {
  DMD_CHECK(h && grad_out && grads && workspace, "denoiser_backward: null argument");
  Plan* plp = find_train_plan(h, B, H, W, workspace);
  DMD_CHECK(plp && plp->train, "denoiser_backward: no matching dmd_inner_model_forward_train on this workspace (B=%d H=%d W=%d)", B, H, W);
  Plan& pl = *plp;
  DMD_CHECK(grads_numel >= h->grad_total, "denoiser_backward: gradient buffer too small (%lld < %lld floats)", grads_numel, h->grad_total);
  DMD_CHECK(((uintptr_t)grads & 15) == 0, "denoiser_backward: gradient buffer must be 16-byte aligned");
  return run_backward(h, pl, grad_out, grads, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------- sampler
namespace {

__global__ void fill_scalar_kernel(float* p, float v) { *p = v; }
struct SigmaList { float v[kMaxSamplerEvals]; };
__global__ void write_sigmas_kernel(float* dst, SigmaList s, int n) { if ((int)threadIdx.x < n) dst[threadIdx.x] = s.v[threadIdx.x]; }

struct SamplerIO { const float* obs; const int64_t* act; StackView sv; float* traj; const float* eps; float* out; };

// DiffusionSampler.sample (diffusion_sampler.py:31-58).  traj[0] holds x ~ N(0, 1) on entry; traj[i+1] receives the iterate after
// step i (the reference's `trajectory` list); the last iterate additionally goes to io.out when that is not the last
// trajectory slot (e.g. straight into the WorldModelEnv's frame ring).  No staging copies: every buffer is used in place.
int sampler_body(dmd_denoiser* h, const dmd_sampler_config* sc, const SamplerIO& io, cudaStream_t st) {
  Plan& pl = h->plan;
  const dmd_denoiser_config& c = h->cfg;
  const int n = sc->num_sigmas;
  const size_t img_elems = (size_t)pl.B * c.img_channels * pl.H * pl.W;
  const int total = (int)img_elems;
  // diffusion_sampler.py:35  gamma_ = min(s_churn / (len(sigmas) - 1), 2**0.5 - 1)
  const double gamma_ = std::fmin((double)sc->s_churn / (double)(n - 1), std::sqrt(2.0) - 1.0);
  // ---- the sigma of every U-Net evaluation is host-known: conditioning (Fourier + action embedding -> cond MLP -> all 44 FiLM
  //      linears) of ALL evaluations in four launches up front instead of four per evaluation inside the loop
  SigmaList sl; int K = 0; bool hoist = true;
  for (int i = 0; i + 1 < n && hoist; ++i) {
    const float sigma = sc->sigmas_host[i], next_sigma = sc->sigmas_host[i + 1];
    if (K + 2 > kMaxSamplerEvals) { hoist = false; break; }
    sl.v[K++] = sigma;   // the network is conditioned on sigma, NOT sigma_hat (diffusion_sampler.py:44)
    if (!(sc->order == 1 || next_sigma == 0.0f)) sl.v[K++] = next_sigma;
  }
  float* sig_dev = pl.cs + (size_t)pl.B * 4;  // spare slot after cs: the un-hoisted fallback's scalar sigma
  if (hoist) {
    write_sigmas_kernel<<<1, 32, 0, st>>>(pl.sig_all, sl, K);
    DMD_LAUNCH_OK();
    const int rows = K * pl.B, CC = c.cond_channels;
    cond_embed_kernel<<<(rows * CC + 255) / 256, 256, 0, st>>>(nullptr, pl.sig_all, c.sigma_data, c.sigma_offset_noise, io.act, h->ptrs[h->i_fourier],
                                                               h->ptrs[h->i_actemb], pl.cemb_all, rows, pl.B, CC, c.num_steps_conditioning, c.num_actions, io.sv);
    DMD_LAUNCH_OK();
    if (linear_launch(pl.cemb_all, h->ptrs[h->i_cp0w], h->ptrs[h->i_cp0b], pl.chid_all, rows, CC, CC, 1, st)) return 1;
    if (linear_launch(pl.chid_all, h->ptrs[h->i_cp2w], h->ptrs[h->i_cp2b], pl.cond_all, rows, CC, CC, 0, st)) return 1;
    if (linear_launch(pl.cond_all, (const float*)(h->packed + h->film_w_off), (const float*)(h->packed + h->film_b_off), pl.film_all,
                      rows, CC, h->film_rows, 0, st)) return 1;
  }
  int k = 0;
  auto forward = [&](const float* x, float sigma_value) -> int {
    if (hoist) { const int kk = k++; return run_forward(h, pl, x, pl.sig_all + kk, 1, io.obs, io.act, st, 0, io.sv, kk); }
    fill_scalar_kernel<<<1, 1, 0, st>>>(sig_dev, sigma_value);
    DMD_LAUNCH_OK();
    return run_forward(h, pl, x, sig_dev, 1, io.obs, io.act, st, 0, io.sv, -1);
  };
  for (int i = 0; i + 1 < n; ++i) {
    const float sigma = sc->sigmas_host[i], next_sigma = sc->sigmas_host[i + 1];
    const double gamma = (sc->s_tmin <= sigma && sigma <= sc->s_tmax) ? gamma_ : 0.0;
    const float sigma_hat = sigma * (float)(gamma + 1.0);
    const float* x = io.traj + (size_t)i * img_elems;
    float* xn = io.traj + (size_t)(i + 1) * img_elems;
    if (gamma > 0.0) {  // churn: x + eps * sqrt(sigma_hat^2 - sigma^2) (diffusion_sampler.py:41-43); the trajectory keeps the un-churned x
      DMD_CHECK(io.eps != nullptr, "sampler: s_churn > 0 needs eps noise from the caller");
      DMD_CHECK(sc->s_noise == 1.0f, "sampler: s_noise != 1 not built yet");
      const float cfac = std::sqrt(sigma_hat * sigma_hat - sigma * sigma);
      axpy_kernel<<<(total + 255) / 256, 256, 0, st>>>(x, io.eps + (size_t)i * img_elems, cfac, pl.s_xc, total);
      DMD_LAUNCH_OK();
      x = pl.s_xc;
    }
    if (forward(x, sigma)) return 1;
    const float dt = next_sigma - sigma_hat;
    if (sc->order == 1 || next_sigma == 0.0f) {
      if (run_wrap(h, pl, x, nullptr, nullptr, xn, nullptr, nullptr, nullptr, 1, sigma_hat, dt, st)) return 1;
    } else {
      // Heun: x_2 = x + d*dt ; denoise(x_2, next_sigma) ; x = x + ((d + d_2)/2)*dt
      if (run_wrap(h, pl, x, nullptr, nullptr, pl.s_x2, pl.s_d, nullptr, nullptr, 1, sigma_hat, dt, st)) return 1;
      if (forward(pl.s_x2, next_sigma)) return 1;
      if (run_wrap(h, pl, pl.s_x2, nullptr, nullptr, xn, nullptr, pl.s_d, x, 2, next_sigma, dt, st)) return 1;
    }
  }
  float* last = io.traj + (size_t)(n - 1) * img_elems;
  if (io.out && io.out != last) DMD_CUDA(cudaMemcpyAsync(io.out, last, img_elems * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace

extern "C" int dmd_sampler_sample(dmd_denoiser* h, const dmd_sampler_config* sc, int B, int H, int W, const float* prev_obs,
                                  const int64_t* prev_act, int ring_head, float* traj, const float* eps, float* out_x,
                                  void* workspace, size_t workspace_bytes, int use_graph, void* stream) {
  DMD_CHECK(h && sc && prev_obs && prev_act && traj, "sampler: null argument");
  DMD_CHECK(sc->num_sigmas >= 2 && sc->sigmas_host, "sampler: need at least 2 sigmas");
  DMD_CHECK(sc->order == 1 || sc->order == 2, "sampler: order must be 1 or 2");
  cudaStream_t st = (cudaStream_t)stream;
  const dmd_denoiser_config& c = h->cfg;
  const int n = sc->num_sigmas, T = c.num_steps_conditioning;
  DMD_CHECK(ring_head >= -1 && ring_head < T, "sampler: ring_head must be -1 (contiguous stacks) or a slot index < %d", T);
  if (init_kernels()) return 1;
  if (h->need_B != B || h->need_H != H || h->need_W != W) {
    h->need_bytes = dmd_denoiser_workspace_bytes(h, B, H, W);
    h->need_B = B; h->need_H = H; h->need_W = W;
  }
  DMD_CHECK(h->need_bytes > 0, "sampler: %s", g_err.c_str());
  DMD_CHECK(workspace_bytes >= h->need_bytes, "sampler: workspace too small (%zu < %zu)", workspace_bytes, h->need_bytes);
  if (ensure_plan(h, B, H, W, workspace, workspace_bytes)) return 1;
  SamplerIO io; memset(&io, 0, sizeof(io));
  io.obs = prev_obs; io.act = prev_act; io.traj = traj; io.eps = eps; io.out = out_x;
  if (ring_head >= 0) {  // frames (T, B, C, H, W), acts (T, B); logical slot k = physical (ring_head + k) % T
    const long long chw = (long long)c.img_channels * H * W;
    io.sv = StackView{T, ring_head, (long long)B * chw, chw, (long long)B, 1};
  }
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  DMD_CUDA(cudaStreamIsCapturing(st, &cap));
  if (!use_graph || cap != cudaStreamCaptureStatusNone) return sampler_body(h, sc, io, st);

  const float churn[4] = {sc->s_churn, sc->s_tmin, sc->s_tmax, sc->s_noise};
  SamplerGraph* g = nullptr;
  for (auto& cand : h->graphs) {
    if (cand.valid && cand.B == B && cand.H == H && cand.W == W && cand.ws == workspace && cand.order == sc->order &&
        cand.obs == prev_obs && cand.act == prev_act && cand.traj == traj && cand.eps == eps && cand.out == out_x &&
        cand.sv.ring_T == io.sv.ring_T && cand.sv.head == io.sv.head && (int)cand.sigmas.size() == n &&
        memcmp(cand.sigmas.data(), sc->sigmas_host, 4 * n) == 0 && memcmp(cand.churn, churn, sizeof(churn)) == 0) { g = &cand; break; }
  }
  if (!g) {
    // graphs bake the buffer addresses in: one graph per distinct set (a WorldModelEnv cycles through T ring heads); keep 8
    if (h->graphs.size() >= 8) {
      size_t victim = 0;
      for (size_t i = 1; i < h->graphs.size(); ++i) if (h->graphs[i].stamp < h->graphs[victim].stamp) victim = i;
      if (h->graphs[victim].exec) cudaGraphExecDestroy(h->graphs[victim].exec);
      h->graphs.erase(h->graphs.begin() + victim);
    }
    SamplerGraph ng;
    cudaGraph_t graph = nullptr;
    if (!h->cap_stream) DMD_CUDA(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    DMD_CUDA(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
    const long long before = g_launches;
    int rc = sampler_body(h, sc, io, h->cap_stream);
    cudaError_t ce = cudaStreamEndCapture(h->cap_stream, &graph);
    ng.kernels = g_launches - before;
    g_launches = before;  // capture does not execute
    if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
    DMD_CHECK(ce == cudaSuccess, "sampler: graph capture failed: %s", cudaGetErrorString(ce));
    ce = cudaGraphInstantiate(&ng.exec, graph, 0);
    cudaGraphDestroy(graph);
    DMD_CHECK(ce == cudaSuccess, "sampler: graph instantiate failed: %s", cudaGetErrorString(ce));
    ng.valid = true; ng.B = B; ng.H = H; ng.W = W; ng.ws = workspace; ng.order = sc->order; ng.has_eps = eps != nullptr;
    ng.obs = prev_obs; ng.act = prev_act; ng.traj = traj; ng.eps = eps; ng.out = out_x; ng.sv = io.sv;
    ng.sigmas.assign(sc->sigmas_host, sc->sigmas_host + n); memcpy(ng.churn, churn, sizeof(churn));
    h->graphs.push_back(ng);
    g = &h->graphs.back();
  }
  g->stamp = ++h->graph_clock;
  DMD_CUDA(cudaGraphLaunch(g->exec, st));
  g_launches += g->kernels;
  return 0;
}

// ---------------------------------------------------------------------------------------------- actor-critic executor
struct dmd_actor_critic {
  dmd_actor_critic_config cfg;
  int n_tensors = 0;
  struct Level { int cin, cout, down; int gn_w, gn_b; ConvW conv; int has_skip; ConvW skip; };
  ConvW conv0;
  std::vector<Level> levels;
  int i_wih = 0, i_whh = 0, i_bih = 0, i_bhh = 0, i_cw = 0, i_cb = 0, i_aw = 0, i_ab = 0;
  int feat_c = 0, feat_hw = 0;
  size_t packed_bytes = 0;
  std::vector<const float*> ptrs;
  uint8_t* packed = nullptr;
  std::vector<long long> numel, goff;   // flat gradient layout (state_dict order), as for the denoiser
  long long grad_total = 0;
};

namespace {

// Forward convs of the actor-critic encoder run in split-fp16 (error ~2^-22): MaxPool2d (actor_critic.py:109) turns a 2^-11
// operand rounding into a different arg-max in a few windows, which moves the encoder GRADIENTS by several per cent against
// the fp32 reference (measured: 2.6e-2 whole-gradient error with fp16 operands, 1.8e-4 with an exact forward).  The encoder
// is 0.12 GFLOP, so the 3x tensor work is noise.  K = 3 * Cin per tap when that fits in shared memory, else three launches.
ConvW ac_conv(dmd_actor_critic* h, int& idx, size_t& pk, int cout, int cin_real, int taps, int c0_store, bool dgrad) {
  ConvW c; c.w_idx = idx++; c.b_idx = idx++;
  h->numel.push_back((long long)cout * cin_real * taps); h->numel.push_back(cout);
  c.Cout = cout; c.CoutPad = round_up(cout, 16); c.CinReal = cin_real; c.taps = taps;
  c.c0_real = cin_real; c.c0_store = c0_store; c.Cin = round_up(c0_store, 16);
  const size_t w1 = (size_t)taps * c.Cin * c.CoutPad * 2;
  c.precise = (3 * w1 <= 120 * 1024) ? 1 : 0;
  c.three_pass = c.precise ? 0 : 1;
  c.pk_off = pk; pk += w1 * (c.precise ? 3 : 1); pk = (pk + 255) & ~(size_t)255;
  if (c.three_pass) { c.pk_lo_off = pk; pk += w1; pk = (pk + 255) & ~(size_t)255; }
  if (dgrad) {
    c.nsrcT = 1; c.srcC[0] = cin_real; c.srcOff[0] = 0; c.pkT_off[0] = pk;
    pk += (size_t)taps * round_up(cout, 16) * round_up(cin_real, 16) * 2; pk = (pk + 255) & ~(size_t)255;
  }
  return c;
}

struct AcBuffers {
  float* x0; void* opnd; void* opnd_lo; std::vector<float*> r, y, pooled; std::vector<double*> st_in, st_y; float *gates, *hx, *cx; double* stats; size_t stats_bytes; size_t total;
};

// lays out the workspace; base may be null (size query)
int ac_layout(const dmd_actor_critic* h, int B, uint8_t* base, AcBuffers* o) {
  const dmd_actor_critic_config& c = h->cfg;
  Bump sb{base};
  const size_t nl = h->levels.size();
  o->st_in.resize(nl + 1); o->st_y.resize(nl);
  int S = c.img_size;
  // statistics first (one memset)
  for (size_t i = 0; i <= nl; ++i) {
    const int C = i == 0 ? c.channels[0] : h->levels[i - 1].cout;
    o->st_in[i] = (double*)sb.take((size_t)B * (C / gn_group_size(C)) * 2 * 8);
  }
  o->stats = (double*)base; o->stats_bytes = (sb.off + 255) & ~(size_t)255;
  Bump bb{base ? base + o->stats_bytes : nullptr};
  o->x0 = (float*)bb.take((size_t)B * S * S * h->conv0.c0_store * 4);
  o->opnd = bb.take(plc16_bytes(B, S, S, 64));  // one operand buffer: every conv's prep immediately precedes it on the stream
  o->opnd_lo = bb.take(plc16_bytes(B, S, S, 64));  // its fp16 low part (split-fp16 forward)
  float* cur = (float*)bb.take((size_t)B * S * S * c.channels[0] * 4);  // conv0 output
  o->r.assign(nl, nullptr); o->y.assign(nl, nullptr); o->pooled.assign(nl + 1, nullptr);
  o->pooled[0] = cur;
  for (size_t i = 0; i < nl; ++i) {
    const auto& lv = h->levels[i];
    if (lv.has_skip) o->r[i] = (float*)bb.take((size_t)B * S * S * lv.cout * 4);
    o->y[i] = (float*)bb.take((size_t)B * S * S * lv.cout * 4);
    if (lv.down) { S /= 2; o->pooled[i + 1] = (float*)bb.take((size_t)B * S * S * lv.cout * 4); }
    else o->pooled[i + 1] = o->y[i];
  }
  o->gates = (float*)bb.take((size_t)B * 4 * c.lstm_dim * 4);
  o->total = o->stats_bytes + bb.off + 256;
  return 0;
}

}  // namespace

extern "C" dmd_actor_critic* dmd_actor_critic_create(const dmd_actor_critic_config* cfg) {
  if (!cfg || cfg->num_levels < 1 || cfg->num_levels > DMD_MAX_LEVELS) { fail("actor_critic_create: bad config"); return nullptr; }
  for (int i = 0; i < cfg->num_levels; ++i)
    if (cfg->channels[i] % 32 || cfg->channels[i] > 64) { fail("actor_critic_create: channels must be 32 or 64 (got %d)", cfg->channels[i]); return nullptr; }
  if (cfg->lstm_dim % 4) { fail("actor_critic_create: lstm_dim must be a multiple of 4"); return nullptr; }
  if (init_kernels()) return nullptr;
  dmd_actor_critic* h = new dmd_actor_critic();
  h->cfg = *cfg;
  int idx = 0; size_t pk = 0;
  // registration order (actor_critic.py:41-47,101-110): encoder.encoder.{0: Conv3x3, k: SmallResBlock(f.0.norm, f.2, skip_projection),
  // MaxPool...}, lstm.{weight_ih, weight_hh, bias_ih, bias_hh}, critic_linear, actor_linear
  h->conv0 = ac_conv(h, idx, pk, cfg->channels[0], cfg->img_channels, 9, round_up(cfg->img_channels, 16), false);
  int S = cfg->img_size;
  for (int i = 0; i < cfg->num_levels; ++i) {
    dmd_actor_critic::Level lv;
    lv.cin = cfg->channels[i > 0 ? i - 1 : 0]; lv.cout = cfg->channels[i]; lv.down = cfg->down[i] ? 1 : 0;
    lv.gn_w = idx++; lv.gn_b = idx++;
    h->numel.push_back(lv.cin); h->numel.push_back(lv.cin);
    lv.conv = ac_conv(h, idx, pk, lv.cout, lv.cin, 9, lv.cin, true);
    lv.has_skip = lv.cin != lv.cout;
    if (lv.has_skip) lv.skip = ac_conv(h, idx, pk, lv.cout, lv.cin, 1, lv.cin, true);
    h->levels.push_back(lv);
    if (lv.down) S /= 2;
  }
  h->feat_c = cfg->channels[cfg->num_levels - 1]; h->feat_hw = S * S;
  h->i_wih = idx++; h->i_whh = idx++; h->i_bih = idx++; h->i_bhh = idx++;
  h->i_cw = idx++; h->i_cb = idx++; h->i_aw = idx++; h->i_ab = idx++;
  {
    const long long D = cfg->lstm_dim, K = (long long)h->feat_c * h->feat_hw;
    for (long long n : {4 * D * K, 4 * D * D, 4 * D, 4 * D, D, 1ll, (long long)cfg->num_actions * D, (long long)cfg->num_actions}) h->numel.push_back(n);
  }
  h->n_tensors = idx; h->packed_bytes = pk + 256;
  h->goff.assign(idx, 0);
  for (int i = 0; i < idx; ++i) { h->goff[i] = h->grad_total; h->grad_total += (h->numel[i] + 3) & ~3ll; }
  return h;
}
extern "C" void dmd_actor_critic_destroy(dmd_actor_critic* h) { delete h; }
extern "C" int dmd_actor_critic_num_tensors(const dmd_actor_critic* h) { return h->n_tensors; }
extern "C" size_t dmd_actor_critic_packed_bytes(const dmd_actor_critic* h) { return h->packed_bytes; }

extern "C" int dmd_actor_critic_set_weights(dmd_actor_critic* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream) {
  DMD_CHECK(h && ptrs_host && packed, "ac set_weights: null argument");
  DMD_CHECK(n_ptrs == h->n_tensors, "ac set_weights: expected %d tensors (ActorCritic.state_dict order), got %d", h->n_tensors, n_ptrs);
  h->ptrs.assign(ptrs_host, ptrs_host + n_ptrs);
  h->packed = (uint8_t*)packed;
  auto pack = [&](const ConvW& c) {
    if (dmd_pack_conv_weight(h->ptrs[c.w_idx], h->packed + c.pk_off, c.Cout, c.CoutPad, c.CinReal, c.Cin, c.taps, c.c0_real, c.c0_store, c.precise, stream)) return 1;
    if (c.three_pass && dmd_pack_conv_weight(h->ptrs[c.w_idx], h->packed + c.pk_lo_off, c.Cout, c.CoutPad, c.CinReal, c.Cin, c.taps, c.c0_real, c.c0_store, 2, stream)) return 1;
    for (int k = 0; k < c.nsrcT; ++k)
      if (dmd_pack_conv_weight_dgrad(h->ptrs[c.w_idx], h->packed + c.pkT_off[k], c.Cout, c.CinReal, c.srcOff[k], c.srcC[k], c.taps, stream)) return 1;
    return 0;
  };
  if (pack(h->conv0)) return 1;
  for (auto& lv : h->levels) { if (pack(lv.conv)) return 1; if (lv.has_skip && pack(lv.skip)) return 1; }
  return 0;
}

extern "C" size_t dmd_actor_critic_workspace_bytes(const dmd_actor_critic* h, int B) {
  AcBuffers b; ac_layout(h, B, nullptr, &b); return b.total;
}

extern "C" int dmd_actor_critic_forward(dmd_actor_critic* h, int B, const float* obs, const float* hx_in, const float* cx_in,
                                        float* logits, float* val, float* hx_out, float* cx_out, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  DMD_CHECK(h && obs && hx_in && cx_in && logits && val && hx_out && cx_out && workspace, "ac forward: null argument");
  DMD_CHECK(!h->ptrs.empty() && h->packed, "ac forward: call dmd_actor_critic_set_weights first");
  DMD_CHECK(((uintptr_t)workspace & 255) == 0, "ac forward: workspace must be 256-byte aligned");
  const dmd_actor_critic_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  AcBuffers b; ac_layout(h, B, (uint8_t*)workspace, &b);
  DMD_CHECK(workspace_bytes >= b.total, "ac forward: workspace too small (%zu < %zu)", workspace_bytes, b.total);
  DMD_CUDA(cudaMemsetAsync(b.stats, 0, b.stats_bytes, st));
  int S = c.img_size;
  if (dmd_nchw_to_nhwc(obs, b.x0, B, c.img_channels, h->conv0.c0_store, S * S, st)) return 1;
  uint8_t* opnd = (uint8_t*)b.opnd;
  uint8_t* opnd_lo = (uint8_t*)b.opnd_lo;
  auto run_conv = [&](const ConvW& cw, const float* src, int Csrc, int hw, int pro, int gamma_idx, int beta_idx, const double* st_in,
                      const float* resid, float* out, double* st_out) -> int {
    dmd_prep_desc pd; memset(&pd, 0, sizeof(pd));
    pd.src0 = src; pd.C0 = Csrc; pd.B = B; pd.Hs = hw; pd.Ws = hw; pd.mode = pro; pd.silu = pro ? 1 : 0;
    pd.stats0 = st_in; pd.gs0 = pro ? gn_group_size(Csrc) : 0;
    if (pro) { pd.gamma = h->ptrs[gamma_idx]; pd.beta = h->ptrs[beta_idx]; }
    pd.eps = kGnEps; pd.dst0 = opnd; pd.dst_lo0 = opnd_lo;   // hi + lo parts: the forward is split-fp16 (see ac_conv)
    PrepParams pp; int nsrc;
    if (prep_fill(&pd, &pp, &nsrc) || prep_launch(pp, nsrc, st)) return 1;
    // passes: one launch with K = 3*Cin, or (A_hi W_hi) then (A_lo W_hi) and (A_hi W_lo) accumulated in place through `residual`
    const int npass = cw.three_pass ? 3 : 1;
    for (int pass = 0; pass < npass; ++pass) {
      dmd_conv_desc d; memset(&d, 0, sizeof(d));
      d.src0 = (pass == 1) ? opnd_lo : opnd; d.C0 = round_up(Csrc, 16); d.B = B; d.H = hw; d.W = hw; d.taps = cw.taps; d.stride = 1;
      if (cw.precise) { d.precise = 1; d.src0_lo = opnd_lo; }
      d.wpk = h->packed + (pass == 2 ? cw.pk_lo_off : cw.pk_off); d.bias = pass == 0 ? h->ptrs[cw.b_idx] : nullptr;
      d.Cout = cw.Cout; d.CoutPad = cw.CoutPad;
      d.residual = pass == 0 ? resid : out; d.out = out;
      d.out_stats = pass == npass - 1 ? st_out : nullptr; d.out_gs = gn_group_size(cw.Cout);
      ConvParams p; size_t smem; int cols;
      if (conv_fill(&d, &p, &smem, &cols)) return 1;
      if (conv_launch(p, smem, cols, st)) return 1;
    }
    return 0;
  };
  // conv0 feeds the first GroupNorm -> statistics in its epilogue
  if (run_conv(h->conv0, b.x0, h->conv0.c0_store, S, 0, 0, 0, nullptr, nullptr, b.pooled[0], b.st_in[0])) return 1;
  for (size_t i = 0; i < h->levels.size(); ++i) {
    const auto& lv = h->levels[i];
    const float* x = b.pooled[i];
    const float* r = x;
    if (lv.has_skip) { if (run_conv(lv.skip, x, lv.cin, S, 0, 0, 0, nullptr, nullptr, b.r[i], nullptr)) return 1; r = b.r[i]; }
    // SmallResBlock: skip(x) + conv3x3(silu(GroupNorm(x)))  (blocks.py:122-123)
    double* st_y = lv.down ? nullptr : b.st_in[i + 1];
    if (run_conv(lv.conv, x, lv.cin, S, 2, lv.gn_w, lv.gn_b, b.st_in[i], r, b.y[i], st_y)) return 1;
    if (lv.down) {
      const int total = (S / 2) * (S / 2) * lv.cout;
      maxpool2_stats_kernel<<<dim3((total + 255) / 256, B), 256, 0, st>>>(b.y[i], b.pooled[i + 1], i + 1 < h->levels.size() ? b.st_in[i + 1] : nullptr,
                                                                         S, S, lv.cout, gn_group_size(lv.cout));
      DMD_LAUNCH_OK();
      S /= 2;
    }
  }
  const float* feat = b.pooled[h->levels.size()];
  const int K = h->feat_c * h->feat_hw, D = c.lstm_dim;
  if (linear_launch(feat, h->ptrs[h->i_wih], h->ptrs[h->i_bih], b.gates, B, K, 4 * D, 0, st, 0, h->feat_hw)) return 1;
  if (linear_launch(hx_in, h->ptrs[h->i_whh], h->ptrs[h->i_bhh], b.gates, B, D, 4 * D, 0, st, 1, 0)) return 1;
  lstm_gates_kernel<<<(B * D + 255) / 256, 256, 0, st>>>(b.gates, cx_in, hx_out, cx_out, B, D);
  DMD_LAUNCH_OK();
  if (linear_launch(hx_out, h->ptrs[h->i_aw], h->ptrs[h->i_ab], logits, B, D, c.num_actions, 0, st)) return 1;
  if (linear_launch(hx_out, h->ptrs[h->i_cw], h->ptrs[h->i_cb], val, B, D, 1, 0, st)) return 1;
  return 0;
}


// ---------------------------------------------------------------------------------------------- actor-critic training
// ActorCritic.predict_act_value under autograd (actor_critic.py:68-73, called with grad from env_loop.py:31,57): the forward
// above leaves every activation in its workspace; dmd_actor_critic_backward consumes it.  One call = one autograd node of
// the BPTT graph; torch's engine chains the nodes through (g_hx_in, g_cx_in) and accumulates the parameter gradients.
namespace {

struct AcScratch {
  float *g_a, *g_b, *tA; uint8_t *gy_op, *x_op; float *dgates, *g_h, *g_xflat, *x_flat, *nsum, *scale, *partial; unsigned int* amax; size_t total;
};
int ac_scratch_layout(const dmd_actor_critic* h, int B, uint8_t* base, AcScratch* o) {
  const dmd_actor_critic_config& c = h->cfg;
  Bump bb{base};
  const int S = c.img_size;
  const size_t act = (size_t)B * S * S * 64 * 4;
  o->g_a = (float*)bb.take(act); o->g_b = (float*)bb.take(act); o->tA = (float*)bb.take(act);
  o->gy_op = (uint8_t*)bb.take(plc16_bytes(B, S, S, 64)); o->x_op = (uint8_t*)bb.take(plc16_bytes(B, S, S, 64));
  const int D = c.lstm_dim, K = h->feat_c * h->feat_hw;
  o->dgates = (float*)bb.take((size_t)B * 4 * D * 4); o->g_h = (float*)bb.take((size_t)B * D * 4);
  o->g_xflat = (float*)bb.take((size_t)B * K * 4); o->x_flat = (float*)bb.take((size_t)B * K * 4);
  o->nsum = (float*)bb.take((size_t)2 * B * kMaxCin * 4);
  o->scale = (float*)bb.take(256); o->amax = (unsigned int*)bb.take(256);
  if (init_kernels()) return 1;
  o->partial = (float*)bb.take(wgrad_partial_bytes(g_num_sms));
  o->total = bb.off + 256;
  return 0;
}

}  // namespace

extern "C" size_t dmd_actor_critic_backward_scratch_bytes(const dmd_actor_critic* h, int B) {
  AcScratch s; if (ac_scratch_layout(h, B, nullptr, &s)) return 0; return s.total;
}
extern "C" long long dmd_actor_critic_grad_layout(const dmd_actor_critic* h, long long* offsets, long long* numels, int n) {
  if (!h || n != h->n_tensors) { fail("ac grad_layout: expected %d entries", h ? h->n_tensors : 0); return -1; }
  for (int i = 0; i < n; ++i) { if (offsets) offsets[i] = h->goff[i]; if (numels) numels[i] = h->numel[i]; }
  return h->grad_total;
}

static int ac_backward_impl(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                            const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx,
                            float* grads, long long grads_numel, int accumulate, float* g_hx_in, float* g_cx_in, void* workspace,
                            void* scratch, size_t scratch_bytes, void* stream);
extern "C" int dmd_actor_critic_backward(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                                         const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx,
                                         float* grads, long long grads_numel, float* g_hx_in, float* g_cx_in, void* workspace,
                                         void* scratch, size_t scratch_bytes, void* stream) {
  return ac_backward_impl(h, B, hx_in, cx_in, hx_out, g_logits, g_val, g_hx, g_cx, grads, grads_numel, 0, g_hx_in, g_cx_in, workspace, scratch, scratch_bytes, stream);
}
extern "C" int dmd_actor_critic_backward_accumulate(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                                                    const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx,
                                                    float* grads, long long grads_numel, float* g_hx_in, float* g_cx_in, void* workspace,
                                                    void* scratch, size_t scratch_bytes, void* stream) {
  return ac_backward_impl(h, B, hx_in, cx_in, hx_out, g_logits, g_val, g_hx, g_cx, grads, grads_numel, 1, g_hx_in, g_cx_in, workspace, scratch, scratch_bytes, stream);
}
// every parameter-gradient writer below ADDS its (un-scaled) contribution, so "accumulate" is simply "do not clear the buffer first"
static int ac_backward_impl(dmd_actor_critic* h, int B, const float* hx_in, const float* cx_in, const float* hx_out,
                            const float* g_logits, const float* g_val, const float* g_hx, const float* g_cx,
                            float* grads, long long grads_numel, int accumulate, float* g_hx_in, float* g_cx_in, void* workspace,
                            void* scratch, size_t scratch_bytes, void* stream) {
  DMD_CHECK(h && hx_in && cx_in && hx_out && grads && g_hx_in && g_cx_in && workspace && scratch, "ac backward: null argument");
  DMD_CHECK(!h->ptrs.empty() && h->packed, "ac backward: call dmd_actor_critic_set_weights first");
  DMD_CHECK(grads_numel >= h->grad_total && ((uintptr_t)grads & 15) == 0, "ac backward: bad gradient buffer");
  DMD_CHECK(((uintptr_t)scratch & 255) == 0, "ac backward: scratch must be 256-byte aligned");
  const dmd_actor_critic_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  AcBuffers b; ac_layout(h, B, (uint8_t*)workspace, &b);
  AcScratch sc; if (ac_scratch_layout(h, B, (uint8_t*)scratch, &sc)) return 1;
  DMD_CHECK(scratch_bytes >= sc.total, "ac backward: scratch too small (%zu < %zu)", scratch_bytes, sc.total);
  const int D = c.lstm_dim, A = c.num_actions, K = h->feat_c * h->feat_hw;
  auto G = [&](int idx) { return grads + h->goff[idx]; };
  auto sgemm = [&](const float* Am, long long sam, long long sak, const float* Bm, long long sbk, long long sbn, float* C, long long ldc,
                   int M, int N, int Kd, int acc) -> int {
    sgemm_kernel<<<dim3((N + 63) / 64, (M + 63) / 64), 256, 0, st>>>(Am, sam, sak, Bm, sbk, sbn, C, ldc, M, N, Kd, nullptr, acc);
    DMD_LAUNCH_OK();
    return 0;
  };
  auto colsum = [&](const float* x, long long rows, int C, int Creal, float* out, float* out2, const float* inv) -> int {
    const int L4 = (C < 256 ? C : 256) >> 2, lanes = 256 / L4;
    long long blocks = (rows + (long long)lanes * 8 - 1) / ((long long)lanes * 8);
    blocks = blocks > 592 ? 592 : (blocks < 1 ? 1 : blocks);
    colsum_kernel<<<dim3((unsigned)blocks, (C + 255) / 256), 256, 0, st>>>(x, out, out2, inv, rows, C, Creal);
    DMD_LAUNCH_OK();
    return 0;
  };
  if (!accumulate) DMD_CUDA(cudaMemsetAsync(grads, 0, (size_t)h->grad_total * 4, st));
  DMD_CUDA(cudaMemsetAsync(sc.amax, 0, 256, st));
  // ---- heads (actor_critic.py:73)
  heads_bwd_kernel<<<(B * D + 255) / 256, 256, 0, st>>>(g_hx, g_logits, g_val, h->ptrs[h->i_aw], h->ptrs[h->i_cw], sc.g_h, B, D, A);
  DMD_LAUNCH_OK();
  if (g_logits) {
    if (sgemm(g_logits, 1, A, hx_out, D, 1, G(h->i_aw), D, A, D, B, 1)) return 1;          // dWa += g_logits^T h'
    small_colsum_kernel<<<(A + 31) / 32, 32, 0, st>>>(g_logits, B, A, G(h->i_ab));           // dba (A need not be a multiple of 4)
    DMD_LAUNCH_OK();
  }
  if (g_val) { vec_outer_sum_kernel<<<(D + 127) / 128, 128, 0, st>>>(g_val, hx_out, G(h->i_cw), G(h->i_cb), B, D); DMD_LAUNCH_OK(); }
  // ---- LSTMCell (actor_critic.py:72)
  lstm_cell_bwd_kernel<<<(B * D + 255) / 256, 256, 0, st>>>(b.gates, cx_in, sc.g_h, g_cx, sc.dgates, g_cx_in, B, D);
  DMD_LAUNCH_OK();
  const float* feat = b.pooled[h->levels.size()];
  if (dmd_nhwc_to_nchw(feat, sc.x_flat, B, h->feat_c, h->feat_c, h->feat_hw, st)) return 1;   // x.flatten(start_dim=1) of the NCHW feature map
  if (sgemm(sc.dgates, 1, 4 * D, sc.x_flat, K, 1, G(h->i_wih), K, 4 * D, K, B, 1)) return 1;  // dWih += dgates^T x
  if (sgemm(sc.dgates, 1, 4 * D, hx_in, D, 1, G(h->i_whh), D, 4 * D, D, B, 1)) return 1;      // dWhh += dgates^T hx
  if (colsum(sc.dgates, B, 4 * D, 4 * D, G(h->i_bih), G(h->i_bhh), nullptr)) return 1;
  if (sgemm(sc.dgates, 4 * D, 1, h->ptrs[h->i_whh], D, 1, g_hx_in, D, B, D, 4 * D, 0)) return 1;   // g_hx = dgates Whh
  if (sgemm(sc.dgates, 4 * D, 1, h->ptrs[h->i_wih], K, 1, sc.g_xflat, K, B, K, 4 * D, 0)) return 1;  // g_x = dgates Wih
  // ---- encoder (actor_critic.py:101-113): the feature gradient enters the fp16 tensor-core path with a loss scale
  float* g_cur = sc.g_a;    // gradient of pooled[i+1]; g_a / g_b ping-pong down the encoder
  auto other = [&](float* p) { return p == sc.g_a ? sc.g_b : sc.g_a; };
  if (dmd_nchw_to_nhwc(sc.g_xflat, g_cur, B, h->feat_c, h->feat_c, h->feat_hw, st)) return 1;
  {
    const long long n = (long long)B * K;
    absmax_kernel<<<(int)std::min<long long>((n + 255) / 256, 592), 256, 0, st>>>(g_cur, sc.amax, n);
    DMD_LAUNCH_OK();
    loss_scale_kernel<<<1, 1, 0, st>>>(sc.amax, sc.scale);
    DMD_LAUNCH_OK();
    scale_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g_cur, sc.scale, n);
    DMD_LAUNCH_OK();
  }
  const float* inv = sc.scale + 1;
  auto prep = [&](const float* src, int Csrc, int hw, int mode, int gamma_idx, int beta_idx, const double* stats, uint8_t* dst) -> int {
    dmd_prep_desc pd; memset(&pd, 0, sizeof(pd));
    pd.src0 = src; pd.C0 = Csrc; pd.B = B; pd.Hs = hw; pd.Ws = hw; pd.mode = mode; pd.silu = mode ? 1 : 0;
    pd.stats0 = stats; pd.gs0 = mode ? gn_group_size(Csrc) : 0;
    if (mode) { pd.gamma = h->ptrs[gamma_idx]; pd.beta = h->ptrs[beta_idx]; }
    pd.eps = kGnEps; pd.dst0 = dst;
    PrepParams pp; int nsrc;
    if (prep_fill(&pd, &pp, &nsrc)) return 1;
    return prep_launch(pp, nsrc, st);
  };
  auto wgrad = [&](const ConvW& cw, const uint8_t* gy, const uint8_t* act, int Ca, int hw) -> int {
    WgradLaunch L;
    if (wgrad_fill(gy, round_up(cw.Cout, 16), act, Ca, B, hw, hw, cw.taps, sc.partial, cw.Cout, cw.CinReal, cw.CinReal, 0, inv, 1, 0, &L)) return 1;
    return wgrad_launch(L, G(cw.w_idx), st);
  };
  auto dgrad = [&](const ConvW& cw, const uint8_t* gy, int hw, float* out, bool accumulate) -> int {
    dmd_conv_desc d; memset(&d, 0, sizeof(d));
    d.src0 = gy; d.C0 = round_up(cw.Cout, 16); d.B = B; d.H = hw; d.W = hw; d.taps = cw.taps; d.stride = 1;
    d.wpk = h->packed + cw.pkT_off[0]; d.Cout = cw.srcC[0]; d.CoutPad = round_up(cw.srcC[0], 16);
    d.out = out; d.residual = accumulate ? out : nullptr;
    ConvParams p; size_t smem; int cols;
    if (conv_fill(&d, &p, &smem, &cols)) return 1;
    return conv_launch(p, smem, cols, st);
  };
  // spatial size of every level's input
  std::vector<int> size_in(h->levels.size() + 1);
  { int S = c.img_size; for (size_t i = 0; i < h->levels.size(); ++i) { size_in[i] = S; if (h->levels[i].down) S /= 2; } size_in[h->levels.size()] = S; }
  for (int i = (int)h->levels.size() - 1; i >= 0; --i) {
    const auto& lv = h->levels[i];
    const int S = size_in[i];
    const float* gy = g_cur;            // gradient of the SmallResBlock output y[i] (NHWC, S x S x cout)
    float* gx = other(g_cur);           // gradient of the block input pooled[i]
    if (lv.down) {                      // un-pool into the other buffer; the pooled gradient's buffer then takes gx
      const int total = (S / 2) * (S / 2) * lv.cout;
      maxpool2_bwd_kernel<<<dim3((total + 255) / 256, B), 256, 0, st>>>(b.y[i], g_cur, other(g_cur), S, S, lv.cout);
      DMD_LAUNCH_OK();
      gy = other(g_cur);
      gx = g_cur;
    }
    const long long pix = (long long)B * S * S;
    // SmallResBlock (blocks.py:116-123): y = skip(x) + conv3x3(silu(GroupNorm(x)))
    if (prep(gy, lv.cout, S, 0, 0, 0, nullptr, sc.gy_op)) return 1;
    if (colsum(gy, pix, lv.cout, lv.cout, G(lv.conv.b_idx), lv.has_skip ? G(lv.skip.b_idx) : nullptr, inv)) return 1;
    if (prep(b.pooled[i], lv.cin, S, 2, lv.gn_w, lv.gn_b, b.st_in[i], sc.x_op)) return 1;
    if (wgrad(lv.conv, sc.gy_op, sc.x_op, round_up(lv.cin, 16), S)) return 1;
    if (dgrad(lv.conv, sc.gy_op, S, sc.tA, false)) return 1;
    {
      NormBwdParams nb; memset(&nb, 0, sizeof(nb));
      nb.x = b.pooled[i]; nb.gy = sc.tA; nb.stats = b.st_in[i]; nb.B = B; nb.HW = S * S; nb.C = lv.cin; nb.gs = gn_group_size(lv.cin);
      nb.mode = 2; nb.act = 1; nb.gamma = h->ptrs[lv.gn_w]; nb.beta = h->ptrs[lv.gn_b]; nb.eps = kGnEps;
      nb.sumA = sc.nsum; nb.sumB = sc.nsum + (size_t)B * kMaxCin; nb.sum_stride = kMaxCin;
      nb.gx = gx; nb.addend = lv.has_skip ? nullptr : gy; nb.accumulate = 0;
      DMD_CUDA(cudaMemsetAsync(sc.nsum, 0, (size_t)2 * B * kMaxCin * 4, st));
      int ppb = nb.HW;
      while (ppb > 32 && (long long)B * ((nb.HW + ppb - 1) / ppb) < 2 * 148) ppb >>= 1;
      const int chunks = (nb.HW + ppb - 1) / ppb;
      norm_bwd_pass1_kernel<<<dim3(chunks, B), kNormThreads, 0, st>>>(nb, ppb);
      DMD_LAUNCH_OK();
      affine_param_grad_kernel<<<(nb.C + 127) / 128, 128, 0, st>>>(nb.sumA, nb.sumB, B, nb.C, nb.sum_stride, G(lv.gn_w), G(lv.gn_b), inv);
      DMD_LAUNCH_OK();
      norm_bwd_pass2_kernel<<<dim3(chunks, B), kNormThreads, 0, st>>>(nb, ppb);
      DMD_LAUNCH_OK();
    }
    if (lv.has_skip) {  // 1x1 skip projection on the raw input
      if (prep(b.pooled[i], lv.cin, S, 0, 0, 0, nullptr, sc.x_op)) return 1;
      if (wgrad(lv.skip, sc.gy_op, sc.x_op, round_up(lv.cin, 16), S)) return 1;
      if (dgrad(lv.skip, sc.gy_op, S, gx, true)) return 1;
    }
    g_cur = gx;
  }
  {  // conv0 (Conv3x3(img_channels -> channels[0])): weight / bias gradients only
    const int S = c.img_size;
    if (prep(g_cur, h->conv0.Cout, S, 0, 0, 0, nullptr, sc.gy_op)) return 1;
    if (colsum(g_cur, (long long)B * S * S, h->conv0.Cout, h->conv0.Cout, G(h->conv0.b_idx), nullptr, inv)) return 1;
    if (prep(b.x0, h->conv0.c0_store, S, 0, 0, 0, nullptr, sc.x_op)) return 1;
    WgradLaunch L;
    if (wgrad_fill(sc.gy_op, round_up(h->conv0.Cout, 16), sc.x_op, h->conv0.c0_store, B, S, S, 9, sc.partial, h->conv0.Cout, h->conv0.CinReal,
                   h->conv0.CinReal, 0, inv, 1, 0, &L)) return 1;
    if (wgrad_launch(L, G(h->conv0.w_idx), st)) return 1;
  }
  return 0;
}


// compute_lambda_returns (actor_critic.py:116-143) on the device, bit-identical to the torch expression (SURVEY.md 8 f4).
extern "C" int dmd_lambda_returns(const float* rew, const int64_t* end, const int64_t* trunc, const float* val_bootstrap, float* out,
                                  int B, int T, double gamma, double lambda_, void* stream) {
  DMD_CHECK(rew && end && trunc && val_bootstrap && out && B > 0 && T > 0, "lambda_returns: bad arguments");
  lambda_returns_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rew, (const long long*)end, (const long long*)trunc, val_bootstrap, out, B, T,
                                                                         (float)gamma, (float)lambda_, (float)(1.0 - lambda_));
  DMD_LAUNCH_OK();
  return 0;
}


// ---------------------------------------------------------------------------------------------- reward / termination model
// RewEndModel.predict_rew_end (src/models/rew_end_model.py:42-55; SURVEY.md 8 f1): runs once per imagined step between the
// sampler and the policy (world_model_env.py:97), and over the burn-in frames of every fresh episode (:120-129).
//   encoder (conv_in + ResBlocks at C = 32 conditioned on the action embedding + two attention ResBlocks) -> (b t) features
//   -> single-layer LSTM over time -> Linear / SiLU / Linear head -> 3 reward logits + 2 termination logits.
// Rows are processed TIME-MAJOR (row = k * b + n) so that every LSTM step reads b contiguous feature rows.
struct dmd_rew_end {
  dmd_rew_end_config cfg;
  dmd_denoiser core;     // parameter pointers / packed weights / FiLM table / plan of the encoder (reuses the U-Net block executor)
  ConvW conv_in;
  std::vector<std::vector<ResBlockW>> blocks;
  std::vector<ConvW> downs;
  int i_actemb = 0, i_wih = 0, i_whh = 0, i_bih = 0, i_bhh = 0, i_h0w = 0, i_h0b = 0, i_h2w = 0;
  int feat_c = 0, feat_hw = 0;
  Tens feat;
  int planB = 0; void* plan_ws = nullptr;
  float *x_gates = nullptr, *y = nullptr, *hid = nullptr, *logits_tm = nullptr, *hc[2] = {nullptr, nullptr};
  // Training plans (core.tplans, apart from the inference plan core.plan) run the encoder's ResBlock and Downsample convs in
  // split-fp16: with single-fp16 operands the forward's rounding reaches the LSTM / head weight gradients (emulated: 1.3e-3
  // whole-gradient error vs fp32; split: 3.3e-4, DESIGN.md section 2).  Copies of those convs with their own split packs;
  // the backward-data packs are shared.
  std::vector<std::vector<ResBlockW>> tblocks;
  std::vector<ConvW> tdowns;
  EncoderDef enc{};
};

namespace {

__global__ void pack_rew_end_input_kernel(const float* __restrict__ obs, const float* __restrict__ next_obs, const int64_t* __restrict__ act,
                                          const float* __restrict__ act_emb, float* __restrict__ xin, float* __restrict__ cond, int b, int t,
                                          int C, int CP, int HW, int CC, int num_actions, int64_t* __restrict__ act_tm = nullptr) {
  // row r = k * b + n (time-major)  <-  obs[n][k], next_obs[n][k], act[n][k]
  const int r = blockIdx.y, k = r / b, n = r - k * b;
  const size_t src = ((size_t)n * t + k) * C * HW;
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0) {
    long long a = act[(size_t)n * t + k];
    a = a < 0 ? 0 : (a >= num_actions ? num_actions - 1 : a);
    for (int j = threadIdx.x; j < CC; j += blockDim.x) cond[(size_t)r * CC + j] = act_emb[(size_t)a * CC + j];
    if (act_tm && threadIdx.x == 0) act_tm[r] = a;   // training: the embedding backward reads the actions in row order
  }
  if (pix >= HW) return;
  float* o = xin + ((size_t)r * HW + pix) * CP;
  for (int ch = 0; ch < CP; ++ch) {
    float v = 0.f;
    if (ch < C) v = obs[src + (size_t)ch * HW + pix];
    else if (ch < 2 * C) v = next_obs[src + (size_t)(ch - C) * HW + pix];
    o[ch] = v;
  }
}
// logits_tm [t*b][5] (time-major) -> rew [b][t][3], end [b][t][2]
__global__ void split_logits_kernel(const float* __restrict__ tm, float* __restrict__ rew, float* __restrict__ end, int b, int t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b * t) return;
  const int n = i / t, k = i - n * t;
  const float* s = tm + ((size_t)k * b + n) * 5;
  rew[(size_t)i * 3] = s[0]; rew[(size_t)i * 3 + 1] = s[1]; rew[(size_t)i * 3 + 2] = s[2];
  end[(size_t)i * 2] = s[3]; end[(size_t)i * 2 + 1] = s[4];
}
// the adjoint of split_logits_kernel: g_rew [b][t][3], g_end [b][t][2] -> g_tm [t*b][5] (time-major)
__global__ void merge_logits_grad_kernel(const float* __restrict__ g_rew, const float* __restrict__ g_end, float* __restrict__ g_tm, int b, int t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b * t) return;
  const int n = i / t, k = i - n * t;
  float* d = g_tm + ((size_t)k * b + n) * 5;
  d[0] = g_rew[(size_t)i * 3]; d[1] = g_rew[(size_t)i * 3 + 1]; d[2] = g_rew[(size_t)i * 3 + 2];
  d[3] = g_end[(size_t)i * 2]; d[4] = g_end[(size_t)i * 2 + 1];
}

// the encoder's forward op list (inference and training plans alike)
int run_encoder_ops(const Plan& pl, cudaStream_t st) {
  for (const Op& op : pl.ops) {
    if (op.kind == OP_CONV) { if (conv_launch(op.conv, op.smem, op.cols, st)) return 1; }
    else if (op.kind == OP_PREP) { if (prep_launch(op.prep, op.prep_nsrc, st)) return 1; }
    else if (op.kind == OP_FUSED) { if (fused_launch(op.fused, op.smem, op.cols, st)) return 1; }
    else { if (attn_launch(op.attn, pl.B, st)) return 1; }
  }
  return 0;
}

int rew_end_layout(dmd_rew_end* h, int B, int H, int W, uint8_t* base, size_t* total) {
  dmd_denoiser* core = &h->core;
  Plan& pl = core->plan;
  pl.train = false; pl.B = B; pl.H = H; pl.W = W; pl.ops.clear();
  Bump b0{nullptr}, s0{nullptr};
  Tens feat;
  { Plan tmp; tmp.B = B; tmp.H = H; tmp.W = W; PlanBuilder pb{core, &tmp, &b0, &s0}; if (pb.build_rew_end(h->blocks, h->downs, h->conv_in, &feat)) return 1; }
  const size_t stats_bytes = (s0.off + 255) & ~(size_t)255;
  Bump sb{base}, bb{base ? base + stats_bytes : nullptr};
  if (base) {
    pl.base = base; pl.stats = (double*)base; pl.stats_bytes = stats_bytes;
    PlanBuilder pb{core, &pl, &bb, &sb};
    if (pb.build_rew_end(h->blocks, h->downs, h->conv_in, &h->feat)) return 1;
  } else bb.off = b0.off;
  const int D = h->cfg.lstm_dim;
  h->x_gates = (float*)bb.take((size_t)B * 4 * D * 4);
  h->y = (float*)bb.take((size_t)B * D * 4); h->hid = (float*)bb.take((size_t)B * D * 4);
  h->logits_tm = (float*)bb.take((size_t)B * 5 * 4);
  h->hc[0] = (float*)bb.take((size_t)B * D * 4); h->hc[1] = (float*)bb.take((size_t)B * D * 4);
  if (total) *total = stats_bytes + bb.off + 512;
  return 0;
}

}  // namespace

extern "C" dmd_rew_end* dmd_rew_end_create(const dmd_rew_end_config* cfg) {
  if (!cfg || cfg->num_levels < 1 || cfg->num_levels >= DMD_MAX_LEVELS) { fail("rew_end_create: bad config"); return nullptr; }
  if (cfg->cond_channels % 32 || cfg->cond_channels > 256) { fail("rew_end_create: cond_channels must be a multiple of 32, <= 256"); return nullptr; }
  for (int i = 0; i < cfg->num_levels; ++i)
    if (cfg->channels[i] % 32 || cfg->channels[i] > 64) { fail("rew_end_create: channels must be 32 or 64 per level (got %d)", cfg->channels[i]); return nullptr; }
  if (cfg->lstm_dim % 4) { fail("rew_end_create: lstm_dim must be a multiple of 4"); return nullptr; }
  if (init_kernels()) return nullptr;
  dmd_rew_end* h = new dmd_rew_end();
  h->cfg = *cfg;
  dmd_denoiser* core = &h->core;
  memset(&core->cfg, 0, sizeof(core->cfg));
  core->cfg.img_channels = cfg->img_channels; core->cfg.num_steps_conditioning = 1; core->cfg.cond_channels = cfg->cond_channels;
  core->cfg.num_levels = cfg->num_levels; core->cfg.num_actions = cfg->num_actions;
  for (int i = 0; i < cfg->num_levels; ++i) { core->cfg.depths[i] = cfg->depths[i]; core->cfg.channels[i] = cfg->channels[i]; core->cfg.attn_depths[i] = cfg->attn_depths[i]; }
  // registration order (rew_end_model.py:27-41, :93-125): encoder.{conv_in, blocks[0..L], downsamples[1..L-1]}, act_emb, lstm, head
  Walker w{core};
  core->numel.clear();
  const int L = cfg->num_levels;
  const int cin_real = 2 * cfg->img_channels;
  h->conv_in = w.conv(cfg->channels[0], cin_real, 9, cin_real, round_up(cin_real, 16), 0, 1, false);
  h->blocks.resize(L + 1);
  for (int i = 0; i < L; ++i) {
    const int c1 = cfg->channels[i > 0 ? i - 1 : 0], c2 = cfg->channels[i];
    for (int k = 0; k < cfg->depths[i]; ++k) h->blocks[i].push_back(w.resblock(k == 0 ? c1 : c2, 0, c2, cfg->attn_depths[i] != 0));
  }
  for (int k = 0; k < 2; ++k) h->blocks[L].push_back(w.resblock(cfg->channels[L - 1], 0, cfg->channels[L - 1], true));
  h->downs.resize(L);
  for (int i = 1; i < L; ++i) h->downs[i] = w.conv(cfg->channels[i - 1], cfg->channels[i - 1], 9, cfg->channels[i - 1], cfg->channels[i - 1], 0);
  const int S = cfg->img_size >> (L - 1);
  h->feat_c = cfg->channels[L - 1]; h->feat_hw = S * S;
  const long long D = cfg->lstm_dim, K = (long long)h->feat_c * h->feat_hw;
  h->i_actemb = w.next((long long)cfg->num_actions * cfg->cond_channels);
  h->i_wih = w.next(4 * D * K); h->i_whh = w.next(4 * D * D); h->i_bih = w.next(4 * D); h->i_bhh = w.next(4 * D);
  h->i_h0w = w.next(D * D); h->i_h0b = w.next(D); h->i_h2w = w.next(5 * D);
  core->n_tensors = w.idx;
  core->goff.assign(core->n_tensors, 0);
  core->grad_total = 0;
  for (int i = 0; i < core->n_tensors; ++i) { core->goff[i] = core->grad_total; core->grad_total += (core->numel[i] + 3) & ~3ll; }  // 16-byte aligned slices
  size_t pk = w.pk;
  auto split_copy = [&](ConvW c) {
    c.precise = 1; c.trs = 0; c.pk_off = pk;
    pk += (size_t)c.taps * c.Cin * c.CoutPad * 2 * 3; pk = (pk + 255) & ~(size_t)255;
    return c;
  };
  h->tblocks = h->blocks;
  for (auto& lv : h->tblocks) for (auto& r : lv) { r.c1 = split_copy(r.c1); r.c2 = split_copy(r.c2); }
  h->tdowns = h->downs;
  for (int i = 1; i < L; ++i) h->tdowns[i] = split_copy(h->downs[i]);
  h->enc = EncoderDef{&h->tblocks, &h->tdowns, &h->conv_in, h->i_actemb};
  core->film_w_off = pk; pk += (size_t)core->film_rows * cfg->cond_channels * 4; pk = (pk + 255) & ~(size_t)255;
  core->film_b_off = pk; pk += (size_t)core->film_rows * 4; pk = (pk + 255) & ~(size_t)255;
  core->packed_bytes = pk;
  return h;
}
extern "C" void dmd_rew_end_destroy(dmd_rew_end* h) { delete h; }
extern "C" int dmd_rew_end_num_tensors(const dmd_rew_end* h) { return h->core.n_tensors; }
extern "C" size_t dmd_rew_end_packed_bytes(const dmd_rew_end* h) { return h->core.packed_bytes; }

extern "C" int dmd_rew_end_set_weights(dmd_rew_end* h, const float* const* ptrs_host, int n_ptrs, void* packed, void* stream) {
  DMD_CHECK(h && ptrs_host && packed, "rew_end set_weights: null argument");
  dmd_denoiser* core = &h->core;
  DMD_CHECK(n_ptrs == core->n_tensors, "rew_end set_weights: expected %d tensors (RewEndModel.state_dict order), got %d", core->n_tensors, n_ptrs);
  cudaStream_t st = (cudaStream_t)stream;
  // training plans bake parameter and packed-weight addresses in: drop them when these move
  const bool moved = core->packed != (uint8_t*)packed || core->ptrs.empty() || memcmp(core->ptrs.data(), ptrs_host, sizeof(float*) * n_ptrs) != 0;
  if (moved) core->tplans.clear();
  core->ptrs.assign(ptrs_host, ptrs_host + n_ptrs);
  core->packed = (uint8_t*)packed;
  h->planB = 0;
  if (pack_one(core, h->conv_in, st)) return 1;
  for (auto& lv : h->blocks) for (auto& r : lv) if (pack_rb(core, r, st)) return 1;
  for (int i = 1; i < h->cfg.num_levels; ++i) if (pack_one(core, h->downs[i], st)) return 1;
  auto pack_split = [&](const ConvW& c) {   // the training copies' forward packs (their backward-data packs are the ones above)
    return dmd_pack_conv_weight(core->ptrs[c.w_idx], core->packed + c.pk_off, c.Cout, c.CoutPad, c.CinReal, c.Cin, c.taps, c.c0_real, c.c0_store, 1, st);
  };
  for (auto& lv : h->tblocks) for (auto& r : lv) if (pack_split(r.c1) || pack_split(r.c2)) return 1;
  for (int i = 1; i < h->cfg.num_levels; ++i) if (pack_split(h->tdowns[i])) return 1;
  return 0;
}

extern "C" size_t dmd_rew_end_workspace_bytes(dmd_rew_end* h, int rows) {
  size_t total = 0;
  h->planB = 0;
  if (rew_end_layout(h, rows, h->cfg.img_size, h->cfg.img_size, nullptr, &total)) return 0;
  return total;
}

// obs / next_obs (b, t, C, S, S) fp32, act (b, t) int64, hx_in / cx_in (b, lstm_dim) or NULL (zeros).
// Outputs: logits_rew (b, t, 3), logits_end (b, t, 2), hx_out / cx_out (b, lstm_dim).
extern "C" int dmd_rew_end_predict(dmd_rew_end* h, int b, int t, const float* obs, const float* next_obs, const int64_t* act,
                                   const float* hx_in, const float* cx_in, float* logits_rew, float* logits_end, float* hx_out,
                                   float* cx_out, void* workspace, size_t workspace_bytes, void* stream) {
  DMD_CHECK(h && obs && next_obs && act && logits_rew && logits_end && hx_out && cx_out && workspace, "rew_end predict: null argument");
  dmd_denoiser* core = &h->core;
  DMD_CHECK(!core->ptrs.empty() && core->packed, "rew_end predict: call dmd_rew_end_set_weights first");
  DMD_CHECK(((uintptr_t)workspace & 255) == 0, "rew_end predict: workspace must be 256-byte aligned");
  const dmd_rew_end_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = b * t, S = c.img_size, HW = S * S, D = c.lstm_dim, CC = c.cond_channels;
  if (h->planB != rows || h->plan_ws != workspace) {
    size_t need = 0;
    h->planB = 0;
    if (rew_end_layout(h, rows, S, S, nullptr, &need)) return 1;
    DMD_CHECK(workspace_bytes >= need, "rew_end predict: workspace too small (%zu < %zu)", workspace_bytes, need);
    if (rew_end_layout(h, rows, S, S, (uint8_t*)workspace, nullptr)) return 1;
    h->planB = rows; h->plan_ws = workspace;
  }
  Plan& pl = core->plan;
  DMD_CUDA(cudaMemsetAsync(pl.stats, 0, pl.stats_bytes, st));
  pack_rew_end_input_kernel<<<dim3((HW + 255) / 256, rows), 256, 0, st>>>(obs, next_obs, act, core->ptrs[h->i_actemb], pl.xin, pl.cond, b, t,
                                                                          c.img_channels, pl.CP_in, HW, CC, c.num_actions);
  DMD_LAUNCH_OK();
  if (linear_launch(pl.cond, (const float*)(core->packed + core->film_w_off), (const float*)(core->packed + core->film_b_off), pl.film,
                    rows, CC, core->film_rows, 0, st)) return 1;
  if (run_encoder_ops(pl, st)) return 1;
  // LSTM over time (torch.nn.LSTM, gate order i f g o), rows of step k are the contiguous block [k*b, (k+1)*b)
  const int K = h->feat_c * h->feat_hw;
  const float* hprev = hx_in; const float* cprev = cx_in;
  if (!hx_in) { DMD_CUDA(cudaMemsetAsync(h->hc[0], 0, (size_t)b * D * 4, st)); hprev = h->hc[0]; }
  if (!cx_in) { DMD_CUDA(cudaMemsetAsync(h->hc[1], 0, (size_t)b * D * 4, st)); cprev = h->hc[1]; }
  for (int k = 0; k < t; ++k) {
    const float* xk = h->feat.data + (size_t)k * b * K;
    if (linear_launch(xk, core->ptrs[h->i_wih], core->ptrs[h->i_bih], h->x_gates, b, K, 4 * D, 0, st, 0, h->feat_hw)) return 1;
    if (linear_launch(hprev, core->ptrs[h->i_whh], core->ptrs[h->i_bhh], h->x_gates, b, D, 4 * D, 0, st, 1, 0)) return 1;
    float* hk = h->y + (size_t)k * b * D;   // y rows of step k (time-major); also the next step's h
    lstm_gates_kernel<<<(b * D + 255) / 256, 256, 0, st>>>(h->x_gates, cprev, hk, cx_out, b, D);
    DMD_LAUNCH_OK();
    hprev = hk; cprev = cx_out;
  }
  DMD_CUDA(cudaMemcpyAsync(hx_out, hprev, (size_t)b * D * 4, cudaMemcpyDeviceToDevice, st));
  // head: Linear(D, D) + SiLU + Linear(D, 5, bias=False) over all (t b) rows
  if (linear_launch(h->y, core->ptrs[h->i_h0w], core->ptrs[h->i_h0b], h->hid, rows, D, D, 1, st)) return 1;
  if (linear_launch(h->hid, core->ptrs[h->i_h2w], nullptr, h->logits_tm, rows, D, 5, 0, st)) return 1;
  split_logits_kernel<<<(rows + 127) / 128, 128, 0, st>>>(h->logits_tm, logits_rew, logits_end, b, t);
  DMD_LAUNCH_OK();
  return 0;
}

// ---------------------------------------------------------------------------------------------- reward / termination training
// RewEndModel.forward under autograd (rew_end_model.py:57-90, trainer.py:349-388).  dmd_rew_end_forward_train runs the
// encoder on a training plan of its own (core.tplans: a later predict_rew_end keeps its inference plan) and keeps every
// activation: the encoder tape, all t steps of LSTM gates and cell states, and the head input.  dmd_rew_end_backward
// then runs the head backward, BPTT through the LSTM (fp32), and the encoder backward under one power-of-two loss scale.
// Workspace = [encoder training plan][RewEndTrain buffers below]; rows are time-major (r = k * b + n).
namespace {

struct RewEndTrain {
  int64_t* act_tm; float *gates, *cells, *y, *hid, *logits_tm, *zeros;                 // forward
  float *g_logits, *hpre, *g_pre, *g_hid, *g_y, *dgates, *g_c[2], *x_flat, *g_xflat;     // backward
  size_t bytes;
};

void rew_end_train_layout(const dmd_rew_end* h, int b, int t, uint8_t* base, RewEndTrain* o) {
  Bump bb{base};
  const size_t rows = (size_t)b * t, D = h->cfg.lstm_dim, K = (size_t)h->feat_c * h->feat_hw;
  o->act_tm = (int64_t*)bb.take(rows * 8);
  o->gates = (float*)bb.take(rows * 4 * D * 4); o->cells = (float*)bb.take(rows * D * 4);
  o->y = (float*)bb.take(rows * D * 4); o->hid = (float*)bb.take(rows * D * 4);
  o->logits_tm = (float*)bb.take(rows * 5 * 4); o->zeros = (float*)bb.take((size_t)b * D * 4);
  o->g_logits = (float*)bb.take(rows * 5 * 4);
  o->hpre = (float*)bb.take(rows * D * 4); o->g_pre = (float*)bb.take(rows * D * 4);
  o->g_hid = (float*)bb.take(rows * D * 4); o->g_y = (float*)bb.take(rows * D * 4);
  o->dgates = (float*)bb.take(rows * 4 * D * 4);
  o->g_c[0] = (float*)bb.take((size_t)b * D * 4); o->g_c[1] = (float*)bb.take((size_t)b * D * 4);
  o->x_flat = (float*)bb.take(rows * K * 4); o->g_xflat = (float*)bb.take(rows * K * 4);
  o->bytes = bb.off + 256;
}

// bytes of the encoder training plan (its buffers start the workspace); 0 with dmd_last_error set when it cannot be built
size_t rew_end_plan_bytes(dmd_rew_end* h, int rows) {
  Plan tmp; size_t need = 0;
  const int S = h->cfg.img_size;
  if (make_train_plan(&h->core, &tmp, rows, S, S, nullptr, &need, &h->enc)) return 0;
  return (need + 255) & ~(size_t)255;
}

int rew_end_check_bt(int b, int t, const char* who) {
  DMD_CHECK(b > 0 && t > 0, "%s: b and t must be positive (got b=%d t=%d)", who, b, t);
  DMD_CHECK((long long)b * t < (1ll << 24), "%s: b * t = %lld rows is too many", who, (long long)b * t);
  return 0;
}

}  // namespace

extern "C" size_t dmd_rew_end_train_workspace_bytes(dmd_rew_end* h, int b, int t) {
  if (!h) { fail("rew_end train_workspace_bytes: null handle"); return 0; }
  if (rew_end_check_bt(b, t, "rew_end train_workspace_bytes")) return 0;
  const size_t plan = rew_end_plan_bytes(h, b * t);
  if (!plan) return 0;
  RewEndTrain r; rew_end_train_layout(h, b, t, nullptr, &r);
  return plan + r.bytes;
}

extern "C" long long dmd_rew_end_grad_layout(const dmd_rew_end* h, long long* offsets, long long* numels, int n) {
  if (!h || n != h->core.n_tensors) { fail("rew_end grad_layout: expected %d entries", h ? h->core.n_tensors : 0); return -1; }
  for (int i = 0; i < n; ++i) { if (offsets) offsets[i] = h->core.goff[i]; if (numels) numels[i] = h->core.numel[i]; }
  return h->core.grad_total;
}

extern "C" int dmd_rew_end_forward_train(dmd_rew_end* h, int b, int t, const float* obs, const float* next_obs, const int64_t* act,
                                         float* logits_rew, float* logits_end, void* workspace, size_t workspace_bytes, void* stream) {
  DMD_CHECK(h && obs && next_obs && act && logits_rew && logits_end && workspace, "rew_end forward_train: null argument");
  if (rew_end_check_bt(b, t, "rew_end forward_train")) return 1;
  dmd_denoiser* core = &h->core;
  DMD_CHECK(!core->ptrs.empty() && core->packed, "rew_end forward_train: call dmd_rew_end_set_weights first");
  DMD_CHECK(((uintptr_t)workspace & 255) == 0, "rew_end forward_train: workspace must be 256-byte aligned");
  const dmd_rew_end_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = b * t, S = c.img_size, HW = S * S, D = c.lstm_dim, CC = c.cond_channels, K = h->feat_c * h->feat_hw;
  const size_t plan_bytes = rew_end_plan_bytes(h, rows);
  if (!plan_bytes) return 1;
  RewEndTrain r; rew_end_train_layout(h, b, t, nullptr, &r);
  DMD_CHECK(workspace_bytes >= plan_bytes + r.bytes, "rew_end forward_train: workspace too small (%zu < %zu)", workspace_bytes, plan_bytes + r.bytes);
  Plan* pl = nullptr;
  if (ensure_train_plan(core, rows, S, S, workspace, plan_bytes, st, &pl, &h->enc)) return 1;
  rew_end_train_layout(h, b, t, (uint8_t*)workspace + plan_bytes, &r);
  pl->seq_b = 0; pl->seq_t = 0;   // set again once the forward has been issued
  pl->t_act = r.act_tm;
  DMD_CUDA(cudaMemsetAsync(pl->stats, 0, pl->stats_bytes, st));
  pack_rew_end_input_kernel<<<dim3((HW + 255) / 256, rows), 256, 0, st>>>(obs, next_obs, act, core->ptrs[h->i_actemb], pl->xin, pl->cond, b, t,
                                                                          c.img_channels, pl->CP_in, HW, CC, c.num_actions, r.act_tm);
  DMD_LAUNCH_OK();
  if (linear_launch(pl->cond, (const float*)(core->packed + core->film_w_off), (const float*)(core->packed + core->film_b_off), pl->film,
                    rows, CC, core->film_rows, 0, st)) return 1;
  if (run_encoder_ops(*pl, st)) return 1;
  // LSTM from a zero state (rew_end_model.py:53); the input projection of all t steps at once, then the recurrence.  Gates
  // (pre-activations) and cell states of every step stay for the backward.
  if (linear_launch(pl->enc_out.data, core->ptrs[h->i_wih], core->ptrs[h->i_bih], r.gates, rows, K, 4 * D, 0, st, 0, h->feat_hw)) return 1;
  DMD_CUDA(cudaMemsetAsync(r.zeros, 0, (size_t)b * D * 4, st));
  for (int k = 0; k < t; ++k) {
    float* gk = r.gates + (size_t)k * b * 4 * D;
    const float* hprev = k ? r.y + (size_t)(k - 1) * b * D : r.zeros;
    const float* cprev = k ? r.cells + (size_t)(k - 1) * b * D : r.zeros;
    if (linear_launch(hprev, core->ptrs[h->i_whh], core->ptrs[h->i_bhh], gk, b, D, 4 * D, 0, st, 1, 0)) return 1;
    lstm_gates_kernel<<<(b * D + 255) / 256, 256, 0, st>>>(gk, cprev, r.y + (size_t)k * b * D, r.cells + (size_t)k * b * D, b, D);
    DMD_LAUNCH_OK();
  }
  if (linear_launch(r.y, core->ptrs[h->i_h0w], core->ptrs[h->i_h0b], r.hid, rows, D, D, 1, st)) return 1;
  if (linear_launch(r.hid, core->ptrs[h->i_h2w], nullptr, r.logits_tm, rows, D, 5, 0, st)) return 1;
  split_logits_kernel<<<(rows + 127) / 128, 128, 0, st>>>(r.logits_tm, logits_rew, logits_end, b, t);
  DMD_LAUNCH_OK();
  pl->seq_b = b; pl->seq_t = t;
  return 0;
}

// g_logits_rew (b, t, 3), g_logits_end (b, t, 2): dL/dlogits.  Writes (assigns) every parameter gradient into `grads`.
extern "C" int dmd_rew_end_backward(dmd_rew_end* h, int b, int t, const float* g_logits_rew, const float* g_logits_end, float* grads,
                                    long long grads_numel, void* workspace, void* stream) {
  DMD_CHECK(h && g_logits_rew && g_logits_end && grads && workspace, "rew_end backward: null argument");
  if (rew_end_check_bt(b, t, "rew_end backward")) return 1;
  dmd_denoiser* core = &h->core;
  const int rows = b * t, S = h->cfg.img_size, D = h->cfg.lstm_dim, K = h->feat_c * h->feat_hw;
  Plan* plp = find_train_plan(core, rows, S, S, workspace);
  DMD_CHECK(plp && plp->train && plp->seq_b == b && plp->seq_t == t,
            "rew_end backward: no matching dmd_rew_end_forward_train on this workspace (b=%d t=%d)", b, t);
  Plan& pl = *plp;
  DMD_CHECK(grads_numel >= core->grad_total, "rew_end backward: gradient buffer too small (%lld < %lld floats)", grads_numel, core->grad_total);
  DMD_CHECK(((uintptr_t)grads & 15) == 0, "rew_end backward: gradient buffer must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  RewEndTrain r; rew_end_train_layout(h, b, t, (uint8_t*)workspace + rew_end_plan_bytes(h, rows), &r);
  auto G = [&](int idx) { return grads + core->goff[idx]; };
  auto W = [&](int idx) { return core->ptrs[idx]; };
  // C (+)= A B with A(m, k) = A[m * sam + k * sak], B(k, n) = B[k * sbk + n * sbn]  (fp32)
  auto sgemm = [&](const float* A, long long sam, long long sak, const float* Bm, long long sbk, long long sbn, float* C, long long ldc,
                   int M, int N, int Kd, int acc) -> int {
    sgemm_kernel<<<dim3((N + 63) / 64, (M + 63) / 64), 256, 0, st>>>(A, sam, sak, Bm, sbk, sbn, C, ldc, M, N, Kd, nullptr, acc);
    DMD_LAUNCH_OK();
    return 0;
  };
  auto colsum = [&](const float* x, long long nrows, int C, float* out, float* out2) -> int {
    const int L4 = (C < 256 ? C : 256) >> 2, lanes = 256 / L4;
    long long blocks = (nrows + (long long)lanes * 8 - 1) / ((long long)lanes * 8);
    blocks = blocks > 592 ? 592 : (blocks < 1 ? 1 : blocks);
    colsum_kernel<<<dim3((unsigned)blocks, (C + 255) / 256), 256, 0, st>>>(x, out, out2, nullptr, nrows, C, C);
    DMD_LAUNCH_OK();
    return 0;
  };
  DMD_CUDA(cudaMemsetAsync(grads, 0, (size_t)core->grad_total * 4, st));
  DMD_CUDA(cudaMemsetAsync(pl.zero_begin, 0, pl.zero_bytes, st));
  // ---- head: logits = silu(y W0^T + b0) W2^T  (rew_end_model.py:35-39)
  merge_logits_grad_kernel<<<(rows + 127) / 128, 128, 0, st>>>(g_logits_rew, g_logits_end, r.g_logits, b, t);
  DMD_LAUNCH_OK();
  if (sgemm(r.g_logits, 1, 5, r.hid, D, 1, G(h->i_h2w), D, 5, D, rows, 1)) return 1;                 // dW2 = g^T hid
  if (sgemm(r.g_logits, 5, 1, W(h->i_h2w), D, 1, r.g_hid, D, rows, D, 5, 0)) return 1;               // g_hid = g W2
  if (linear_launch(r.y, W(h->i_h0w), W(h->i_h0b), r.hpre, rows, D, D, 0, st)) return 1;             // pre-activation again
  dsilu_mul_kernel<<<(unsigned)(((long long)rows * D + 255) / 256), 256, 0, st>>>(r.hpre, r.g_hid, r.g_pre, (long long)rows * D);
  DMD_LAUNCH_OK();
  if (sgemm(r.g_pre, 1, D, r.y, D, 1, G(h->i_h0w), D, D, D, rows, 1)) return 1;                      // dW0 = g_pre^T y
  if (colsum(r.g_pre, rows, D, G(h->i_h0b), nullptr)) return 1;
  if (sgemm(r.g_pre, D, 1, W(h->i_h0w), D, 1, r.g_y, D, rows, D, D, 0)) return 1;                    // g_y = g_pre W0
  // ---- LSTM, backward through time: g_h(k) = g_y(k) + dgates(k+1) W_hh ; g_c carried in two ping-pong buffers
  for (int k = t - 1, cur = 0; k >= 0; --k, cur ^= 1) {
    float* gyk = r.g_y + (size_t)k * b * D;
    if (k + 1 < t && sgemm(r.dgates + (size_t)(k + 1) * b * 4 * D, 4 * D, 1, W(h->i_whh), D, 1, gyk, D, b, D, 4 * D, 1)) return 1;
    const float* cprev = k ? r.cells + (size_t)(k - 1) * b * D : r.zeros;
    lstm_cell_bwd_kernel<<<(b * D + 255) / 256, 256, 0, st>>>(r.gates + (size_t)k * b * 4 * D, cprev, gyk, k + 1 < t ? r.g_c[cur] : nullptr,
                                                             r.dgates + (size_t)k * b * 4 * D, r.g_c[cur ^ 1], b, D);
    DMD_LAUNCH_OK();
  }
  // parameter gradients of all steps at once; x is the NCHW flatten of the encoder output (rew_end_model.py:52)
  if (dmd_nhwc_to_nchw(pl.enc_out.data, r.x_flat, rows, h->feat_c, h->feat_c, h->feat_hw, st)) return 1;
  if (sgemm(r.dgates, 1, 4 * D, r.x_flat, K, 1, G(h->i_wih), K, 4 * D, K, rows, 1)) return 1;                   // dW_ih = dgates^T x
  if (t > 1 && sgemm(r.dgates + (size_t)b * 4 * D, 1, 4 * D, r.y, D, 1, G(h->i_whh), D, 4 * D, D, rows - b, 1)) return 1;   // dW_hh = sum_k dgates(k)^T h(k-1)
  if (colsum(r.dgates, rows, 4 * D, G(h->i_bih), G(h->i_bhh))) return 1;
  if (sgemm(r.dgates, 4 * D, 1, W(h->i_wih), K, 1, r.g_xflat, K, rows, K, 4 * D, 0)) return 1;                  // g_x = dgates W_ih
  // ---- encoder: the feature gradient (NHWC) enters the fp16 tensor-core backward under a power-of-two loss scale
  float* gfeat = pl.enc_out.grad;
  if (dmd_nchw_to_nhwc(r.g_xflat, gfeat, rows, h->feat_c, h->feat_c, h->feat_hw, st)) return 1;
  const long long n = (long long)rows * K;
  absmax_kernel<<<(int)std::min<long long>((n + 255) / 256, 1184), 256, 0, st>>>(gfeat, pl.amax, n);
  DMD_LAUNCH_OK();
  loss_scale_kernel<<<1, 1, 0, st>>>(pl.amax, pl.scale);
  DMD_LAUNCH_OK();
  scale_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(gfeat, pl.scale, n);
  DMD_LAUNCH_OK();
  return run_bops(core, pl, grads, st);
}
