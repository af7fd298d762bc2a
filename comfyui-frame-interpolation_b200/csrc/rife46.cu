// Context, weight repacking, the RIFE-4.6 forward schedule and the C ABI (include/vfi_b200.h).
//
// Forward schedule of one internal pass over B (pair, timestep) tasks - reference IFNet.forward,
// rife_arch.py:465-732, arch "4.6" (blocks (7,192) (12,128) (12,96) (12,64), rife_arch.py:404-408):
//   prep_frames (once per source frame)                       clamp / pad           :476-485
//   for block i, scale s_i:                                                          :519-704
//     front      -> x      [B, Hs/2, Ws/2, 4*16]  16-bit      warp+concat+1/s       :31-70,:238-249,:589-596
//     tapconv    -> c00    [B, Hs/4, Ws/4, 4*c/2] 16-bit      conv0.0 (+lrelu)      :181-184
//     tapconv    -> feat   [B, Hs/4, Ws/4, c]     16-bit      conv0.1 (+lrelu)
//     8x tapconv -> feat                                       ResConv               :20-28
//     tapconv    -> tmp    [B, Hs, Ws] float4 + float          ConvT+PixelShuffle    :215-218
//     (flow(p) = F(p) + sum_j up(T_j)(p)*s_j: F is stored only by fronts that visit every pixel)  :263-266,:694-696
//   final        -> out [B, H, W, 3] fp32                      warp, sigmoid blend, crop, clamp :703-717,:732
#include <cuda_fp16.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <mutex>
#include <thread>

#include "../../include/vfi_b200.h"
#include "vfi_internal.h"
#include "hoststage.h"

namespace vfi {

static thread_local std::string g_err;
void set_error(const std::string& s) { g_err = s; }

namespace {

const int kBlockC[kMaxBlocks] = {192, 128, 96, 64, 32};  // (the fifth block exists in arch 4.26 only)
const int kBlockCinReal[4] = {7, 12, 12, 12};        // arch 4.6: img0,img1,t | w0,w1,t,mask + flow
const int kBlockCinReal47[4] = {15, 20, 20, 20};     // arch 4.7: + encoded features f0,f1 (4 ch each)
const int kBlockCinReal417[4] = {23, 28, 28, 28};    // arch 4.17: + Head_417 features f0,f1 (8 ch each)
const int kBlockCinReal426[kMaxBlocks] = {15, 28, 28, 28, 28};  // arch 4.26: f0,f1 (4 each) [+ mask, 8 fed-back features, flow]
inline int num_blocks(int arch) { return arch == 426 ? 5 : 4; }

uint16_t to_operand(float v, int op_type) {
  if (op_type == OP_BF16) {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    uint16_t u;
    std::memcpy(&u, &h, 2);
    return u;
  }
  __half h = __float2half_rn(v);
  uint16_t u;
  std::memcpy(&u, &h, 2);
  return u;
}

// Packed weights = the SWIZZLE_128B K-major UMMA B operand, bit for bit: [split][K16/4 (padded)][n][128-byte row of
// four K=16 steps], 16-byte chunks XOR-swizzled with (n & 7); bulk-copied to shared memory verbatim.
template <class F>
std::vector<uint16_t> pack_weights(const TapConvLayer& L, int op_type, F wfun) {
  const size_t per_split = (size_t)((L.ktotal16 + 3) / 4) * L.n_cta * 64;
  std::vector<uint16_t> v((size_t)L.nsplit * per_split, 0);
  for (int sp = 0; sp < L.nsplit; ++sp) {
    int j = 0;
    for (int e = 0; e < L.ntaps; ++e)
      for (int i = 0; i < L.taps[e].nk16; ++i, ++j)
        for (int c = 0; c < 16; ++c) {
          const int chunk = (j & 3) * 2 + (c >> 3);
          for (int nl = 0; nl < L.n_cta; ++nl) {
            const float val = wfun(e, i * 16 + c, sp * L.n_cta + nl);
            v[sp * per_split + ((size_t)(j >> 2) * L.n_cta + nl) * 64 + (size_t)((chunk ^ (nl & 7)) * 8 + (c & 7))] =
                to_operand(val, op_type);
          }
        }
  }
  return v;
}

// choose the output-channel split: smallest split reaching `want_stages`, else the one with most stages
void choose_split(TapConvLayer& L, const std::vector<int>& splits, int want_stages) {
  int best_split = -1, best_stages = 0;
  for (int sp : splits) {
    if (L.n_total % sp) continue;
    const int nc = L.n_total / sp;
    if (nc % 16) continue;
    L.nsplit = sp;
    L.n_cta = nc;
    TapConvParams p{};
    const int st = tapconv_plan(L, &p);
    if (st >= want_stages) {
      best_split = sp;
      best_stages = st;
      break;
    }
    if (st > best_stages) {
      best_stages = st;
      best_split = sp;
    }
  }
  L.nsplit = best_split;
  L.n_cta = L.n_total / best_split;
}

// CTA-pair form (tapconv.cu, cta_group::2): pair-split s covers n_epi = n_total / psp output channels, each CTA of the
// pair holding half of them as its B rows (packed slices 2s and 2s+1).  Returns false when no split reaches
// `want_stages` (the caller then keeps the single-CTA plan).  VFI_PAIR=0 switches the form off (A/B runs).
bool choose_split_pair(TapConvLayer& L, const std::vector<int>& psplits, int want_stages) {
  static const bool on = [] {
    const char* e = std::getenv("VFI_PAIR");
    return !(e && e[0] == '0');
  }();
  if (!on) return false;
  const TapConvLayer keep = L;
  for (int psp : psplits) {
    if (L.n_total % (2 * psp)) continue;
    const int n_epi = L.n_total / psp;
    if ((n_epi & 15) || n_epi > 128) continue;
    L.pair = 1;
    L.nsplit = 2 * psp;
    L.n_cta = n_epi / 2;
    TapConvParams p{};
    if (tapconv_plan(L, &p) >= want_stages) return true;
  }
  L = keep;
  return false;
}

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

}  // namespace
}  // namespace vfi

using namespace vfi;

struct vfi_ctx {
  int device = 0;
  int num_sms = 148;
  int batch = 8;
  int op_type = OP_F16;
  bool loaded = false;
  int64_t launches = 0;
  TapConvLayer layers[kMaxBlocks][12];  // [block][0=conv0.0, 1=conv0.1, 2..9=ResConv, 10=lastconv (flow + mask),
                                        //          11 = arch 4.26: the 8 feature channels of lastconv]
  std::vector<void*> weight_allocs;
  // workspace
  DevBuf imgs, imgs_h, flow, mask, x, c00, featA, featB, tF[kMaxBlocks], tM[kMaxBlocks], raw, outdev;
  DevBuf tE[kMaxBlocks];         // arch 4.26: block outputs' 8 feature channels [B, Hp/s, Wp/s, 8] 16-bit
  int arch = 46;                 // 46 | 47 (rife47.pth / rife49.pth)
  DevBuf feats, e16;             // arch 4.7: encoded features per source frame (float4), half-res temp
  float* enc[4] = {nullptr, nullptr, nullptr, nullptr};  // encode.0.weight/.bias, encode.1.weight/.bias (fp32)
  TapConvLayer head[3];          // arch 4.17 / 4.26: Head cnn1, cnn2 (+ LeakyReLU), cnn3 (ConvTranspose), 32 (padded) channels
  DevBuf hA, hB;                 // arch 4.17: half-resolution 32-channel scratch of the head (ping-pong)
  int ws_Hp = 0, ws_Wp = 0, ws_B = 0;
  FlowState last_fs{};
  int last_lo = 0;
  bool last_have_base = false;
  DevBuf dbgF, dbgM;
  cudaStream_t s_h2d = nullptr, s_comp = nullptr, s_d2h = nullptr;
  DevBuf ops_a, ops_b;           // scratch of the channel-last op kernels (splat, 9 x 9 volumes)
  cudaEvent_t ops_done = nullptr;  // recorded on the stream of the last call that used ops_a / ops_b (ops_scratch_acquire)
  vfi::PinnedBuf pin_in, pin_out;
  // per-kernel-group timing of the forward schedule (vfi_rife_profile): CUDA events recorded on the launching stream
  // around each group while `profile` is set; read (and summed per group id) by vfi_rife_profile_read
  bool profile = false;
  struct ProfSpan { int id; cudaEvent_t e0, e1; };
  std::vector<ProfSpan> prof_spans;  // pinned staging rings of the host-pointer path (pageable caller memory)
  vfi::FilmState* film = nullptr;  // FILM weights and workspace (film.cu)
  vfi::SepState* sep = nullptr;    // Sepconv weights and workspace (sepconv.cu)
};

namespace vfi {
CtxInfo ctx_info(::vfi_ctx* c) { return CtxInfo{c->device, c->num_sms, c->s_h2d, c->s_comp, c->s_d2h}; }
FilmState*& ctx_film(::vfi_ctx* c) { return c->film; }
SepState*& ctx_sep(::vfi_ctx* c) { return c->sep; }
void ctx_add_launches(::vfi_ctx* c, int n) { c->launches += n; }
}  // namespace vfi

namespace {

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      set_error(std::string(#call) + ": " + cudaGetErrorString(_e));                               \
      return VFI_E_CUDA;                                                                           \
    }                                                                                              \
  } while (0)

int fail(int code, const std::string& msg) {
  set_error(msg);
  return code;
}

void free_weights(vfi_ctx* c) {
  for (void* p : c->weight_allocs) cudaFree(p);
  c->weight_allocs.clear();
  c->loaded = false;
}

template <class T>
int upload(vfi_ctx* c, const std::vector<T>& h, void** dptr) {
  void* d = nullptr;
  CK(cudaMalloc(&d, h.size() * sizeof(T)));
  c->weight_allocs.push_back(d);
  CK(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dptr = d;
  return VFI_OK;
}

// stride-2 3x3 conv on a space-to-depth input: kernel row ky reads s2d row offset dy and sub-row a
void s2_map(int k, int* d, int* a) {
  if (k == 0) { *d = -1; *a = 1; } else { *d = 0; *a = k - 1; }
}

int build_conv_s2(vfi_ctx* c, TapConvLayer& L, int Cs, int creal, int cout, int out_s2d, const float* w,
                  const float* bias) {
  L = TapConvLayer{};
  L.cin = 4 * Cs;
  L.n_total = cout;
  L.ntaps = 9;
  L.ktotal16 = 9 * (Cs / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 1; L.halo_w = kTileW + 1;
  L.epi_mode = EPI_BIAS_LRELU;
  L.out_s2d = out_s2d;
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) {
      int dy, a, dx, b;
      s2_map(ky, &dy, &a);
      s2_map(kx, &dx, &b);
      TapEntry& t = L.taps[ky * 3 + kx];
      t.dy = (int16_t)dy; t.dx = (int16_t)dx;
      t.chunk0 = (int16_t)(((a * 2 + b) * Cs) / 8);
      t.nk16 = (int16_t)(Cs / 16);
    }
  choose_split(L, {1, 2, 3, 4, 6, 8, 12}, 2);
  auto wf = [&](int e, int ci, int n) -> float {
    if (ci >= creal) return 0.f;
    const int ky = e / 3, kx = e % 3;
    return w[(((size_t)n * creal + ci) * 3 + ky) * 3 + kx];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(bias, bias + cout);
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

// 3x3 taps over all `ch` input channels.  ring: k-block-major (kb, tap) entries of 64 channels each, the order the
// ring pipeline consumes the window in (tapconv.cu); the packed weights follow the same order.
void set_taps_3x3(TapConvLayer& L, int ch, bool ring) {
  L.ring = ring ? 1 : 0;
  const int nkb = ring ? ch / 64 : 1;
  L.ntaps = 9 * nkb;
  for (int kb = 0; kb < nkb; ++kb)
    for (int e = 0; e < 9; ++e) {
      TapEntry& t = L.taps[kb * 9 + e];
      t.dy = (int16_t)(e / 3 - 1);
      t.dx = (int16_t)(e % 3 - 1);
      t.chunk0 = (int16_t)(kb * 8);
      t.nk16 = (int16_t)(ring ? 4 : ch / 16);
    }
}

// Wide, deep layers (c = 128, 192): with the whole window staged per tile the resident weight slice leaves room for
// only n_cta = 16..32 output channels, and one tcgen05.mma costs ~80 cycles whatever its N (profiles/README.md), so
// the layer time is ~ 1/n_cta.  The ring pipeline stages one 64-channel k-block at a time, which frees shared
// memory for n_cta = 48 (c = 192) / 64 (c = 128).  VFI_RING=0 disables it (A/B runs).
bool want_ring(int ch) {
  static const bool on = [] {
    const char* e = std::getenv("VFI_RING");
    return !(e && e[0] == '0');
  }();
  return on && ch >= 128 && ch % 64 == 0;
}

int build_resconv(vfi_ctx* c, TapConvLayer& L, int ch, const float* beta, const float* w, const float* bias) {
  L = TapConvLayer{};
  L.cin = ch;
  L.n_total = ch;
  L.ntaps = 9;
  L.ktotal16 = 9 * (ch / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 2; L.halo_w = kTileW + 2;
  L.epi_mode = EPI_RESCONV;
  const bool ring = want_ring(ch);
  set_taps_3x3(L, ch, ring);
  // CTA pairs where they halve the output-channel splits (c >= 96).  Measured at the 1080p geometry, batch 8
  // (profiles/r02_b_layers_b8_{pair,nopair}.json): c = 96 60.4 -> 46.1 us, c = 128 33.8 -> 31.7, c = 192 29.7 -> 25.6; at
  // c = 64, where a single CTA already holds all 64 columns, the pair is SLOWER (82.9 -> 91.2 us: half of every MMA's B
  // operand then comes from the peer SM's shared memory), so the 64-channel layers stay single-CTA.
  if (!(ch >= 96 && choose_split_pair(L, {1, 2, 3, 4, 6}, ring ? 2 : 3)))
    choose_split(L, {1, 2, 3, 4, 6, 8, 12}, ring ? 2 : 3);
  // (conv(x) + b) * beta + x  ==  conv_{w*beta}(x) + b*beta + x : beta is folded into the packed weights (one 16-bit
  // rounding of w*beta instead of w) so the epilogue is a pure add
  auto wf = [&](int e, int ci, int n) -> float {  // e = kb * 9 + tap (kb = 0 unless ring), ci relative to the k-block
    const int tap = e % 9, cin = (e / 9) * 64 + ci;
    return w[(((size_t)n * ch + cin) * 3 + tap / 3) * 3 + tap % 3] * beta[n];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(ch);
  for (int i = 0; i < ch; ++i) sh[i] = bias[i] * beta[i];
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

// ConvTranspose2d(c, 24, 4, 2, 1) + PixelShuffle(2) as ONE 3x3 conv producing, per feature cell, the 4x4 sub-pixel
// patch of the 5 used channels: n = c5*16 + py*4 + px, (py,px) = (2a+i, 2b+j), convT channel oc = 4*c5 + 2i + j at
// convT position (2y+a, 2x+b); tap (dy,dx) uses transposed-kernel element ky = a+1-2dy, kx = b+1-2dx.
int build_lastconv(vfi_ctx* c, TapConvLayer& L, int ch, int cout, const float* wt, const float* bias) {
  L = TapConvLayer{};
  L.cin = ch;
  L.n_total = 80;
  L.ntaps = 9;
  L.ktotal16 = 9 * (ch / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 2; L.halo_w = kTileW + 2;
  L.epi_mode = EPI_LASTCONV;
  const bool ring = want_ring(ch);
  set_taps_3x3(L, ch, ring);
  // all 80 columns in one CTA pair (40 B rows each) only where single CTAs would need five splits (c = 192: 27.6 ->
  // 19.5 us); elsewhere the single-CTA form is as fast or faster (c = 64: 93.2 vs 111.6 us, same measurement as above)
  if (!(ch >= 192 && choose_split_pair(L, {1}, 2))) {
    choose_split(L, {1, 5}, 2);
    if (ring && L.nsplit != 1) {  // the ring only pays when it keeps all 80 columns in one CTA (c = 128)
      set_taps_3x3(L, ch, false);
      choose_split(L, {1, 5}, 2);
    }
  }
  auto oc_of = [](int n) {
    const int c5 = n >> 4, pos = n & 15, py = pos >> 2, px = pos & 3;
    return 4 * c5 + 2 * (py & 1) + (px & 1);
  };
  auto wf = [&](int e, int cr, int n) -> float {  // e = kb * 9 + tap, cr relative to the k-block
    const int tap = e % 9, ci = (e / 9) * 64 + cr;
    const int dy = tap / 3 - 1, dx = tap % 3 - 1;
    const int pos = n & 15, py = pos >> 2, px = pos & 3;
    const int ky = (py >> 1) + 1 - 2 * dy, kx = (px >> 1) + 1 - 2 * dx;
    if (ky < 0 || ky > 3 || kx < 0 || kx > 3) return 0.f;
    return wt[(((size_t)ci * cout + oc_of(n)) * 4 + ky) * 4 + kx];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(80);
  for (int n = 0; n < 80; ++n) sh[n] = bias[oc_of(n)];
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

// arch 4.26: channels 5..12 of ConvTranspose2d(c, 52, 4, 2, 1) + PixelShuffle(2) (rife_arch.py:230-233, :272) - the 8
// feature channels handed to the next block - as a second 3x3 tap conv over the same input: column
// n = (py*4 + px)*8 + f holds feature f at sub-pixel (py, px) of the cell's 4x4 patch, so 16 consecutive columns are
// two x-adjacent sub-pixels x 8 channels = 32 contiguous bytes of the [B, 4H, 4W, 8] output (out_s2d = 2).
int build_lastfeat(vfi_ctx* c, TapConvLayer& L, int ch, int cout, const float* wt, const float* bias) {
  L = TapConvLayer{};
  L.cin = ch;
  L.n_total = 128;
  L.ntaps = 9;
  L.ktotal16 = 9 * (ch / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 2; L.halo_w = kTileW + 2;
  L.epi_mode = EPI_BIAS;
  L.out_s2d = 2;
  const bool ring = want_ring(ch);
  set_taps_3x3(L, ch, ring);
  choose_split(L, {2, 4, 8}, 2);
  auto oc_of = [](int n) {
    const int f = n & 7, pos = n >> 3, py = pos >> 2, px = pos & 3;
    return 4 * (5 + f) + 2 * (py & 1) + (px & 1);
  };
  auto wf = [&](int e, int cr, int n) -> float {  // e = kb * 9 + tap, cr relative to the k-block
    const int tap = e % 9, ci = (e / 9) * 64 + cr;
    const int dy = tap / 3 - 1, dx = tap % 3 - 1;
    const int pos = n >> 3, py = pos >> 2, px = pos & 3;
    const int ky = (py >> 1) + 1 - 2 * dy, kx = (px >> 1) + 1 - 2 * dx;
    if (ky < 0 || ky > 3 || kx < 0 || kx > 3) return 0.f;
    return wt[(((size_t)ci * cout + oc_of(n)) * 4 + ky) * 4 + kx];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(128);
  for (int n = 0; n < 128; ++n) sh[n] = bias[oc_of(n)];
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

// Head_417.cnn1 / cnn2: plain 3x3 conv + LeakyReLU on a 32-channel half-resolution tensor (one 32-channel k-block).
// `creal` < ch: arch 4.26's 16-channel Head layers run zero-padded to 32 channels (the kernel's smallest k-block).
int build_conv3x3_lrelu(vfi_ctx* c, TapConvLayer& L, int ch, int creal, const float* w, const float* bias) {
  L = TapConvLayer{};
  L.cin = ch;
  L.n_total = ch;
  L.ktotal16 = 9 * (ch / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 2; L.halo_w = kTileW + 2;
  L.epi_mode = EPI_BIAS_LRELU;
  set_taps_3x3(L, ch, false);
  choose_split(L, {1}, 2);
  auto wf = [&](int e, int ci, int n) -> float {
    if (ci >= creal || n >= creal) return 0.f;
    return w[(((size_t)n * creal + ci) * 3 + e / 3) * 3 + e % 3];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(ch, 0.f);
  for (int i = 0; i < creal; ++i) sh[i] = bias[i];
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

// Head_417.cnn3 = ConvTranspose2d(ch, cout, 4, 2, 1), no activation, as ONE 3x3 conv producing the 2x2 sub-pixels of
// every input cell: n = (a*2 + b)*cout + oc at output position (2y+a, 2x+b); tap (dy,dx) uses transposed-kernel element
// ky = a+1-2dy, kx = b+1-2dx.  The NHWC output [Hh][Wh][4*cout] IS the space-to-depth form of the feature map.
int build_deconv_s2d(vfi_ctx* c, TapConvLayer& L, int ch, int creal, int cout, const float* wt, const float* bias) {
  L = TapConvLayer{};
  L.cin = ch;
  L.n_total = 4 * cout;
  L.ktotal16 = 9 * (ch / 16);
  L.halo_y0 = -1; L.halo_x0 = -1; L.halo_h = kTileH + 2; L.halo_w = kTileW + 2;
  L.epi_mode = EPI_BIAS;
  set_taps_3x3(L, ch, false);
  choose_split(L, {1}, 2);
  auto wf = [&](int e, int ci, int n) -> float {
    const int dy = e / 3 - 1, dx = e % 3 - 1;
    const int sub = n / cout, oc = n % cout, a = sub >> 1, b = sub & 1;
    const int ky = a + 1 - 2 * dy, kx = b + 1 - 2 * dx;
    if (ky < 0 || ky > 3 || kx < 0 || kx > 3 || ci >= creal) return 0.f;
    return wt[(((size_t)ci * cout + oc) * 4 + ky) * 4 + kx];
  };
  std::vector<uint16_t> pk = pack_weights(L, c->op_type, wf);
  std::vector<float> sh(4 * cout);
  for (int n = 0; n < 4 * cout; ++n) sh[n] = bias[n % cout];
  int r;
  if ((r = upload(c, pk, &L.w))) return r;
  if ((r = upload(c, sh, (void**)&L.shift))) return r;
  return VFI_OK;
}

struct Geometry {
  int Hp, Wp;
  int nb;  // blocks: 4, arch 4.26: 5
  int s[kMaxBlocks];  // block scale (>= 1); 1 for an up-scaled block
  int k[kMaxBlocks];  // 1, or the up-scaling factor 2 / 4 of a block whose scale is 1/k (node scale_factor 2 / 4)
};

int make_geometry(int arch, int H, int W, float scale_factor, Geometry* g) {
  g->Hp = ((H - 1) / 64 + 1) * 64;  // rife_arch.py:480-482
  g->Wp = ((W - 1) / 64 + 1) * 64;
  g->nb = num_blocks(arch);
  for (int i = 0; i < g->nb; ++i) {
    const float sf = (float)(1 << (g->nb - 1 - i)) / scale_factor;  // [8,4,2,1] or [16,8,4,2,1] / scale_factor, rife/__init__.py:156-160
    g->k[i] = 1;
    if (sf < 1.f) {  // a block that UP-scales its input by k = 1 / scale (scale_factor 2: last block, 4: last two)
      const int ki = (int)std::lround(1.f / sf);
      if (std::fabs(1.f / sf - (float)ki) > 1e-6f || (ki != 2 && ki != 4))
        return fail(VFI_E_INVALID, "scale_factor must be one of 0.25, 0.5, 1, 2, 4");
      g->k[i] = ki;
      g->s[i] = 1;
      continue;
    }
    const int si = (int)std::lround(sf);
    if (std::fabs(sf - (float)si) > 1e-6f || si < 1 || (si & (si - 1)))
      return fail(VFI_E_INVALID, "scale_factor must be one of 0.25, 0.5, 1, 2, 4");
    g->s[i] = si;
    if ((g->Hp / si) % 4 || (g->Wp / si) % 4 || g->Hp % si || g->Wp % si)
      return fail(VFI_E_INVALID,
                  "padded size / scale is not a multiple of 4: the reference fails with a shape mismatch for this "
                  "size and scale_factor as well");
  }
  return VFI_OK;
}

int ensure_workspace(vfi_ctx* c, const Geometry& g, int B, int n_frames_window) {
  size_t x = 0, c00 = 0, feat = 0;
  for (int i = 0; i < g.nb; ++i) {
    const size_t Hs = (size_t)g.Hp * g.k[i] / g.s[i], Ws = (size_t)g.Wp * g.k[i] / g.s[i];
    x = std::max(x, (size_t)B * (Hs / 2) * (Ws / 2) * (c->arch != 46 ? 128 : 64) * 2);
    c00 = std::max(c00, (size_t)B * (Hs / 4) * (Ws / 4) * 2 * kBlockC[i] * 2);
    feat = std::max(feat, (size_t)B * (Hs / 4) * (Ws / 4) * kBlockC[i] * 2);
    CK(c->tF[i].ensure((size_t)B * Hs * Ws * sizeof(float4)));  // block output T_i (flow increments at 1/s_i)
    CK(c->tM[i].ensure((size_t)B * Hs * Ws * sizeof(float)));
    if (c->arch == 426 && i + 1 < g.nb) CK(c->tE[i].ensure((size_t)B * Hs * Ws * 16));
  }
  const size_t px = (size_t)g.Hp * g.Wp;
  CK(c->imgs.ensure((size_t)n_frames_window * px * sizeof(float4)));
  CK(c->imgs_h.ensure((size_t)n_frames_window * px * sizeof(uint2)));
  if (c->arch == 47) {
    CK(c->feats.ensure((size_t)n_frames_window * px * sizeof(uint2)));  // half4 features
    CK(c->e16.ensure((size_t)(kMaxBatch + 2) * (px / 4) * 16 * sizeof(float)));
  }
  if (c->arch == 417 || c->arch == 426) {
    // features: 8 (4.26: 4) x 16-bit per pixel, space-to-depth cells of 32 (16) values; head scratch: 32 ch at 1/2 res
    CK(c->feats.ensure((size_t)n_frames_window * px * (c->arch == 417 ? 16 : 8)));
    CK(c->hA.ensure((size_t)(kMaxBatch + 2) * (px / 4) * 32 * 2));
    CK(c->hB.ensure((size_t)(kMaxBatch + 2) * (px / 4) * 32 * 2));
  }
  CK(c->flow.ensure((size_t)B * px * sizeof(float4)));
  CK(c->mask.ensure((size_t)B * px * sizeof(float)));
  CK(c->x.ensure(x));
  CK(c->c00.ensure(c00));
  CK(c->featA.ensure(feat));
  CK(c->featB.ensure(feat));
  c->ws_Hp = g.Hp;
  c->ws_Wp = g.Wp;
  return VFI_OK;
}

#define LAUNCH(call)                                               \
  do {                                                             \
    cudaError_t _e = (call);                                       \
    c->launches++;                                                 \
    if (_e != cudaSuccess) {                                       \
      set_error(std::string(#call) + ": " + cudaGetErrorString(_e)); \
      return VFI_E_CUDA;                                           \
    }                                                              \
  } while (0)

// encode head of arch 4.7 / 4.17 for frames [f, f + n) of the prepared window (n <= kMaxBatch + 2), once per source frame
int run_encode(vfi_ctx* c, const Geometry& g, int f, int n, cudaStream_t st) {
  const size_t px = (size_t)g.Hp * g.Wp;
  const float4* imgs = (const float4*)c->imgs.p + (size_t)f * px;
  if (c->arch == 47) {
    LAUNCH(launch_encode(imgs, c->enc[0], c->enc[1], c->enc[2], c->enc[3], (float*)c->e16.p,
                         (uint2*)c->feats.p + (size_t)f * px, n, g.Hp, g.Wp, st));
  } else if (c->arch == 417 || c->arch == 426) {
    const int Hh = g.Hp / 2, Wh = g.Wp / 2;
    const size_t fbytes = c->arch == 417 ? 16 : 8;  // feature bytes per full-resolution pixel
    LAUNCH(launch_head0(c->op_type, imgs, c->enc[0], c->enc[1], c->hA.p, n, g.Hp, g.Wp, st));
    LAUNCH(launch_tapconv(c->head[0], c->op_type, c->hA.p, c->hB.p, nullptr, nullptr, n, Hh, Wh, c->num_sms, false, st));
    LAUNCH(launch_tapconv(c->head[1], c->op_type, c->hB.p, c->hA.p, nullptr, nullptr, n, Hh, Wh, c->num_sms, false, st));
    LAUNCH(launch_tapconv(c->head[2], c->op_type, c->hA.p, (uint8_t*)c->feats.p + (size_t)f * px * fbytes, nullptr, nullptr,
                          n, Hh, Wh, c->num_sms, false, st));
  }
  return VFI_OK;
}

// one internal pass: tasks (indices into the prepared frame window c->imgs) -> out [n, H, W, 3]
int forward_pass(vfi_ctx* c, const Geometry& g, const BatchTasks& tasks, int H, int W, float* out, cudaStream_t st) {
  const int B = tasks.n;
  const float4* imgs = (const float4*)c->imgs.p;
  const uint2* imgs_h = (const uint2*)c->imgs_h.p;
  const void* feats = c->arch != 46 ? c->feats.p : nullptr;
  const int feat_ch = c->arch == 417 ? 8 : 4;
  const int nb = g.nb;
  float4* F = (float4*)c->flow.p;  // accumulated full-resolution flow / mask, written only by "dense" fronts
  float* M = (float*)c->mask.p;
  FlowState fs{};
  fs.n = nb;
  for (int i = 0; i < nb; ++i) {
    fs.f[i] = (float4*)c->tF[i].p;
    fs.m[i] = (float*)c->tM[i].p;
    fs.s[i] = g.s[i];
  }
  fs.mask_replace = (c->arch != 46) ? 1 : 0;
  int dense = nb;  // first block whose front visits every full-resolution pixel (scale <= 2)
  for (int i = nb - 1; i >= 1; --i)
    if (g.s[i] <= 2) dense = i;
  bool have_base = false;
  int lo = 0;  // levels [lo, i) are not yet folded into F
  // group ids of vfi_rife_profile: 10 * block + {0 front, 1 conv0.0, 2 conv0.1, 3 the 8 ResConvs, 4 lastconv(s)}, 90 final
  auto span_begin = [&](int id) {
    if (!c->profile) return;
    vfi_ctx::ProfSpan sp{id, nullptr, nullptr};
    cudaEventCreate(&sp.e0);
    cudaEventCreate(&sp.e1);
    cudaEventRecord(sp.e0, st);
    c->prof_spans.push_back(sp);
  };
  auto span_end = [&]() {
    if (c->profile) cudaEventRecord(c->prof_spans.back().e1, st);
  };
  // The last block's front stores the accumulated flow too and `final` adds one level to it.  VFI_FLOW_STORE_LAST=0: it
  // does not, `final` adds the last TWO levels on the fly.  Measured r02 (profiles/r02_c_bench*.log, per pair): the
  // largest front 38.1 -> 33.6 us without its 20 B/px store, but `final` 35.8 -> 45.4 us (the second level's eight taps
  // per pixel make it instruction bound) - a net loss, so storing stays the default.
  static const bool store_last = [] {
    const char* e = std::getenv("VFI_FLOW_STORE_LAST");
    return !(e && e[0] == '0');
  }();
  for (int i = 0; i < nb; ++i) {
    const int s = g.s[i];
    const int Hs = g.Hp * g.k[i] / s, Ws = g.Wp * g.k[i] / s;
    const void* pfeat = (c->arch == 426 && i > 0) ? c->tE[i - 1].p : nullptr;  // previous block's 8 feature channels
    const int ps = i > 0 ? g.s[i - 1] : 1;
    span_begin(10 * i);
    if (g.k[i] > 1) {
      // up-scaled block: fold every level so far into the dense planes, build the k-times finer input from them
      if (i == 0) return fail(VFI_E_INVALID, "the first block cannot be up-scaled");
      if (lo < i) {
        FlowState part = fs;
        part.n = i;
        LAUNCH(launch_materialize(part, lo, have_base ? F : nullptr, have_base ? M : nullptr, F, M, B, g.Hp, g.Wp, st));
        have_base = true;
        lo = i;
      }
      LAUNCH(launch_front_up(c->op_type, c->arch, imgs_h, feats, pfeat, ps, g.k[i - 1], F, M, tasks, g.Hp, g.Wp, g.k[i], c->x.p,
                             st));
    } else if (i == 0 || i < dense) {
      LAUNCH(launch_front(c->op_type, c->arch, imgs, imgs_h, feats, feat_ch, pfeat, ps, fs, i, 0, nullptr, nullptr, nullptr,
                          nullptr, tasks, g.Hp, g.Wp, s, c->x.p, st));
    } else if (i == nb - 1 && have_base && !store_last && i - lo + 1 <= 2) {
      // last block: read the dense planes (+ the levels since), store nothing; `final` adds those levels and this one
      LAUNCH(launch_front(c->op_type, c->arch, imgs, imgs_h, feats, feat_ch, pfeat, ps, fs, i, lo, F, M, nullptr, nullptr, tasks,
                          g.Hp, g.Wp, s, c->x.p, st));
    } else {
      LAUNCH(launch_front(c->op_type, c->arch, imgs, imgs_h, feats, feat_ch, pfeat, ps, fs, i, lo, have_base ? F : nullptr,
                          have_base ? M : nullptr, F, M, tasks, g.Hp, g.Wp, s, c->x.p, st));
      have_base = true;
      lo = i;
    }
    span_end();
    span_begin(10 * i + 1);
    LAUNCH(launch_tapconv(c->layers[i][0], c->op_type, c->x.p, c->c00.p, nullptr, nullptr, B, Hs / 2, Ws / 2,
                          c->num_sms, false, st));
    span_end();
    span_begin(10 * i + 2);
    LAUNCH(launch_tapconv(c->layers[i][1], c->op_type, c->c00.p, c->featA.p, nullptr, nullptr, B, Hs / 4, Ws / 4,
                          c->num_sms, false, st));
    span_end();
    void* a = c->featA.p;
    void* b = c->featB.p;
    span_begin(10 * i + 3);
    for (int j = 0; j < 8; ++j) {
      LAUNCH(launch_tapconv(c->layers[i][2 + j], c->op_type, a, b, nullptr, nullptr, B, Hs / 4, Ws / 4, c->num_sms,
                            false, st));
      std::swap(a, b);
    }
    span_end();
    span_begin(10 * i + 4);
    LAUNCH(launch_tapconv(c->layers[i][10], c->op_type, a, nullptr, fs.f[i], fs.m[i], B, Hs / 4, Ws / 4, c->num_sms,
                          false, st));
    if (c->arch == 426 && i + 1 < nb)  // the 8 feature channels of lastconv, for the next block's input
      LAUNCH(launch_tapconv(c->layers[i][11], c->op_type, a, c->tE[i].p, nullptr, nullptr, B, Hs / 4, Ws / 4, c->num_sms,
                            false, st));
    if (g.k[i] > 1) {  // the up-scaled block's output goes straight back onto the dense planes
      LAUNCH(launch_fold_down(fs.f[i], fs.m[i], g.k[i], F, M, B, g.Hp, g.Wp, fs.mask_replace, st));
      lo = i + 1;
    }
    span_end();
  }
  span_begin(90);
  LAUNCH(launch_final(imgs, fs, lo, have_base ? F : nullptr, have_base ? M : nullptr, tasks, g.Hp, g.Wp, H, W, out, st));
  span_end();
  c->last_fs = fs;
  c->last_lo = lo;
  c->last_have_base = have_base;
  c->ws_B = B;
  return VFI_OK;
}

int check_tasks(const int32_t* f0, const int32_t* f1, int n_tasks, int lo, int hi) {
  for (int i = 0; i < n_tasks; ++i)
    if (f0[i] < lo || f0[i] >= hi || f1[i] < lo || f1[i] >= hi) return fail(VFI_E_INVALID, "task frame index out of range");
  return VFI_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char* vfi_last_error(void) { return g_err.c_str(); }
const char* vfi_version(void) { return "vfi_b200 0.2 (sm_100a; RIFE 4.6/4.7/4.17/4.26, FILM, Sepconv, GMFSS Fortuna building blocks; built " __DATE__ " " __TIME__ ")"; }

int vfi_create(int device, vfi_ctx** out) {
  if (!out) return fail(VFI_E_INVALID, "null out");
  int n = 0;
  CK(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) return fail(VFI_E_INVALID, "no such CUDA device");
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(VFI_E_INVALID, "libvfi_b200 needs a compute-capability 10.x (B200, sm_100a) GPU");
  vfi_ctx* c = new vfi_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  {
    // VFI_NUM_SMS=n: size the persistent grids for n SMs (an even number, at least 2), leaving the rest to kernels of other
    // streams - e.g. NCCL's receive kernels on the rank that gathers every other rank's frames
    const int want = env_int("VFI_NUM_SMS", 0, 0, 4096);
    if (want >= 2 && want < c->num_sms) c->num_sms = want & ~1;
  }
  CK(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&c->ops_done, cudaEventDisableTiming));
  *out = c;
  return VFI_OK;
}

int vfi_destroy(vfi_ctx* c) {
  if (!c) return VFI_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  free_weights(c);
  film_destroy(c->film);
  c->film = nullptr;
  sepconv_destroy(c->sep);
  c->sep = nullptr;
  for (DevBuf* b : {&c->imgs, &c->imgs_h, &c->flow, &c->mask, &c->x, &c->c00, &c->featA, &c->featB, &c->raw, &c->outdev, &c->feats, &c->e16, &c->hA, &c->hB, &c->dbgF,
                    &c->dbgM, &c->ops_a, &c->ops_b})
    b->release();
  for (int i = 0; i < kMaxBlocks; ++i) {
    c->tF[i].release();
    c->tM[i].release();
    c->tE[i].release();
  }
  c->pin_in.release();
  c->pin_out.release();
  if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
  if (c->s_comp) cudaStreamDestroy(c->s_comp);
  if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
  if (c->ops_done) cudaEventDestroy(c->ops_done);
  delete c;
  return VFI_OK;
}

int64_t vfi_launch_count(const vfi_ctx* c) { return c ? c->launches : 0; }

int vfi_set_batch(vfi_ctx* c, int batch) {
  if (!c || batch < 1 || batch > kMaxBatch) return fail(VFI_E_INVALID, "batch must be in [1,16]");
  c->batch = batch;
  return VFI_OK;
}

// Per-group device times of the forward schedule: CUDA events on the launching stream around each kernel group of every
// pass run while profiling is on (the groups and their ids are listed in forward_pass).  Off by default: the event
// records break the dependent-launch chaining between groups, so the timed bench steps run without it.
int vfi_rife_profile(vfi_ctx* c, int enable) {
  if (!c) return fail(VFI_E_INVALID, "null ctx");
  CK(cudaSetDevice(c->device));
  CK(cudaDeviceSynchronize());
  for (auto& sp : c->prof_spans) {
    cudaEventDestroy(sp.e0);
    cudaEventDestroy(sp.e1);
  }
  c->prof_spans.clear();
  c->profile = enable != 0;
  return VFI_OK;
}

// Synchronises, then sums the recorded spans per group id: ids[i], total_ms[i], count[i] for up to `cap` groups; returns
// the number of groups through *n_out and clears the record.
int vfi_rife_profile_read(vfi_ctx* c, int32_t* ids, float* total_ms, int32_t* count, int cap, int* n_out) {
  if (!c || !ids || !total_ms || !count || !n_out || cap < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  CK(cudaDeviceSynchronize());
  int n = 0;
  for (auto& sp : c->prof_spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, sp.e0, sp.e1) != cudaSuccess) ms = 0.f;
    int k = 0;
    while (k < n && ids[k] != sp.id) ++k;
    if (k == n) {
      if (n == cap) continue;
      ids[n] = sp.id;
      total_ms[n] = 0.f;
      count[n] = 0;
      ++n;
    }
    total_ms[k] += ms;
    count[k] += 1;
    cudaEventDestroy(sp.e0);
    cudaEventDestroy(sp.e1);
  }
  c->prof_spans.clear();
  *n_out = n;
  return VFI_OK;
}

int vfi_sync(vfi_ctx* c) {
  if (!c) return fail(VFI_E_INVALID, "null ctx");
  CK(cudaSetDevice(c->device));
  CK(cudaDeviceSynchronize());
  return VFI_OK;
}

int vfi_rife46_load(vfi_ctx* c, const float* const* T, const int64_t* numel, int n_tensors, int operand_type) {
  return vfi_rife_load(c, 46, T, numel, n_tensors, operand_type);
}

int vfi_rife_load(vfi_ctx* c, int arch, const float* const* T, const int64_t* numel, int n_tensors, int operand_type) {
  if (!c || !T || !numel) return fail(VFI_E_INVALID, "null argument");
  if (arch != 46 && arch != 47 && arch != 417 && arch != 426)
    return fail(VFI_E_NOTIMPL,
                "RIFE arch must be 46 (rife46.pth), 47 (rife47/rife49.pth), 417 (rife417.pth) or 426 (rife426.pth)");
  if (n_tensors != (arch == 46 ? VFI_RIFE46_NUM_TENSORS : arch == 47 ? VFI_RIFE47_NUM_TENSORS
                    : arch == 417 ? VFI_RIFE417_NUM_TENSORS : VFI_RIFE426_NUM_TENSORS))
    return fail(VFI_E_INVALID,
                "wrong number of state_dict tensors for this RIFE arch (4.6: 120, 4.7: 124, 4.17: 128, 4.26: 158)");
  if (operand_type != OP_F16 && operand_type != OP_BF16) return fail(VFI_E_INVALID, "operand_type");
  CK(cudaSetDevice(c->device));
  free_weights(c);
  c->op_type = operand_type;
  c->arch = arch;
  int k = 0;
  auto expect = [&](int idx, int64_t want) { return numel[idx] == want; };
  const int nb = num_blocks(arch);
  const int nlast = arch == 426 ? 52 : 24;  // lastconv = ConvTranspose2d(c, 4*6 | 4*13, 4, 2, 1) - rife_arch.py:215-218, :230-233
  for (int b = 0; b < nb; ++b) {
    const int ch = kBlockC[b];
    const int cin = (arch == 426 ? kBlockCinReal426 : arch == 417 ? kBlockCinReal417 : arch == 47 ? kBlockCinReal47
                                                                                                  : kBlockCinReal)[b];
    if (!expect(k, (int64_t)(ch / 2) * cin * 9) || !expect(k + 1, ch / 2) || !expect(k + 2, (int64_t)ch * (ch / 2) * 9) ||
        !expect(k + 3, ch))
      return fail(VFI_E_INVALID, "conv0 tensor sizes do not match RIFE 4.6");
    int r;
    if ((r = build_conv_s2(c, c->layers[b][0], arch != 46 ? 32 : 16, cin, ch / 2, 1, T[k], T[k + 1]))) return r;
    if ((r = build_conv_s2(c, c->layers[b][1], ch / 2, ch / 2, ch, 0, T[k + 2], T[k + 3]))) return r;
    k += 4;
    for (int j = 0; j < 8; ++j) {
      if (!expect(k, ch) || !expect(k + 1, (int64_t)ch * ch * 9) || !expect(k + 2, ch))
        return fail(VFI_E_INVALID, "convblock tensor sizes do not match RIFE 4.6");
      if ((r = build_resconv(c, c->layers[b][2 + j], ch, T[k], T[k + 1], T[k + 2]))) return r;
      k += 3;
    }
    if (!expect(k, (int64_t)ch * nlast * 16) || !expect(k + 1, nlast))
      return fail(VFI_E_INVALID, "lastconv tensor sizes do not match this RIFE arch");
    if ((r = build_lastconv(c, c->layers[b][10], ch, nlast, T[k], T[k + 1]))) return r;
    if (arch == 426 && b + 1 < nb && (r = build_lastfeat(c, c->layers[b][11], ch, nlast, T[k], T[k + 1]))) return r;
    k += 2;
  }
  if (arch == 47) {  // encode = Conv2d(3,16,3,2,1) + ConvTranspose2d(16,4,4,2,1), fp32 on the CUDA cores
    const int64_t want[4] = {16 * 3 * 9, 16, 16 * 4 * 16, 4};
    for (int i = 0; i < 4; ++i) {
      if (numel[k + i] != want[i]) return fail(VFI_E_INVALID, "encode tensor sizes do not match RIFE 4.7");
      std::vector<float> h(T[k + i], T[k + i] + want[i]);
      int r;
      if ((r = upload(c, h, (void**)&c->enc[i]))) return r;
    }
    k += 4;
  }
  if (arch == 417) {  // encode = Head_417: cnn0 on the CUDA cores (fp32 weights), cnn1..cnn3 as tapconv layers
    const int64_t want[8] = {32 * 3 * 9, 32, 32 * 32 * 9, 32, 32 * 32 * 9, 32, 32 * 8 * 16, 8};
    for (int i = 0; i < 8; ++i)
      if (numel[k + i] != want[i]) return fail(VFI_E_INVALID, "encode tensor sizes do not match RIFE 4.17");
    int r;
    for (int i = 0; i < 2; ++i) {
      std::vector<float> h(T[k + i], T[k + i] + want[i]);
      if ((r = upload(c, h, (void**)&c->enc[i]))) return r;
    }
    if ((r = build_conv3x3_lrelu(c, c->head[0], 32, 32, T[k + 2], T[k + 3]))) return r;
    if ((r = build_conv3x3_lrelu(c, c->head[1], 32, 32, T[k + 4], T[k + 5]))) return r;
    if ((r = build_deconv_s2d(c, c->head[2], 32, 32, 8, T[k + 6], T[k + 7]))) return r;
    for (int i = 0; i < 3; ++i)
      if (c->head[i].nsplit < 1) return fail(VFI_E_STATE, "a head layer has no shared-memory plan");
    k += 8;
  }
  if (arch == 426) {
    // encode = Head (rife_arch.py:378-395): the 16-channel layers run zero-padded to 32 channels - cnn0 on the CUDA
    // cores (fp32 weights, outputs 16..31 have zero weights and bias), cnn1..cnn3 as tapconv layers; cnn3's 4 output
    // channels x 2x2 sub-pixels = 16 columns = the space-to-depth form of the 4-channel feature map
    const int64_t want[8] = {16 * 3 * 9, 16, 16 * 16 * 9, 16, 16 * 16 * 9, 16, 16 * 4 * 16, 4};
    for (int i = 0; i < 8; ++i)
      if (numel[k + i] != want[i]) return fail(VFI_E_INVALID, "encode tensor sizes do not match RIFE 4.26");
    int r;
    std::vector<float> w0(32 * 27, 0.f), b0(32, 0.f);
    std::copy(T[k], T[k] + 16 * 27, w0.begin());
    std::copy(T[k + 1], T[k + 1] + 16, b0.begin());
    if ((r = upload(c, w0, (void**)&c->enc[0]))) return r;
    if ((r = upload(c, b0, (void**)&c->enc[1]))) return r;
    if ((r = build_conv3x3_lrelu(c, c->head[0], 32, 16, T[k + 2], T[k + 3]))) return r;
    if ((r = build_conv3x3_lrelu(c, c->head[1], 32, 16, T[k + 4], T[k + 5]))) return r;
    if ((r = build_deconv_s2d(c, c->head[2], 32, 16, 4, T[k + 6], T[k + 7]))) return r;
    for (int i = 0; i < 3; ++i)
      if (c->head[i].nsplit < 1) return fail(VFI_E_STATE, "a head layer has no shared-memory plan");
    k += 8;
  }
  for (int b = 0; b < nb; ++b)
    for (int l = 0; l < (arch == 426 && b + 1 < nb ? 12 : 11); ++l)
      if (c->layers[b][l].nsplit < 1) return fail(VFI_E_STATE, "a layer has no shared-memory plan");
  c->loaded = true;
  return VFI_OK;
}

int vfi_rife46_forward(vfi_ctx* c, const float* frames, int n_frames, int H, int W, int C, const int32_t* f0,
                       const int32_t* f1, const float* t, int n_tasks, float scale_factor, float* out, void* stream) {
  if (!c || !frames || !out || (n_tasks > 0 && (!f0 || !f1 || !t))) return fail(VFI_E_INVALID, "null argument");
  if (!c->loaded) return fail(VFI_E_STATE, "vfi_rife46_load has not been called");
  if (C < 3 || H < 1 || W < 1 || n_frames < 1) return fail(VFI_E_INVALID, "bad frame shape");
  if (n_tasks == 0) return VFI_OK;
  int r;
  if ((r = check_tasks(f0, f1, n_tasks, 0, n_frames))) return r;
  CK(cudaSetDevice(c->device));
  Geometry g;
  if ((r = make_geometry(c->arch, H, W, scale_factor, &g))) return r;
  int lo = n_frames, hi = 0;
  for (int i = 0; i < n_tasks; ++i) {
    lo = std::min(lo, std::min(f0[i], f1[i]));
    hi = std::max(hi, std::max(f0[i], f1[i]) + 1);
  }
  const int B = std::min(c->batch, n_tasks);
  if ((r = ensure_workspace(c, g, B, hi - lo))) return r;
  cudaStream_t st = (cudaStream_t)stream;
  LAUNCH(launch_prep_frames(frames + (size_t)lo * H * W * C, hi - lo, H, W, C, (float4*)c->imgs.p, (uint2*)c->imgs_h.p,
                            g.Hp, g.Wp, st));
  if (c->arch != 46) {  // encode head, once per source frame, in groups that fit the half-resolution scratch
    for (int f = 0; f < hi - lo; f += kMaxBatch) {
      const int cnt = std::min(kMaxBatch, hi - lo - f);
      if ((r = run_encode(c, g, f, cnt, st))) return r;
    }
  }
  for (int pos = 0; pos < n_tasks; pos += B) {
    BatchTasks bt{};
    bt.n = std::min(B, n_tasks - pos);
    for (int i = 0; i < bt.n; ++i) {
      bt.f0[i] = f0[pos + i] - lo;
      bt.f1[i] = f1[pos + i] - lo;
      bt.t[i] = t[pos + i];
    }
    if ((r = forward_pass(c, g, bt, H, W, out + (size_t)pos * H * W * 3, st))) return r;
  }
  return VFI_OK;
}

int vfi_rife46_interpolate_host(vfi_ctx* c, const float* frames, int n_frames, int H, int W, int C, int frame_lo,
                                int frame_hi, const int32_t* f0, const int32_t* f1, const float* t,
                                const int32_t* out_slot, const int32_t* frame_slot, int n_tasks, float scale_factor,
                                float* out) {
  if (!c || !frames || (n_tasks > 0 && (!out || !f0 || !f1 || !t))) return fail(VFI_E_INVALID, "null argument");
  if (!c->loaded) return fail(VFI_E_STATE, "vfi_rife46_load has not been called");
  if (C < 3 || H < 1 || W < 1 || frame_lo < 0 || frame_hi > n_frames || frame_lo >= frame_hi)
    return fail(VFI_E_INVALID, "bad frame shape / range");
  if (n_tasks == 0) return VFI_OK;
  int r;
  if ((r = check_tasks(f0, f1, n_tasks, frame_lo, frame_hi))) return r;
  for (int i = 1; i < n_tasks; ++i)
    if (std::min(f0[i], f1[i]) < std::min(f0[i - 1], f1[i - 1]))
      return fail(VFI_E_INVALID, "tasks must be ordered by frame index (as RIFE_VFI.vfi builds them)");
  CK(cudaSetDevice(c->device));
  Geometry g;
  if ((r = make_geometry(c->arch, H, W, scale_factor, &g))) return r;
  const int nf = frame_hi - frame_lo;
  const int B = std::min(c->batch, n_tasks);
  const size_t frame_elems = (size_t)H * W * C, out_elems = (size_t)H * W * 3;
  const size_t frame_bytes = frame_elems * sizeof(float), out_bytes = out_elems * sizeof(float);
  // pass sizes: full batches in the middle; on a long clip the first and the last passes are small (1, 2, 4 pairs) so
  // that the exposed head (upload before the first pass) and tail (download after the last) are one or two frames
  // instead of a whole batch (r01: 64 frames e2e = 63 x 0.574 ms + 7.3 ms of head and tail with uniform passes)
  std::vector<int> pass_pos, pass_n;
  {
    const bool ramp = B >= 8 && n_tasks >= 4 * B;
    int pos = 0;
    if (ramp)
      for (int n = 1; n < B && n <= 4; n *= 2) { pass_pos.push_back(pos); pass_n.push_back(n); pos += n; }
    const int tail = ramp ? 7 : 0;
    while (n_tasks - pos - tail >= B || (!ramp && pos < n_tasks)) {
      const int n = std::min(B, n_tasks - pos);
      pass_pos.push_back(pos); pass_n.push_back(n); pos += n;
    }
    if (ramp) {
      const int rest = n_tasks - pos;  // 7 .. B + 6 pairs left: [rest - 3, 2, 1] or [rest - 7, 4, 2, 1]
      int tail_n[4], nt = 0;
      if (rest - 3 <= B) { tail_n[nt++] = rest - 3; } else { tail_n[nt++] = rest - 7; tail_n[nt++] = 4; }
      tail_n[nt++] = 2;
      tail_n[nt++] = 1;
      for (int i = 0; i < nt; ++i) { pass_pos.push_back(pos); pass_n.push_back(tail_n[i]); pos += tail_n[i]; }
    }
  }
  const int nb = (int)pass_n.size();

  // ---- the prepared-frame window is a RING: only frames some task references are uploaded, in order of first use, into
  // slot (upload counter % R).  R covers every frame from its upload to the pass after its last use, so that the slot a
  // pass's uploads overwrite was last read two passes ago (the copy stream runs one pass ahead of the compute stream
  // without waiting) - 2 B + 1 slots for consecutive pairs instead of the whole clip (r01: 50-67 MB per 1080p frame for
  // every frame of the clip; a few thousand frames did not fit).  An event wait keeps any reuse correct regardless.
  std::vector<int> first_pass(nf, -1), last_pass(nf, -1), ctr(nf, -1), up_frames, up_end(nb, 0);
  for (int k = 0; k < nb; ++k)
    for (int i = 0; i < pass_n[k]; ++i)
      for (int f : {f0[pass_pos[k] + i] - frame_lo, f1[pass_pos[k] + i] - frame_lo}) {
        if (first_pass[f] < 0) first_pass[f] = k;
        last_pass[f] = k;
      }
  {
    std::vector<std::vector<int>> by_pass(nb);
    for (int f = 0; f < nf; ++f)
      if (first_pass[f] >= 0) by_pass[first_pass[f]].push_back(f);
    for (int k = 0; k < nb; ++k) {
      for (int f : by_pass[k]) {
        ctr[f] = (int)up_frames.size();
        up_frames.push_back(f);
      }
      up_end[k] = (int)up_frames.size();
    }
  }
  int R = 1;
  for (int f = 0; f < nf; ++f)
    if (ctr[f] >= 0) R = std::max(R, up_end[std::min(last_pass[f] + 1, nb - 1)] - ctr[f]);
  if ((r = ensure_workspace(c, g, B, R))) return r;
  const int kRaw = 2 * kMaxBatch + 4;  // raw upload ring (frames), overwritten in stream order on the copy stream
  CK(c->raw.ensure((size_t)kRaw * frame_bytes));
  CK(c->outdev.ensure((size_t)2 * B * out_bytes));

  // ---- host staging.  Pinned caller memory is copied from / to directly.  Pageable memory (what a ComfyUI IMAGE
  // tensor is) goes through a small ring of pinned buffers: an uploader thread memcpy's frame by frame into it ahead of
  // the H2D copies, a downloader thread empties the D2H ring into the caller's tensor; each uses a few copy threads.
  // Pass-through frames (frame_slot): source frame f is also wanted unchanged (first 3 channels) at out + frame_slot[f].
  // The uploader thread makes that copy - and when `out` is page-locked the frame is then UPLOADED FROM THERE: the one
  // host copy the node contract needs anyway doubles as the staging copy (r02: staging and pass-through as two separate
  // copies ran at ~20 GB/s each on the box's cgroup-limited host cores and were the critical path, 91 ms for a 40 ms
  // pipeline).
  const bool stage_out = !is_pinned_host(out);
  auto via_out = [&](int f_abs) { return frame_slot != nullptr && !stage_out && frame_slot[f_abs] >= 0; };
  bool any_ring = false, any_pt = false;
  const bool src_pinned = is_pinned_host(frames + (size_t)frame_lo * frame_elems);
  for (int f : up_frames) any_ring = any_ring || (!src_pinned && !via_out(f + frame_lo));
  if (frame_slot)
    for (int f = frame_lo; f < frame_hi; ++f) any_pt = any_pt || frame_slot[f] >= 0;
  const bool stage_in = any_ring;
  const int copy_threads = env_int("VFI_COPY_THREADS", 12, 1, 32);
  const size_t ring_mb = (size_t)env_int("VFI_STAGE_MB", 384, 32, 8192);
  const int force_slots = env_int("VFI_STAGE_SLOTS", 0, 0, 64);  // tests: a ring far smaller than the clip
  const int NS = !stage_in ? 0 : force_slots ? force_slots : (int)std::max<size_t>(4, std::min<size_t>(32, (ring_mb << 20) / frame_bytes));
  const int ND = !stage_out ? 0 : force_slots ? force_slots : (int)std::max<size_t>(4, std::min<size_t>(48, (ring_mb << 20) / out_bytes));
  if (stage_in) CK(c->pin_in.ensure((size_t)NS * frame_bytes));
  if (stage_out) CK(c->pin_out.ensure((size_t)ND * out_bytes));

  std::vector<cudaEvent_t> ev_up(nb), ev_comp(nb), ev_down(nb), ev_in(NS), ev_out(ND);
  auto mk = [](std::vector<cudaEvent_t>& v) {
    for (auto& e : v)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return false;
    return true;
  };
  for (auto& e : ev_up) e = nullptr;
  for (auto& e : ev_comp) e = nullptr;
  for (auto& e : ev_down) e = nullptr;
  for (auto& e : ev_in) e = nullptr;
  for (auto& e : ev_out) e = nullptr;
  if (!(mk(ev_up) && mk(ev_comp) && mk(ev_down) && mk(ev_in) && mk(ev_out))) return fail(VFI_E_CUDA, "cudaEventCreate failed");

  // shared progress counters of the three host threads (all under one mutex; the hand-offs are per frame, ~0.5 ms apart)
  std::mutex mu;
  std::condition_variable cv;
  bool abort_all = false;
  int staged = 0;        // uploader: frames [0, staged) of up_frames sit in the pinned ring
  int h2d_issued = 0;    // main: H2D copies [0, h2d_issued) have been enqueued (their ev_in is recorded)
  int d2h_issued = 0;    // main: D2H copies [0, d2h_issued) have been enqueued (their ev_out is recorded)
  int drained = 0;       // downloader: output frames [0, drained) have been copied to the caller's tensor
  std::vector<int> d2h_slot;  // output slot of D2H copy i
  d2h_slot.reserve(n_tasks);
  const int n_up = (int)up_frames.size();
  // upload u comes from: the caller's pinned tensor (-2), its pass-through slot in the pinned output (-1), or pinned
  // staging ring entry ring_of[u] >= 0 (a running count of ring uploads)
  std::vector<int> ring_of(n_up, -2);
  {
    int nr = 0;
    for (int u = 0; u < n_up; ++u) {
      const int fa = up_frames[u] + frame_lo;
      if (via_out(fa)) ring_of[u] = -1;
      else if (!src_pinned) ring_of[u] = nr++;
    }
  }
  const size_t px_frame = (size_t)H * W;

  // VFI_TRACE=1: where the host threads spent their time (stderr, one line per call)
  const bool trace = env_int("VFI_TRACE", 0, 0, 1) != 0;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
    return std::chrono::duration<double>(b - a).count();
  };
  double up_copy_s = 0, up_wait_s = 0, dn_copy_s = 0, dn_wait_s = 0, main_wait_stage_s = 0, main_wait_drain_s = 0;
  const auto t_call = now();

  std::thread uploader, downloader;
  if (stage_in || any_pt)
    uploader = std::thread([&] {
      cudaSetDevice(c->device);
      CopyPool pool(copy_threads);
      std::vector<char> pt_done(nf, 0);
      for (int u = 0; u < n_up; ++u) {
        const auto tw = now();
        const int fa = up_frames[u] + frame_lo;
        const float* src = frames + (size_t)fa * frame_elems;
        const int ri = ring_of[u];
        if (ri >= NS && ri >= 0) {  // the H2D copy that last read this pinned slot has been enqueued, then: has completed
          {
            std::unique_lock<std::mutex> l(mu);
            cv.wait(l, [&] { return abort_all || h2d_issued > ri - NS; });
            if (abort_all) return;
          }
          cudaEventSynchronize(ev_in[ri % NS]);
        }
        const auto tc = now();
        if (ri >= 0) pool.copy((uint8_t*)c->pin_in.p + (size_t)(ri % NS) * frame_bytes, src, frame_bytes);
        if (frame_slot && frame_slot[fa] >= 0) {
          pool.copy_rgb(out + (size_t)frame_slot[fa] * out_elems, src, px_frame, C);
          pt_done[fa - frame_lo] = 1;
        }
        up_wait_s += secs(tw, tc);
        up_copy_s += secs(tc, now());
        {
          std::lock_guard<std::mutex> l(mu);
          staged = u + 1;
        }
        cv.notify_all();
      }
      if (frame_slot)  // pass-through frames no task references (skipped pairs)
        for (int f = frame_lo; f < frame_hi; ++f)
          if (frame_slot[f] >= 0 && !pt_done[f - frame_lo]) {
            const auto tc = now();
            pool.copy_rgb(out + (size_t)frame_slot[f] * out_elems, frames + (size_t)f * frame_elems, px_frame, C);
            up_copy_s += secs(tc, now());
          }
    });
  if (stage_out)
    downloader = std::thread([&] {
      cudaSetDevice(c->device);
      CopyPool pool(copy_threads);
      for (int v = 0; v < n_tasks; ++v) {
        int slot;
        const auto tw = now();
        {
          std::unique_lock<std::mutex> l(mu);
          cv.wait(l, [&] { return abort_all || d2h_issued > v; });
          if (abort_all) return;
          slot = d2h_slot[v];
        }
        cudaEventSynchronize(ev_out[v % ND]);
        const auto tc = now();
        pool.copy(out + (size_t)slot * out_elems, (const uint8_t*)c->pin_out.p + (size_t)(v % ND) * out_bytes, out_bytes);
        dn_wait_s += secs(tw, tc);
        dn_copy_s += secs(tc, now());
        {
          std::lock_guard<std::mutex> l(mu);
          drained = v + 1;
        }
        cv.notify_all();
      }
    });

  int rc = VFI_OK;
  auto body = [&]() -> int {
    int up = 0, down = 0;  // upload / download counters
    for (int k = 0; k < nb; ++k) {
      const int pos = pass_pos[k], n = pass_n[k];
      // H2D + prep of the frames this pass uses for the first time, on the copy stream
      while (up < up_end[k]) {
        const int slot = up % R, rslot = up % kRaw;
        int run = std::min(std::min(up_end[k] - up, kRaw / 2), std::min(R - slot, kRaw - rslot));
        // a run is prepared by one kernel launch: its frames must have the same channel stride (3 from the output's
        // pass-through slots, C otherwise)
        const bool run_rgb = ring_of[up] == -1;
        for (int j = 1; j < run; ++j)
          if ((ring_of[up + j] == -1) != run_rgb) run = j;
        const size_t run_elems = run_rgb ? out_elems : frame_elems;
        for (int j = 0; j < run; ++j) {
          const int u = up + j;
          if (u >= R) CK(cudaStreamWaitEvent(c->s_h2d, ev_comp[last_pass[up_frames[u - R]]], 0));  // slot's last reader
          const int fa = up_frames[u] + frame_lo;
          const int ri = ring_of[u];
          const float* src = frames + (size_t)fa * frame_elems;
          if (ri != -2) {  // staged by the uploader thread
            const auto tw = now();
            std::unique_lock<std::mutex> l(mu);
            cv.wait(l, [&] { return staged > u; });
            src = (ri == -1) ? out + (size_t)frame_slot[fa] * out_elems
                             : (const float*)((const uint8_t*)c->pin_in.p + (size_t)(ri % NS) * frame_bytes);
            main_wait_stage_s += secs(tw, now());
          }
          CK(cudaMemcpyAsync((float*)c->raw.p + (size_t)rslot * frame_elems + (size_t)j * run_elems, src,
                             run_elems * sizeof(float), cudaMemcpyHostToDevice, c->s_h2d));
          if (ri >= 0) {
            CK(cudaEventRecord(ev_in[ri % NS], c->s_h2d));
            {
              std::lock_guard<std::mutex> l(mu);
              h2d_issued = ri + 1;
            }
            cv.notify_all();
          }
        }
        const size_t px = (size_t)g.Hp * g.Wp;
        LAUNCH(launch_prep_frames((float*)c->raw.p + (size_t)rslot * frame_elems, run, H, W, run_rgb ? 3 : C,
                                  (float4*)c->imgs.p + (size_t)slot * px, (uint2*)c->imgs_h.p + (size_t)slot * px, g.Hp, g.Wp,
                                  c->s_h2d));
        if (c->arch != 46) {
          const int r3 = run_encode(c, g, slot, run, c->s_h2d);
          if (r3) return r3;
        }
        up += run;
      }
      CK(cudaEventRecord(ev_up[k], c->s_h2d));
      CK(cudaStreamWaitEvent(c->s_comp, ev_up[k], 0));
      if (k >= 2) CK(cudaStreamWaitEvent(c->s_comp, ev_down[k - 2], 0));  // output slot free again
      BatchTasks bt{};
      bt.n = n;
      for (int i = 0; i < n; ++i) {
        bt.f0[i] = ctr[f0[pos + i] - frame_lo] % R;
        bt.f1[i] = ctr[f1[pos + i] - frame_lo] % R;
        bt.t[i] = t[pos + i];
      }
      float* od = (float*)c->outdev.p + (size_t)(k & 1) * B * out_elems;
      int r2 = forward_pass(c, g, bt, H, W, od, c->s_comp);
      if (r2) return r2;
      CK(cudaEventRecord(ev_comp[k], c->s_comp));
      CK(cudaStreamWaitEvent(c->s_d2h, ev_comp[k], 0));
      if (stage_out) {
        for (int i = 0; i < n; ++i, ++down) {
          {  // the downloader has emptied the pinned slot this copy lands in
            const auto tw = now();
            std::unique_lock<std::mutex> l(mu);
            cv.wait(l, [&] { return drained > down - ND; });
            main_wait_drain_s += secs(tw, now());
          }
          CK(cudaMemcpyAsync((uint8_t*)c->pin_out.p + (size_t)(down % ND) * out_bytes, od + (size_t)i * out_elems, out_bytes,
                             cudaMemcpyDeviceToHost, c->s_d2h));
          CK(cudaEventRecord(ev_out[down % ND], c->s_d2h));
          {
            std::lock_guard<std::mutex> l(mu);
            d2h_slot.push_back(out_slot ? out_slot[pos + i] : pos + i);
            d2h_issued = down + 1;
          }
          cv.notify_all();
        }
      } else if (!out_slot) {
        CK(cudaMemcpyAsync(out + (size_t)pos * out_elems, od, (size_t)n * out_bytes, cudaMemcpyDeviceToHost, c->s_d2h));
      } else {
        for (int i = 0; i < n; ++i)
          CK(cudaMemcpyAsync(out + (size_t)out_slot[pos + i] * out_elems, od + (size_t)i * out_elems, out_bytes,
                             cudaMemcpyDeviceToHost, c->s_d2h));
      }
      CK(cudaEventRecord(ev_down[k], c->s_d2h));
    }
    CK(cudaStreamSynchronize(c->s_d2h));
    CK(cudaStreamSynchronize(c->s_comp));
    CK(cudaStreamSynchronize(c->s_h2d));
    return VFI_OK;
  };
  rc = body();
  if (rc != VFI_OK) {
    {
      std::lock_guard<std::mutex> l(mu);
      abort_all = true;
    }
    cv.notify_all();
    cudaDeviceSynchronize();
  }
  if (uploader.joinable()) uploader.join();
  if (downloader.joinable()) downloader.join();
  if (trace)
    fprintf(stderr,
            "vfi trace: interpolate_host dev %d  %d tasks  %d uploads (ring %d)  total %.1f ms | stage_in=%d NS=%d copy %.1f ms "
            "wait %.1f ms | stage_out=%d ND=%d copy %.1f ms wait %.1f ms | main waited %.1f ms for staging, %.1f ms for draining\n",
            c->device, n_tasks, n_up, R, 1e3 * secs(t_call, now()), (int)stage_in, NS, 1e3 * up_copy_s, 1e3 * up_wait_s, (int)stage_out,
            ND, 1e3 * dn_copy_s, 1e3 * dn_wait_s, 1e3 * main_wait_stage_s, 1e3 * main_wait_drain_s);
  for (auto* v : {&ev_up, &ev_comp, &ev_down, &ev_in, &ev_out})
    for (auto e : *v)
      if (e) cudaEventDestroy(e);
  return rc;
}

// Host utility of the node: copy source frame i (first 3 of C channels) to out + slot[i] * H * W * 3 for every i with
// slot[i] >= 0, with `threads` copy threads - the pass-through frames of the output clip (rife/__init__.py:227-231 does a
// torch.cat of per-frame tensors).  Plain host memory on both sides; runs beside vfi_rife46_interpolate_host.
int vfi_host_copy_frames(const float* frames, int n_frames, int H, int W, int C, const int32_t* slot, float* out, int threads) {
  if (!frames || !slot || !out || n_frames < 1 || H < 1 || W < 1 || C < 3) return fail(VFI_E_INVALID, "bad argument");
  if (threads < 1) threads = 1;
  if (threads > 64) threads = 64;
  const size_t px = (size_t)H * W;
  std::vector<std::thread> th;
  std::atomic<int> next{0};
  for (int k = 0; k < threads; ++k)
    th.emplace_back([&] {
      // work items: (frame, quarter of the frame) so that a handful of frames still spreads over all threads
      for (;;) {
        const int item = next.fetch_add(1);
        const int f = item >> 2, q = item & 3;
        if (f >= n_frames) return;
        if (slot[f] < 0) continue;
        const size_t lo = px * q / 4, hi = px * (q + 1) / 4;
        const float* s = frames + (size_t)f * px * C;
        float* d = out + (size_t)slot[f] * px * 3;
        if (C == 3) {
          stream_copy(d + lo * 3, s + lo * 3, (hi - lo) * 3 * sizeof(float));
        } else {
          for (size_t i = lo; i < hi; ++i) {
            d[i * 3 + 0] = s[i * C + 0];
            d[i * 3 + 1] = s[i * C + 1];
            d[i * 3 + 2] = s[i * C + 2];
          }
        }
      }
    });
  for (auto& t : th) t.join();
  return VFI_OK;
}

int vfi_warp_bilinear_border(vfi_ctx* c, const float* img, const float* flow, float* out, int B, int H, int W, int C,
                             void* stream) {
  if (!c || !img || !flow || !out || B < 1 || H < 1 || W < 1 || C < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  LAUNCH(launch_warp(img, flow, out, B, H, W, C, (cudaStream_t)stream));
  return VFI_OK;
}

// ops_a / ops_b belong to the context, not to a stream, and the op entry points run on whatever stream the caller passes.
// A call that uses them first makes its stream wait for the previous user (ops_done), and after its launches records
// ops_done on its own stream, so calls on different streams take turns on the scratch instead of overwriting each other's.
// Growing the buffers frees the old ones, so a regrowth first waits on the host for the previous user to finish.
static cudaError_t ops_scratch_acquire(vfi_ctx* c, size_t bytes, cudaStream_t st) {
  cudaError_t e;
  if (bytes > c->ops_a.cap || bytes > c->ops_b.cap) {
    if ((e = cudaEventSynchronize(c->ops_done)) != cudaSuccess) return e;
    if ((e = c->ops_a.ensure(bytes)) != cudaSuccess) return e;
    if ((e = c->ops_b.ensure(bytes)) != cudaSuccess) return e;
  }
  return cudaStreamWaitEvent(st, c->ops_done, 0);
}

static cudaError_t ops_scratch_release(vfi_ctx* c, cudaStream_t st) { return cudaEventRecord(c->ops_done, st); }

int vfi_softsplat_sum(vfi_ctx* c, const float* in, const float* flow, float* out, int N, int C, int H, int W,
                      void* stream) {
  if (!c || !in || !flow || !out || N < 1 || C < 1 || H < 1 || W < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  LAUNCH(launch_softsplat_sum(in, flow, out, N, C, H, W, (cudaStream_t)stream));
  return VFI_OK;
}

int vfi_softsplat_weighted(vfi_ctx* c, const float* in, const float* flow, const float* metric, int mode, int eps, float* out,
                           float* norm, int N, int C, int H, int W, void* stream) {
  if (!c || !in || !flow || !out || !norm || N < 1 || C < 1 || H < 1 || W < 1) return fail(VFI_E_INVALID, "bad argument");
  if (mode < 0 || mode > 2 || eps < 0 || eps > 2 || (mode != 0 && !metric)) return fail(VFI_E_INVALID, "softsplat mode / eps / metric");
  CK(cudaSetDevice(c->device));
  // default: the channel-last form (16-byte vector atomics); VFI_SPLAT_NHWC=0: the NCHW scalar-atomic kernels (A/B runs)
  static const bool nhwc = [] {
    const char* e = std::getenv("VFI_SPLAT_NHWC");
    return !(e && e[0] == '0');
  }();
  if (nhwc && N <= 65535) {
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    CK(ops_scratch_acquire(c, ops_scratch_floats(N, C, H, W) * sizeof(float), st));
    CK(launch_softsplat_weighted_nhwc(in, flow, metric, mode, eps, out, norm, (float*)c->ops_a.p, (float*)c->ops_b.p, N, C, H, W, st));
    CK(ops_scratch_release(c, st));
    c->launches += 3;
    return VFI_OK;
  }
  CK(launch_softsplat_weighted(in, flow, metric, mode, eps, out, norm, N, C, H, W, static_cast<cudaStream_t>(stream)));
  c->launches += 2;
  return VFI_OK;
}

int vfi_costvol_l1(vfi_ctx* c, const float* one, const float* two, float* out, int N, int C, int H, int W,
                   void* stream) {
  if (!c || !one || !two || !out || N < 1 || C < 1 || H < 1 || W < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  // VFI_VOLUME_WARP=1: the warp-per-pixel channel-last form (shuffle reduction over the channels).  Measured r02
  // (profiles/r02_h_bench_ops*.log): 189 / 705 us against 123 / 258 us of the shared-memory tiled kernel on the 64-channel
  // 96x160 and 128-channel 192x320 shapes - each displacement re-reads its channel vector through L1, 81 times per pixel -
  // so the tiled kernel stays the default and this form is kept for comparison.
  static const bool warp_form = [] {
    const char* e = std::getenv("VFI_VOLUME_WARP");
    return e && e[0] == '1';
  }();
  if (warp_form && N <= 65535 && H <= 65535) {
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    CK(ops_scratch_acquire(c, ops_scratch_floats(N, C, H, W) * sizeof(float), st));
    CK(launch_volume81_warp(false, one, two, out, (float*)c->ops_a.p, (float*)c->ops_b.p, N, C, H, W, st));
    CK(ops_scratch_release(c, st));
    c->launches += 3;
    return VFI_OK;
  }
  LAUNCH(launch_volume81(false, one, two, out, N, C, H, W, (cudaStream_t)stream));
  return VFI_OK;
}

int vfi_corr_dot(vfi_ctx* c, const float* first, const float* second, float* out, int N, int C, int H, int W,
                 void* stream) {
  if (!c || !first || !second || !out || N < 1 || C < 1 || H < 1 || W < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  // VFI_VOLUME_WARP=1: the warp-per-pixel channel-last form (shuffle reduction over the channels).  Measured r02
  // (profiles/r02_h_bench_ops*.log): 189 / 705 us against 123 / 258 us of the shared-memory tiled kernel on the 64-channel
  // 96x160 and 128-channel 192x320 shapes - each displacement re-reads its channel vector through L1, 81 times per pixel -
  // so the tiled kernel stays the default and this form is kept for comparison.
  static const bool warp_form = [] {
    const char* e = std::getenv("VFI_VOLUME_WARP");
    return e && e[0] == '1';
  }();
  if (warp_form && N <= 65535 && H <= 65535) {
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    CK(ops_scratch_acquire(c, ops_scratch_floats(N, C, H, W) * sizeof(float), st));
    CK(launch_volume81_warp(true, first, second, out, (float*)c->ops_a.p, (float*)c->ops_b.p, N, C, H, W, st));
    CK(ops_scratch_release(c, st));
    c->launches += 3;
    return VFI_OK;
  }
  LAUNCH(launch_volume81(true, first, second, out, N, C, H, W, (cudaStream_t)stream));
  return VFI_OK;
}

int vfi_sepconv(vfi_ctx* c, const float* in, const float* ver, const float* hor, float* out, int N, int C, int H,
                int W, int Kv, int Kh, void* stream) {
  if (!c || !in || !ver || !hor || !out || N < 1 || C < 1 || H < 1 || W < 1 || Kv < 1 || Kh < 1)
    return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  LAUNCH(launch_sepconv(in, ver, hor, out, N, C, H, W, Kv, Kh, (cudaStream_t)stream));
  return VFI_OK;
}

int vfi_adacof(vfi_ctx* c, const float* in, const float* weight, const float* offset_i, const float* offset_j, float* out, int N,
               int C, int Hin, int Win, int F, int dilation, int Ho, int Wo, void* stream) {
  if (!c || !in || !weight || !offset_i || !offset_j || !out || N < 1 || C < 1 || Ho < 1 || Wo < 1)
    return fail(VFI_E_INVALID, "bad argument");
  if (F < 1 || dilation < 1 || Hin - ((F - 1) * dilation + 1) != Ho - 1 || Win - ((F - 1) * dilation + 1) != Wo - 1)
    return fail(VFI_E_INVALID, "adacof: input size must be output size + (F - 1) * dilation (adacof.py:274-279)");
  CK(cudaSetDevice(c->device));
  CK(launch_adacof(in, weight, offset_i, offset_j, out, N, C, Hin, Win, F, dilation, Ho, Wo, static_cast<cudaStream_t>(stream)));
  c->launches += 1;
  return VFI_OK;
}

int vfi_edt_pass(vfi_ctx* c, const float* data, float* out, int bs, int h, int w, float diam2, void* stream) {
  if (!c || !data || !out || bs < 1 || h < 1 || w < 1) return fail(VFI_E_INVALID, "bad argument");
  CK(cudaSetDevice(c->device));
  CK(launch_edt_pass(data, out, bs, h, w, diam2, static_cast<cudaStream_t>(stream)));
  c->launches += 1;
  return VFI_OK;
}

int vfi_rife46_debug_layer(vfi_ctx* c, int block, int layer, const void* in, void* out, void* out_mask, int B, int H,
                           int W, int impl, void* stream) {
  if (!c || block < 0 || layer < 0 || !in || !out) return fail(VFI_E_INVALID, "bad argument");
  if (!c->loaded) return fail(VFI_E_STATE, "vfi_rife46_load has not been called");
  if (block >= num_blocks(c->arch) || layer > 11 || (layer == 11 && (c->arch != 426 || block + 1 >= num_blocks(c->arch))))
    return fail(VFI_E_INVALID, "no such block / layer in the loaded arch");
  CK(cudaSetDevice(c->device));
  const TapConvLayer& L = c->layers[block][layer];
  if (layer == 10) {
    if (!out_mask) return fail(VFI_E_INVALID, "lastconv needs out_mask");
    LAUNCH(launch_tapconv(L, c->op_type, in, nullptr, (float4*)out, (float*)out_mask, B, H, W, c->num_sms, impl == 1,
                          (cudaStream_t)stream));
  } else {
    LAUNCH(launch_tapconv(L, c->op_type, in, out, nullptr, nullptr, B, H, W, c->num_sms, impl == 1,
                          (cudaStream_t)stream));
  }
  return VFI_OK;
}

int vfi_rife46_debug_state(vfi_ctx* c, float* flow4_out, float* mask_out, int batch, int* Hp, int* Wp) {
  if (!c || !Hp || !Wp) return fail(VFI_E_INVALID, "null argument");
  CK(cudaSetDevice(c->device));
  CK(cudaDeviceSynchronize());
  *Hp = c->ws_Hp;
  *Wp = c->ws_Wp;
  if (!flow4_out && !mask_out) return VFI_OK;
  if (batch < 1 || batch > c->ws_B) return fail(VFI_E_INVALID, "batch larger than the last pass");
  // the full-resolution flow is implicit on the product path; materialise it for the caller
  const size_t n = (size_t)batch * c->ws_Hp * c->ws_Wp;
  CK(c->dbgF.ensure(n * sizeof(float4)));
  CK(c->dbgM.ensure(n * sizeof(float)));
  if (c->last_lo >= c->last_fs.n) {  // every level already folded into the dense planes (up-scaled last blocks)
    CK(cudaMemcpy(c->dbgF.p, c->flow.p, n * sizeof(float4), cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(c->dbgM.p, c->mask.p, n * sizeof(float), cudaMemcpyDeviceToDevice));
  } else {
    LAUNCH(launch_materialize(c->last_fs, c->last_lo, c->last_have_base ? (const float4*)c->flow.p : nullptr,
                              c->last_have_base ? (const float*)c->mask.p : nullptr, (float4*)c->dbgF.p,
                              (float*)c->dbgM.p, batch, c->ws_Hp, c->ws_Wp, 0));
  }
  CK(cudaDeviceSynchronize());
  if (flow4_out) CK(cudaMemcpy(flow4_out, c->dbgF.p, n * sizeof(float4), cudaMemcpyDeviceToDevice));
  if (mask_out) CK(cudaMemcpy(mask_out, c->dbgM.p, n * sizeof(float), cudaMemcpyDeviceToDevice));
  return VFI_OK;
}

int vfi_rife46_layer_plan(vfi_ctx* c, int block, int layer, int* stages, int* n_cta, int* nsplit, int* smem_bytes,
                          int64_t* macs_per_cell) {
  if (!c || block < 0 || layer < 0) return fail(VFI_E_INVALID, "bad argument");
  if (!c->loaded) return fail(VFI_E_STATE, "vfi_rife46_load has not been called");
  if (block >= num_blocks(c->arch) || layer > 11 || (layer == 11 && (c->arch != 426 || block + 1 >= num_blocks(c->arch))))
    return fail(VFI_E_INVALID, "no such block / layer in the loaded arch");
  const TapConvLayer& L = c->layers[block][layer];
  TapConvParams p{};
  const int st = tapconv_plan(L, &p);
  if (stages) *stages = st;
  if (n_cta) *n_cta = L.n_cta;
  if (nsplit) *nsplit = L.nsplit;
  if (smem_bytes) *smem_bytes = (int)p.smem_bytes;
  if (macs_per_cell) *macs_per_cell = (int64_t)L.ktotal16 * 16 * L.n_total;
  return VFI_OK;
}

}  // extern "C"
