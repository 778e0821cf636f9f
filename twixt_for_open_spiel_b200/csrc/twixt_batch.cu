// twixt_batch.cu -- host class TwixTBatch and the extern "C" ABI of
// include/twixt_b200.h.
//
// TwixTBatch owns the env records in HBM, a CUDA stream, a scratch arena used
// to stage host-side inputs/outputs, and the device counters.  It mirrors the
// open_spiel Game/State surface of the reference (twixt.h:31-146) one batched
// method per State method; the C functions at the bottom are thin wrappers
// that translate exceptions-free status codes and keep the last error text.
// There is no CPU implementation behind any of these calls.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/twixt_b200.h"
#include "twixt_engine.cuh"
#include "twixt_kernels.cuh"
#include "twixt_mcts.cuh"

namespace twixt {

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define TW_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t e_ = (expr);                                                               \
    if (e_ != cudaSuccess) return fail(TWIXT_ECUDA, "CUDA error %s at %s:%d (%s)",         \
                                       cudaGetErrorString(e_), __FILE__, __LINE__, #expr); \
  } while (0)

#define TW_TRY(expr)        \
  do {                      \
    int rc_ = (expr);       \
    if (rc_ != TWIXT_OK) return rc_; \
  } while (0)

bool is_device_pointer(const void* p) {
  cudaPointerAttributes attr;
  cudaError_t e = cudaPointerGetAttributes(&attr, p);
  if (e != cudaSuccess) {
    cudaGetLastError();  // unregistered host memory on old drivers: clear and treat as host
    return false;
  }
  return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
}

class DeviceGuard {
 public:
  explicit DeviceGuard(int device) : prev_(-1) {
    cudaGetDevice(&prev_);
    if (prev_ != device) cudaSetDevice(device);
    dev_ = device;
  }
  ~DeviceGuard() {
    if (prev_ >= 0 && prev_ != dev_) cudaSetDevice(prev_);
  }

 private:
  int prev_, dev_;
};

int fill_game_info(int n, twixt_game_info* out) {
  if (n < TWIXT_MIN_BOARD_SIZE || n > TWIXT_MAX_BOARD_SIZE)  // twixt.cc:139-144, same text
    return fail(TWIXT_EINVAL, "board_size out of range [%d..%d]: %d", TWIXT_MIN_BOARD_SIZE, TWIXT_MAX_BOARD_SIZE, n);
  if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  out->board_size = n;
  out->num_distinct_actions = n * n;
  out->num_players = 2;
  out->max_game_length = n * n - 4 + 1;
  out->obs_shape[0] = TWIXT_NUM_OBS_PLANES;
  out->obs_shape[1] = n;
  out->obs_shape[2] = n - 2;
  out->obs_size = TWIXT_NUM_OBS_PLANES * n * (n - 2);
  out->max_legal_actions = n * (n - 2);
  out->record_words = record_words(n);
  out->min_utility = -1.0;
  out->max_utility = 1.0;
  out->utility_sum = 0.0;
  return TWIXT_OK;
}

}  // namespace

// A host output/input that may live on either side of the bus.
struct Staged {
  void* user = nullptr;     // what the caller passed
  void* dev = nullptr;      // what the kernel uses
  void* pin = nullptr;      // host alias of `dev` when the small-transfer arena is used (see PinAlloc)
  size_t bytes = 0;
  bool host = false;
};

class TwixTBatch {
 public:
  TwixTBatch() = default;
  ~TwixTBatch() {
    DeviceGuard g(device_);
    if (stream_ != nullptr) cudaStreamSynchronize(stream_);
    if (records_ != nullptr) cudaFree(records_);
    if (d_stats_ != nullptr) cudaFree(d_stats_);
    if (playout_start_ != nullptr) cudaFree(playout_start_);
    if (pinned_ != nullptr) cudaFreeHost(pinned_);
    for (int k = 0; k < kSlots; ++k)
      if (slot_[k] != nullptr) cudaFree(slot_[k]);
    if (own_stream_ && stream_ != nullptr) cudaStreamDestroy(stream_);
  }

  int Init(int n, int64_t num_envs, int device, uint64_t seed) {
    twixt_game_info info;
    TW_TRY(fill_game_info(n, &info));
    if (num_envs <= 0) return fail(TWIXT_EINVAL, "num_envs must be positive: %lld", static_cast<long long>(num_envs));
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
      cudaGetLastError();
      return fail(TWIXT_ECUDA, "no CUDA device available (%s): libtwixt_b200 has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    }
    if (device < 0 || device >= ndev) return fail(TWIXT_EINVAL, "device %d out of range [0..%d)", device, ndev);
    cudaDeviceProp prop;
    TW_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
      return fail(TWIXT_ECUDA, "device %d is sm_%d%d; libtwixt_b200 is built for sm_100a only", device, prop.major,
                  prop.minor);
    n_ = n;
    num_envs_ = num_envs;
    device_ = device;
    seed_ = seed;
    rw_ = info.record_words;
    DeviceGuard g(device_);
    TW_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    own_stream_ = true;
    const size_t bytes = static_cast<size_t>(num_envs_) * rw_ * sizeof(uint32_t);
    e = cudaMalloc(&records_, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(TWIXT_ENOMEM, "cudaMalloc of %zu bytes for %lld envs failed: %s", bytes,
                  static_cast<long long>(num_envs_), cudaGetErrorString(e));
    }
    TW_CUDA(cudaMalloc(&d_stats_, sizeof(DeviceStats)));
    if (cudaHostAlloc(&pinned_, kPinBytes, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess ||
        cudaHostGetDevicePointer(&pinned_dev_, pinned_, 0) != cudaSuccess) {
      cudaGetLastError();  // no mapped memory on this system: every host transfer takes the staged path
      if (pinned_ != nullptr) cudaFreeHost(pinned_);
      pinned_ = pinned_dev_ = nullptr;
    }
    TW_CUDA(cudaMemsetAsync(d_stats_, 0, sizeof(DeviceStats), stream_));
    TW_CUDA(playout_setup());
    return Reset(0, num_envs_);
  }

  int n() const { return n_; }
  int64_t num_envs() const { return num_envs_; }
  int rw() const { return rw_; }
  int device() const { return device_; }
  const uint32_t* records() const { return records_; }
  cudaStream_t stream() const { return stream_; }

  int SetStream(cudaStream_t s) {
    DeviceGuard g(device_);
    TW_CUDA(cudaStreamSynchronize(stream_));
    if (own_stream_) cudaStreamDestroy(stream_);
    stream_ = s;
    own_stream_ = false;
    return TWIXT_OK;
  }
  int Synchronize() {
    DeviceGuard g(device_);
    TW_CUDA(cudaStreamSynchronize(stream_));
    return TWIXT_OK;
  }

  // One State step for an unbatched caller (see twixt_step in the header): apply (or reset, or nothing),
  // then player / terminal / returns / ascending legal actions of the resulting state, by ONE kernel launch
  // whose outputs land in the pinned arena.
  int Step(int64_t env, int32_t action, twixt_step_result* out, int64_t* out_legal) {
    TW_TRY(CheckRange(env, 1));
    if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
    if (action < TWIXT_STEP_RESET) return fail(TWIXT_EINVAL, "action %d: use an action >= 0, TWIXT_STEP_QUERY or TWIXT_STEP_RESET", action);
    DeviceGuard g(device_);
    ScratchReset();
    Staged res, legal;
    TW_TRY(StageOut(out, sizeof(twixt_step_result), &res, false));
    TW_TRY(StageOut(out_legal, static_cast<size_t>(n_) * (n_ - 2) * sizeof(int64_t), &legal, false));
    TW_CUDA(launch_step(rec(env), n_, action, static_cast<twixt_step_result*>(res.dev), static_cast<int64_t*>(legal.dev),
                        stream_));
    launches_ += 1;
    TW_TRY(Finish(&res));
    TW_TRY(Finish(&legal));
    if (!res.host && !legal.host) return TWIXT_OK;
    TW_TRY(Sync());
    if (res.host && out->status == 1) return fail(TWIXT_EILLEGAL, "Not a legal action: %d", action);  // twixt.h:96
    return TWIXT_OK;
  }
  void SetSeed(uint64_t seed) { seed_ = seed; }
  void SetStreamBase(uint64_t base) { stream_base_ = base; }

  int CheckRange(int64_t first, int64_t count) const {
    if (first < 0 || count < 0 || first + count > num_envs_)
      return fail(TWIXT_EINVAL, "env range [%lld, %lld) outside [0, %lld)", static_cast<long long>(first),
                  static_cast<long long>(first + count), static_cast<long long>(num_envs_));
    return TWIXT_OK;
  }

  int Reset(int64_t first, int64_t count) {
    TW_TRY(CheckRange(first, count));
    DeviceGuard g(device_);
    TW_CUDA(launch_reset(rec(first), count, n_, stream_));
    launches_ += count > 0;
    return TWIXT_OK;
  }

  int Clone(int64_t src_first, int64_t dst_first, int64_t count) {
    TW_TRY(CheckRange(src_first, count));
    TW_TRY(CheckRange(dst_first, count));
    if (count > 0 && src_first < dst_first + count && dst_first < src_first + count)
      return fail(TWIXT_EINVAL, "clone ranges overlap");
    DeviceGuard g(device_);
    TW_CUDA(launch_clone(rec(dst_first), rec(src_first), nullptr, count, n_, num_envs_, dst_first, d_stats_, stream_));
    launches_ += count > 0;
    return TWIXT_OK;
  }

  int CloneGather(const int64_t* src_ids, int64_t dst_first, int64_t count) {
    TW_TRY(CheckRange(dst_first, count));
    if (count == 0) return TWIXT_OK;
    if (src_ids == nullptr) return fail(TWIXT_EINVAL, "null src_ids");
    DeviceGuard g(device_);
    ScratchReset();
    Staged ids;
    TW_TRY(StageIn(src_ids, static_cast<size_t>(count) * sizeof(int64_t), &ids));
    if (ids.host) {
      for (int64_t i = 0; i < count; ++i) {
        const int64_t s = src_ids[i];
        if (s < 0 || s >= num_envs_) return fail(TWIXT_EINVAL, "src_ids[%lld] = %lld out of range", (long long)i, (long long)s);
        if (s >= dst_first && s < dst_first + count) return fail(TWIXT_EINVAL, "src_ids[%lld] lies in the destination range", (long long)i);
      }
    }
    // device-resident ids cannot be checked here: the kernel checks every id (it skips a bad one and reports
    // the lowest offending position), and the flag is read back before the call returns
    TW_CUDA(cudaMemsetAsync(&d_stats_->bad_clone_index, 0xFF, sizeof(unsigned int), stream_));
    TW_CUDA(launch_clone(rec(dst_first), records_, static_cast<const int64_t*>(ids.dev), count, n_, num_envs_,
                         dst_first, d_stats_, stream_));
    launches_ += 1;
    unsigned int bad = 0xFFFFFFFFu;
    TW_CUDA(cudaMemcpyAsync(&bad, &d_stats_->bad_clone_index, sizeof(bad), cudaMemcpyDeviceToHost, stream_));
    TW_TRY(Sync());
    if (bad != 0xFFFFFFFFu)
      return fail(TWIXT_EINVAL, "src_ids[%u] is out of range or lies in the destination range (that env was not copied)", bad);
    return TWIXT_OK;
  }

  int CloneFrom(int64_t dst_first, const TwixTBatch& src, int64_t src_first, int64_t count) {
    TW_TRY(CheckRange(dst_first, count));
    TW_TRY(src.CheckRange(src_first, count));
    if (src.n_ != n_) return fail(TWIXT_EINVAL, "board sizes differ: %d vs %d", src.n_, n_);
    if (count == 0) return TWIXT_OK;
    if (&src == this && src_first < dst_first + count && dst_first < src_first + count)
      return fail(TWIXT_EINVAL, "clone ranges overlap");
    DeviceGuard g(device_);
    const size_t bytes = static_cast<size_t>(count) * rw_ * sizeof(uint32_t);
    // order after the source batch's pending work
    if (src.stream_ != stream_) {
      DeviceGuard gs(src.device_);
      TW_CUDA(cudaStreamSynchronize(src.stream_));
    }
    TW_CUDA(cudaMemcpyAsync(rec(dst_first), src.records_ + src_first * src.rw_, bytes, cudaMemcpyDefault, stream_));
    return TWIXT_OK;
  }

  int LegalActions(int64_t first, int64_t count, void* out_actions, int elem_bytes, int64_t stride,
                   int32_t* out_counts) {
    TW_TRY(CheckRange(first, count));
    if (elem_bytes != 2 && elem_bytes != 4 && elem_bytes != 8)
      return fail(TWIXT_EINVAL, "elem_bytes must be 2, 4 or 8: %d", elem_bytes);
    if (out_actions != nullptr && stride < n_ * (n_ - 2))
      return fail(TWIXT_EINVAL, "stride %lld < max_legal_actions %d", static_cast<long long>(stride), n_ * (n_ - 2));
    if (count == 0) return TWIXT_OK;
    DeviceGuard g(device_);
    ScratchReset();
    Staged acts, cnts;
    TW_TRY(StageOut(out_actions, static_cast<size_t>(count) * stride * elem_bytes, &acts, /*preserve=*/true));
    TW_TRY(StageOut(out_counts, static_cast<size_t>(count) * sizeof(int32_t), &cnts, false));
    TW_CUDA(launch_legal_actions(rec(first), count, n_, acts.dev, elem_bytes, stride,
                                 static_cast<int32_t*>(cnts.dev), stream_));
    launches_ += 1;
    TW_TRY(Finish(&acts));
    TW_TRY(Finish(&cnts));
    return SyncIfHost(acts, cnts);
  }

  int LegalMask(int64_t first, int64_t count, uint8_t* out) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
    DeviceGuard g(device_);
    ScratchReset();
    Staged m;
    TW_TRY(StageOut(out, static_cast<size_t>(count) * n_ * n_, &m, false));
    TW_CUDA(launch_legal_mask(rec(first), count, n_, static_cast<uint8_t*>(m.dev), stream_));
    launches_ += 1;
    TW_TRY(Finish(&m));
    return SyncIfHost(m, m);
  }

  int Apply(int64_t first, int64_t count, const int32_t* actions, int32_t* out_status) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    if (actions == nullptr) return fail(TWIXT_EINVAL, "null actions pointer");
    DeviceGuard g(device_);
    ScratchReset();
    Staged in, st;
    TW_TRY(StageIn(actions, static_cast<size_t>(count) * sizeof(int32_t), &in));
    const size_t status_bytes = static_cast<size_t>(count) * sizeof(int32_t);
    if (out_status == nullptr) PinAlloc(status_bytes, &st);  // small batches: statuses into the arena, read below
    else TW_TRY(StageOut(out_status, status_bytes, &st, false));
    // Where the statuses end up in host-visible memory the first illegal action is found by reading them;
    // otherwise the kernel's device-side flag is reset, and read back after the launch.
    const bool scan_host = st.pin != nullptr;
    if (!scan_host) TW_CUDA(cudaMemsetAsync(&d_stats_->illegal_index, 0xFF, sizeof(unsigned int), stream_));
    TW_CUDA(launch_apply(rec(first), count, n_, static_cast<const int32_t*>(in.dev), static_cast<int32_t*>(st.dev),
                         d_stats_, stream_));
    launches_ += 1;
    TW_TRY(Finish(&st));
    if (out_status != nullptr && !st.host) return TWIXT_OK;  // fully asynchronous: caller inspects the statuses
    int64_t bad = -1;
    if (scan_host) {
      TW_TRY(Sync());
      const int32_t* seen = static_cast<const int32_t*>(st.pin);
      for (int64_t i = 0; i < count && bad < 0; ++i)
        if (seen[i] == 1) bad = i;
    } else {
      unsigned int flag = 0xFFFFFFFFu;
      TW_CUDA(cudaMemcpyAsync(&flag, &d_stats_->illegal_index, sizeof(flag), cudaMemcpyDeviceToHost, stream_));
      TW_TRY(Sync());
      if (flag != 0xFFFFFFFFu) bad = flag;
    }
    if (bad >= 0) {
      int32_t a = 0;
      if (in.host) a = actions[bad];
      else TW_CUDA(cudaMemcpy(&a, actions + bad, sizeof(a), cudaMemcpyDeviceToHost));
      return fail(TWIXT_EILLEGAL, "Not a legal action: %d", a);  // twixt.h:96, same text
    }
    return TWIXT_OK;
  }

  int Query(int64_t first, int64_t count, int8_t* player, uint8_t* terminal, float* returns) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    DeviceGuard g(device_);
    ScratchReset();
    Staged p, t, r;
    TW_TRY(StageOut(player, static_cast<size_t>(count), &p, false));
    TW_TRY(StageOut(terminal, static_cast<size_t>(count), &t, false));
    TW_TRY(StageOut(returns, static_cast<size_t>(count) * 2 * sizeof(float), &r, false));
    TW_CUDA(launch_query(rec(first), count, n_, static_cast<int8_t*>(p.dev), static_cast<uint8_t*>(t.dev),
                         static_cast<float*>(r.dev), stream_));
    launches_ += 1;
    TW_TRY(Finish(&p));
    TW_TRY(Finish(&t));
    TW_TRY(Finish(&r));
    if (p.host || t.host || r.host) TW_TRY(Sync());
    return TWIXT_OK;
  }

  // out_mask != nullptr: the fused producer (tensor + legal mask in one pass over the records)
  int Observation(int64_t first, int64_t count, float* out, uint8_t* out_mask) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
    DeviceGuard g(device_);
    ScratchReset();
    Staged o, m;
    TW_TRY(StageOut(out, static_cast<size_t>(count) * 12 * n_ * (n_ - 2) * sizeof(float), &o, false));
    TW_TRY(StageOut(out_mask, static_cast<size_t>(count) * n_ * n_, &m, false));
    TW_CUDA(launch_observation(rec(first), count, n_, static_cast<float*>(o.dev), static_cast<uint8_t*>(m.dev),
                               stream_));
    launches_ += 1;
    TW_TRY(Finish(&o));
    TW_TRY(Finish(&m));
    return SyncIfHost(o, m);
  }

  int Replay(int64_t first, int64_t count, const int32_t* actions, int64_t stride, const int32_t* lengths,
             int32_t* out_applied) {
    TW_TRY(CheckRange(first, count));
    if (stride < 0) return fail(TWIXT_EINVAL, "stride must be >= 0");
    if (count == 0) return TWIXT_OK;
    if (actions == nullptr && stride > 0) return fail(TWIXT_EINVAL, "null actions pointer");
    DeviceGuard g(device_);
    ScratchReset();
    Staged in, len, ap;
    TW_TRY(StageIn(actions, static_cast<size_t>(count) * stride * sizeof(int32_t), &in));
    TW_TRY(StageIn(lengths, static_cast<size_t>(count) * sizeof(int32_t), &len));
    TW_TRY(StageOut(out_applied, static_cast<size_t>(count) * sizeof(int32_t), &ap, false));
    TW_CUDA(cudaMemsetAsync(&d_stats_->replay_illegal, 0xFF, sizeof(unsigned long long), stream_));
    TW_CUDA(launch_replay(rec(first), count, n_, static_cast<const int32_t*>(in.dev), stride,
                          static_cast<const int32_t*>(len.dev), static_cast<int32_t*>(ap.dev), d_stats_, stream_));
    launches_ += 1;
    TW_TRY(Finish(&ap));
    if (out_applied != nullptr && !ap.host && !in.host && !len.host) return TWIXT_OK;  // asynchronous: caller inspects out_applied
    unsigned long long bad = ~0ull;
    TW_CUDA(cudaMemcpyAsync(&bad, &d_stats_->replay_illegal, sizeof(bad), cudaMemcpyDeviceToHost, stream_));
    TW_TRY(Sync());
    if (bad != ~0ull)  // twixt.h:96, same text
      return fail(TWIXT_EILLEGAL, "Not a legal action: %d", static_cast<int>(static_cast<int32_t>(bad & 0xFFFFFFFFull)));
    return TWIXT_OK;
  }

  int Playout(int64_t first, int64_t count, int32_t max_plies, const uint64_t* stream_ids, float* out_returns,
              int32_t* out_lengths, uint16_t* out_actions, int32_t trace_plies) {
    TW_TRY(CheckRange(first, count));
    if (max_plies < 0) return fail(TWIXT_EINVAL, "max_plies must be >= 0");
    if (out_actions != nullptr && trace_plies <= 0) return fail(TWIXT_EINVAL, "trace_plies must be positive with out_actions");
    if (count == 0) return TWIXT_OK;
    DeviceGuard g(device_);
    ScratchReset();
    Staged ids, ret, len, act;
    TW_TRY(StageIn(stream_ids, static_cast<size_t>(count) * sizeof(uint64_t), &ids));
    TW_TRY(StageOut(out_returns, static_cast<size_t>(count) * 2 * sizeof(float), &ret, false));
    TW_TRY(StageOut(out_lengths, static_cast<size_t>(count) * sizeof(int32_t), &len, false));
    const size_t trace_bytes = out_actions ? static_cast<size_t>(trace_plies) * count * sizeof(uint16_t) : 0;
    TW_TRY(StageOut(out_actions, trace_bytes, &act, false));
    if (act.dev != nullptr) TW_CUDA(cudaMemsetAsync(act.dev, 0xFF, trace_bytes, stream_));
    PlayoutArgs a;
    a.records = rec(first);
    a.count = count;
    a.n = n_;
    a.max_plies = max_plies;
    a.seed = seed_;
    a.stream_base = stream_base_ + static_cast<uint64_t>(first);
    a.stream_ids = static_cast<const uint64_t*>(ids.dev);
    a.out_returns = static_cast<float*>(ret.dev);
    a.out_lengths = static_cast<int32_t*>(len.dev);
    a.out_actions = static_cast<uint16_t*>(act.dev);
    a.trace_plies = out_actions ? trace_plies : 0;
    a.stats = d_stats_;
    a.tickets = &d_stats_->tickets;
    const bool derive = n_ >= kPlayoutDeriveMinN;
    a.start = nullptr;
    if (derive) TW_TRY(PlayoutStart(count, &a.start));
    TW_CUDA(cudaMemsetAsync(&d_stats_->tickets, 0, sizeof(unsigned long long), stream_));
    TW_CUDA(launch_playout(a, stream_));  // the playout kernel (+ the blocked-plane pass)
    launches_ += derive ? 2 : 1;
    TW_TRY(Finish(&ret));
    TW_TRY(Finish(&len));
    TW_TRY(Finish(&act));
    if (ids.host || ret.host || len.host || act.host) TW_TRY(Sync());
    return TWIXT_OK;
  }

  int Export(int64_t first, int64_t count, uint32_t* out) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
    DeviceGuard g(device_);
    ScratchReset();
    const bool dev = is_device_pointer(out);
    TW_CUDA(cudaMemcpyAsync(out, rec(first), static_cast<size_t>(count) * rw_ * sizeof(uint32_t), cudaMemcpyDefault,
                            stream_));
    if (!dev) TW_TRY(Sync());
    return TWIXT_OK;
  }

  // Records from the caller are validated BEFORE they replace any env (validate_kernel,
  // twixt_kernels_api.cu): a host array is staged in device scratch and checked there, a device array is
  // checked where it lies; only then are the records copied in.  On failure the batch is untouched.
  int Import(int64_t first, int64_t count, const uint32_t* in) {
    TW_TRY(CheckRange(first, count));
    if (count == 0) return TWIXT_OK;
    if (in == nullptr) return fail(TWIXT_EINVAL, "null input pointer");
    DeviceGuard g(device_);
    const size_t bytes = static_cast<size_t>(count) * rw_ * sizeof(uint32_t);
    ScratchReset();
    if (!validate_) {  // twixt_set_validation(b, 0): trusted records (e.g. our own exports)
      const bool dev = is_device_pointer(in);
      TW_CUDA(cudaMemcpyAsync(rec(first), in, bytes, cudaMemcpyDefault, stream_));
      if (!dev) TW_TRY(Sync());
      return TWIXT_OK;
    }
    Staged src;
    TW_TRY(StageIn(in, bytes, &src));
    TW_CUDA(cudaMemsetAsync(&d_stats_->invalid_code, 0xFF, sizeof(unsigned long long), stream_));
    TW_CUDA(launch_validate(static_cast<const uint32_t*>(src.dev), count, n_, d_stats_, stream_));
    launches_ += 1;
    unsigned long long code = ~0ull;
    TW_CUDA(cudaMemcpyAsync(&code, &d_stats_->invalid_code, sizeof(code), cudaMemcpyDeviceToHost, stream_));
    TW_TRY(Sync());
    if (code != ~0ull)
      return fail(TWIXT_EINVAL, "invalid state record at index %lld: %s", static_cast<long long>(code >> 8),
                  invalid_reason_text(static_cast<unsigned>(code & 0xFFull)));
    TW_CUDA(cudaMemcpyAsync(rec(first), src.dev, bytes, cudaMemcpyDeviceToDevice, stream_));
    if (src.host) TW_TRY(Sync());
    return TWIXT_OK;
  }
  void SetValidation(bool on) { validate_ = on; }

  int GetStats(twixt_stats* out) {
    if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
    DeviceGuard g(device_);
    ScratchReset();
    DeviceStats h;
    TW_CUDA(cudaMemcpyAsync(&h, d_stats_, sizeof(h), cudaMemcpyDeviceToHost, stream_));
    TW_TRY(Sync());
    out->plies = static_cast<int64_t>(h.plies);
    out->games = static_cast<int64_t>(h.games);
    out->red_wins = static_cast<int64_t>(h.red_wins);
    out->blue_wins = static_cast<int64_t>(h.blue_wins);
    out->draws = static_cast<int64_t>(h.draws);
    out->swaps = static_cast<int64_t>(h.swaps);
    out->max_length = static_cast<int64_t>(h.max_length);
    out->kernel_launches = launches_;
    out->debug_violations = static_cast<int64_t>(h.bounds_violations);
    return TWIXT_OK;
  }

  int ResetStats() {
    DeviceGuard g(device_);
    TW_CUDA(cudaMemsetAsync(d_stats_, 0, sizeof(DeviceStats), stream_));
    return TWIXT_OK;
  }

 private:
  friend class TwixTMCTS;  // searches run on the batch's stream, staging, counters and Philox key
  uint32_t* rec(int64_t env) const { return records_ + env * rw_; }

  // ---- device staging for host-side buffers: a few grow-only slots ------
  void ScratchReset() {
    next_slot_ = 0;
    pin_off_ = 0;
    num_pending_ = 0;
  }

  // Small host-side transfers (the count = 1 calls of a drop-in adapter: a status word, a 4 KB legal list, a
  // 25 KB tensor) go through a pinned, device-mapped arena instead of a device slot + cudaMemcpyAsync: the
  // kernel reads / writes the host memory directly and the call costs one launch and one stream
  // synchronisation.  Returns false when the request does not fit (the caller then uses a device slot).
  bool PinAlloc(size_t bytes, Staged* s) {
    const size_t need = (bytes + 255) & ~static_cast<size_t>(255);
    if (pinned_ == nullptr || bytes > kPinMaxTransfer || pin_off_ + need > kPinBytes || num_pending_ >= kMaxPending)
      return false;
    s->pin = static_cast<char*>(pinned_) + pin_off_;
    s->dev = static_cast<char*>(pinned_dev_) + pin_off_;
    pin_off_ += need;
    return true;
  }

  // stream synchronisation + delivery of what kernels wrote into the pinned arena
  int Sync() {
    TW_CUDA(cudaStreamSynchronize(stream_));
    for (int i = 0; i < num_pending_; ++i) memcpy(pending_[i].user, pending_[i].pin, pending_[i].bytes);
    num_pending_ = 0;
    return TWIXT_OK;
  }

  // the playout's scratch for the blocked-plane pass (PlayoutArgs::start), grown to `count` envs
  int PlayoutStart(int64_t count, uint32_t** out) {
    const size_t bytes = static_cast<size_t>(playout_scratch_words(count, n_)) * sizeof(uint32_t);
    if (bytes > playout_start_cap_) {
      TW_CUDA(cudaStreamSynchronize(stream_));
      if (playout_start_ != nullptr) cudaFree(playout_start_);
      playout_start_ = nullptr;
      playout_start_cap_ = 0;
      cudaError_t e = cudaMalloc(&playout_start_, bytes);
      if (e != cudaSuccess) {
        cudaGetLastError();
        playout_start_ = nullptr;
        return fail(TWIXT_ENOMEM, "cudaMalloc of %zu playout scratch bytes failed: %s", bytes, cudaGetErrorString(e));
      }
      playout_start_cap_ = bytes;
    }
    *out = playout_start_;
    return TWIXT_OK;
  }

  int SlotAlloc(size_t bytes, void** out) {
    if (next_slot_ >= kSlots) return fail(TWIXT_ENOMEM, "internal: out of staging slots");
    const int k = next_slot_++;
    if (bytes > slot_cap_[k]) {
      TW_CUDA(cudaStreamSynchronize(stream_));
      if (slot_[k] != nullptr) cudaFree(slot_[k]);
      slot_[k] = nullptr;
      slot_cap_[k] = 0;
      const size_t want = bytes + (bytes >> 2) + 4096;
      cudaError_t e = cudaMalloc(&slot_[k], want);
      if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(TWIXT_ENOMEM, "cudaMalloc of %zu staging bytes failed: %s", want, cudaGetErrorString(e));
      }
      slot_cap_[k] = want;
    }
    *out = slot_[k];
    return TWIXT_OK;
  }

  int StageIn(const void* user, size_t bytes, Staged* s) {
    s->user = const_cast<void*>(user);
    s->bytes = bytes;
    if (user == nullptr || bytes == 0) { s->dev = nullptr; s->host = false; return TWIXT_OK; }
    if (is_device_pointer(user)) { s->dev = s->user; s->host = false; return TWIXT_OK; }
    s->host = true;
    if (PinAlloc(bytes, s)) {
      memcpy(s->pin, user, bytes);  // visible to the kernel: written before its launch
      return TWIXT_OK;
    }
    TW_TRY(SlotAlloc(bytes, &s->dev));
    TW_CUDA(cudaMemcpyAsync(s->dev, user, bytes, cudaMemcpyHostToDevice, stream_));
    return TWIXT_OK;
  }

  int StageOut(void* user, size_t bytes, Staged* s, bool preserve) {
    s->user = user;
    s->bytes = bytes;
    if (user == nullptr || bytes == 0) { s->dev = nullptr; s->host = false; return TWIXT_OK; }
    if (is_device_pointer(user)) { s->dev = user; s->host = false; return TWIXT_OK; }
    s->host = true;
    if (PinAlloc(bytes, s)) {
      if (preserve) memcpy(s->pin, user, bytes);
      return TWIXT_OK;
    }
    TW_TRY(SlotAlloc(bytes, &s->dev));
    if (preserve) TW_CUDA(cudaMemcpyAsync(s->dev, user, bytes, cudaMemcpyHostToDevice, stream_));
    return TWIXT_OK;
  }

  int Finish(Staged* s) {
    if (s->host && s->pin != nullptr) {
      pending_[num_pending_++] = {s->user, s->pin, s->bytes};  // copied out by Sync()
      return TWIXT_OK;
    }
    if (s->host && s->dev != nullptr)
      TW_CUDA(cudaMemcpyAsync(s->user, s->dev, s->bytes, cudaMemcpyDeviceToHost, stream_));
    return TWIXT_OK;
  }

  int SyncIfHost(const Staged& a, const Staged& b) {
    if (a.host || b.host) TW_TRY(Sync());
    return TWIXT_OK;
  }

  int n_ = 0;
  int rw_ = 0;
  int device_ = 0;
  int64_t num_envs_ = 0;
  uint64_t seed_ = 0;
  uint64_t stream_base_ = 0;
  bool validate_ = true;
  uint32_t* records_ = nullptr;
  DeviceStats* d_stats_ = nullptr;
  uint32_t* playout_start_ = nullptr;  // see PlayoutStart
  size_t playout_start_cap_ = 0;
  cudaStream_t stream_ = nullptr;
  bool own_stream_ = false;
  // pinned, device-mapped arena for small host transfers
  static constexpr size_t kPinBytes = 256 * 1024, kPinMaxTransfer = 96 * 1024;
  static constexpr int kMaxPending = 8;
  struct Pending {
    void* user;
    void* pin;
    size_t bytes;
  };
  void* pinned_ = nullptr;
  void* pinned_dev_ = nullptr;
  size_t pin_off_ = 0;
  Pending pending_[kMaxPending];
  int num_pending_ = 0;
  static constexpr int kSlots = 4;
  void* slot_[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  size_t slot_cap_[kSlots] = {0, 0, 0, 0};
  int next_slot_ = 0;
  int64_t launches_ = 0;
};

// Batched MCTS over the envs of one batch (twixt_mcts_* in the header; kernels in twixt_mcts.cu, storage
// formula in twixt_mcts.cuh).  Every call is queued on the batch's stream; the rollouts are twixt_playout's
// kernel on the search's own rollout slots and count in the batch's twixt_stats.
class TwixTMCTS {
 public:
  TwixTMCTS() = default;
  ~TwixTMCTS() {
    if (arena_mem_ == nullptr) return;
    DeviceGuard g(b_->device_);
    if (log_grown_ != nullptr) cudaFreeAsync(log_grown_, b_->stream_);
    cudaStreamSynchronize(b_->stream_);
    cudaFree(arena_mem_);
    if (map_ != nullptr) cudaFree(map_);
  }

  // leaves_per_step K > 1: K descents per step with virtual loss vl (checked by the caller, twixt_mcts_create_parallel).
  // gumbel: a Gumbel AlphaZero search (puct, solve and K > 1 excluded by the caller, twixt_mcts_create_gumbel) with
  // max_considered >= 1 and c_visit, c_scale finite and >= 0.
  int Init(TwixTBatch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts, double uct_c, bool puct,
           bool solve, int32_t leaves_per_step, double virtual_loss, bool gumbel = false, int32_t max_considered = 0,
           double c_visit = 0.0, double c_scale = 0.0) {
    if (num_trees <= 0) return fail(TWIXT_EINVAL, "num_trees must be positive: %lld", static_cast<long long>(num_trees));
    if (max_simulations <= 0) return fail(TWIXT_EINVAL, "max_simulations must be positive: %d", max_simulations);
    if (n_rollouts <= 0) return fail(TWIXT_EINVAL, "n_rollouts must be positive: %d", n_rollouts);
    if (!std::isfinite(uct_c) || uct_c < 0.0) return fail(TWIXT_EINVAL, "uct_c must be finite and >= 0: %g", uct_c);
    if (static_cast<uint64_t>(max_simulations) * static_cast<uint64_t>(n_rollouts) >= (1ull << 32))
      return fail(TWIXT_EINVAL, "max_simulations * n_rollouts = %llu must be below 2^32 (rollout stream ids)",
                  static_cast<unsigned long long>(max_simulations) * static_cast<unsigned long long>(n_rollouts));
    b_ = b;
    num_trees_ = num_trees;
    max_sims_ = max_simulations;
    c_ = uct_c;
    const int n = b->n_;
    const int K = leaves_per_step;
    const MctsSizes s = mcts_sizes(n, max_simulations, n_rollouts);
    const int64_t cells = static_cast<int64_t>(n) * n;
    const int64_t per_tree =
        gumbel ? mcts_gumbel_bytes_per_tree(s, cells)
               : mcts_parallel_bytes_per_tree(s, solve ? mcts_solve_bytes_per_tree(s, puct)
                                                       : (puct ? mcts_puct_bytes_per_tree(s) : mcts_bytes_per_tree(s)),
                                              K);
    // Gumbel: the considered-visits table, rows m = 0 .. min(max_considered, M), max_simulations - 1 columns
    const int mc = gumbel ? static_cast<int>(max_considered < s.edges ? max_considered : s.edges) : 0;
    const int cols = gumbel ? max_simulations - 1 : 0;
    std::vector<int32_t> considered(gumbel ? static_cast<size_t>(mc + 1) * cols : 0);
    for (int m = 0; gumbel && m <= mc; ++m) mcts_considered_visits(m, cols, considered.data() + static_cast<size_t>(m) * cols);
    // carve one allocation; each array starts on a 256-byte boundary (priors and tie keys are PUCT's, the outcome
    // bytes PUCT's and the solver's, the root codes the solver's, the virtual counts those of K > 1: empty
    // otherwise).  Tree entries, paths and rollout slots are per leaf row: K per tree.
    const int64_t T = num_trees, nodes = T * s.slots, edges = nodes * s.edges, rows = T * K, rolls = rows * s.rollouts;
    const int64_t pe = puct ? edges : 0, oe = (puct || solve) ? edges : 0, rt = solve ? T : 0;
    const int64_t vn = K > 1 ? nodes : 0, ve = K > 1 ? edges : 0;
    const int64_t ge = gumbel ? edges : 0, gn = gumbel ? nodes : 0, gt = gumbel ? T * cells : 0;
    const int64_t sizes[23] = {nodes * s.rw * 4, nodes * 4, nodes * 4, edges * 2, edges * 4, edges * 8, edges * 4,
                               rows * 16, rows * s.path * 8, rolls * s.rw * 4, rolls * 8, rolls * 8, s.slots * 8,
                               pe * 4, pe * 4, oe, rt, vn * 2, ve * 2,
                               ge * 4, gn * 8, gt * 4, static_cast<int64_t>(considered.size()) * 4};
    int64_t offs[23], total = 0;
    for (int i = 0; i < 23; ++i) {
      offs[i] = total;
      total += (sizes[i] + 255) & ~static_cast<int64_t>(255);
    }
    DeviceGuard g(b->device_);
    size_t free_bytes = 0, total_bytes = 0;
    TW_CUDA(cudaMemGetInfo(&free_bytes, &total_bytes));
    if (gumbel && static_cast<uint64_t>(total) > free_bytes)
      return fail(TWIXT_ENOMEM,
                  "Gumbel MCTS arena of %lld bytes (%lld trees x %lld bytes per tree = S*(rw*4 + 16 + 22*M) + 16 + 8*P "
                  "+ R*(rw*4 + 16) + 4*n*n at n = %d, %d simulations, %d rollouts; plus a %lld-byte considered-visits "
                  "table) exceeds the %zu bytes free on device %d",
                  static_cast<long long>(total), static_cast<long long>(T), static_cast<long long>(per_tree), n,
                  max_simulations, n_rollouts, static_cast<long long>(considered.size() * 4), free_bytes, b->device_);
    if (static_cast<uint64_t>(total) > free_bytes)
      return fail(TWIXT_ENOMEM,
                  "MCTS arena of %lld bytes (%lld trees x %lld bytes per tree at n = %d, %d simulations, %d rollouts, "
                  "%d leaves per step) exceeds the %zu bytes free on device %d",
                  static_cast<long long>(total), static_cast<long long>(T), static_cast<long long>(per_tree), n,
                  max_simulations, n_rollouts, K, free_bytes, b->device_);
    cudaError_t e = cudaMalloc(&arena_mem_, static_cast<size_t>(total));
    if (e != cudaSuccess) {
      cudaGetLastError();
      arena_mem_ = nullptr;
      return fail(TWIXT_ENOMEM, "cudaMalloc of %lld bytes for the MCTS arena failed: %s", static_cast<long long>(total),
                  cudaGetErrorString(e));
    }
    char* base = static_cast<char*>(arena_mem_);
    a_.n = n;
    a_.rw = static_cast<int>(s.rw);
    a_.M = static_cast<int>(s.edges);
    a_.S = static_cast<int>(s.slots);
    a_.P = static_cast<int>(s.path);
    a_.R = n_rollouts;
    a_.node_rec = reinterpret_cast<uint32_t*>(base + offs[0]);
    a_.node_legal = reinterpret_cast<int32_t*>(base + offs[1]);
    a_.node_n = reinterpret_cast<uint32_t*>(base + offs[2]);
    a_.edge_action = reinterpret_cast<uint16_t*>(base + offs[3]);
    a_.edge_n = reinterpret_cast<uint32_t*>(base + offs[4]);
    a_.edge_w = reinterpret_cast<double*>(base + offs[5]);
    a_.edge_child = reinterpret_cast<int32_t*>(base + offs[6]);
    a_.tree = reinterpret_cast<int4*>(base + offs[7]);
    a_.path = reinterpret_cast<int2*>(base + offs[8]);
    a_.roll_rec = reinterpret_cast<uint32_t*>(base + offs[9]);
    a_.roll_ids = reinterpret_cast<uint64_t*>(base + offs[10]);
    a_.roll_ret = reinterpret_cast<float*>(base + offs[11]);
    double* table = reinterpret_cast<double*>(base + offs[12]);
    a_.log_table = table;
    a_.edge_p = puct ? reinterpret_cast<float*>(base + offs[13]) : nullptr;
    a_.edge_key = puct ? reinterpret_cast<uint32_t*>(base + offs[14]) : nullptr;
    a_.edge_out = (puct || solve) ? reinterpret_cast<uint8_t*>(base + offs[15]) : nullptr;
    a_.root_out = solve ? reinterpret_cast<uint8_t*>(base + offs[16]) : nullptr;
    a_.node_v = K > 1 ? reinterpret_cast<uint16_t*>(base + offs[17]) : nullptr;
    a_.edge_v = K > 1 ? reinterpret_cast<uint16_t*>(base + offs[18]) : nullptr;
    a_.K = K;
    a_.vl = virtual_loss;
    K_ = K;
    gumbel_ = gumbel;
    if (gumbel) {
      gm_.edge_logit = reinterpret_cast<float*>(base + offs[19]);
      gm_.node_value = reinterpret_cast<double*>(base + offs[20]);
      gm_.root_gumbel = reinterpret_cast<float*>(base + offs[21]);
      gm_.table = reinterpret_cast<const int32_t*>(base + offs[22]);
      gm_.max_considered = mc;
      gm_.cols = cols;
      gm_.c_visit = c_visit;
      gm_.c_scale = c_scale;
      if (!considered.empty())
        TW_CUDA(cudaMemcpyAsync(base + offs[22], considered.data(), considered.size() * sizeof(int32_t),
                                cudaMemcpyHostToDevice, b->stream_));
    }
    log_size_ = s.slots;
    // ln N(s) from the host's libm, so that a CPU restatement of the search computes the same scores
    std::vector<double> logs(static_cast<size_t>(s.slots));
    for (size_t i = 0; i < logs.size(); ++i) logs[i] = std::log(static_cast<double>(i));
    TW_CUDA(cudaMemcpyAsync(table, logs.data(), logs.size() * sizeof(double), cudaMemcpyHostToDevice, b->stream_));
    TW_CUDA(cudaStreamSynchronize(b->stream_));
    return TWIXT_OK;
  }

  int Begin(int64_t root_first, int64_t count) {
    TW_TRY(b_->CheckRange(root_first, count));
    if (count > num_trees_)
      return fail(TWIXT_EINVAL, "count %lld > num_trees %lld", static_cast<long long>(count),
                  static_cast<long long>(num_trees_));
    const uint64_t base = b_->stream_base_;
    if (count > 0 && (base >= (1ull << 32) || static_cast<uint64_t>(root_first + count - 1) >= (1ull << 32) - base))
      return fail(TWIXT_EINVAL, "tree stream ids stream_base + root_first + t must be below 2^32: base %llu, roots [%lld, %lld)",
                  static_cast<unsigned long long>(base), static_cast<long long>(root_first),
                  static_cast<long long>(root_first + count));
    DeviceGuard g(b_->device_);
    TW_CUDA(launch_mcts_begin(a_, b_->rec(root_first), count, b_->stream_));
    b_->launches_ += count > 0;
    if (gumbel_ && count > 0)  // g = 0 until twixt_mcts_set_root_gumbel
      TW_CUDA(cudaMemsetAsync(gm_.root_gumbel, 0, static_cast<size_t>(count) * a_.n * a_.n * sizeof(float),
                              b_->stream_));
    count_ = count;
    key_ = b_->seed_;
    stream0_ = static_cast<uint32_t>(base + static_cast<uint64_t>(root_first));
    sims_ = 0;
    node_bound_ = 1;
    advanced_ = false;
    pending_ = false;
    begun_ = true;
    return TWIXT_OK;
  }

  int Run(int32_t num_simulations) {
    TW_TRY(CheckSimulations(num_simulations, "run"));
    if (num_simulations % K_ != 0)
      return fail(TWIXT_EINVAL, "twixt_mcts_run: %d simulations is not a multiple of leaves_per_step %d",
                  num_simulations, K_);
    if (count_ == 0 || num_simulations == 0) return TWIXT_OK;
    DeviceGuard g(b_->device_);
    TW_TRY(GrowLogTable(num_simulations));
    TwixTBatch& b = *b_;
    PlayoutArgs p;
    p.records = a_.roll_rec;
    p.count = count_ * K_ * a_.R;
    p.n = a_.n;
    p.max_plies = a_.n * a_.n;  // above max_game_length: every rollout plays to the end
    p.seed = key_;
    p.stream_base = 0;
    p.stream_ids = a_.roll_ids;
    p.out_returns = a_.roll_ret;
    p.out_lengths = nullptr;
    p.out_actions = nullptr;
    p.trace_plies = 0;
    p.stats = b.d_stats_;
    p.tickets = &b.d_stats_->tickets;
    p.start = nullptr;  // rollout records are discarded after their returns are read: no blocked-plane pass
    for (int32_t i = 0; i < num_simulations; i += K_) {  // one step: K simulations of every tree
      const uint32_t k = static_cast<uint32_t>(sims_);
      if (gumbel_) TW_CUDA(launch_mcts_gumbel_select(a_, gm_, count_, stream0_, k, nullptr, nullptr, b.stream_));
      else TW_CUDA(launch_mcts_select(a_, count_, key_, stream0_, k, c_, nullptr, nullptr, b.stream_));
      TW_CUDA(cudaMemsetAsync(&b.d_stats_->tickets, 0, sizeof(unsigned long long), b.stream_));
      TW_CUDA(launch_playout(p, b.stream_));
      if (gumbel_) TW_CUDA(launch_mcts_gumbel_backup(a_, gm_, count_, nullptr, nullptr, b.stream_));
      else TW_CUDA(launch_mcts_backup(a_, count_, nullptr, nullptr, key_, stream0_, b.stream_));
      b.launches_ += 3;
      sims_ += K_;
      node_bound_ += K_;
    }
    return TWIXT_OK;
  }

  // K leaf rows per tree: row t*K + j goes to env leaf_first + t*K + j
  int Select(int64_t leaf_first, int32_t* out_leaf_status) {
    TW_TRY(CheckSimulations(K_, "select"));
    TW_TRY(b_->CheckRange(leaf_first, count_ * K_));
    if (count_ == 0) {
      pending_ = true;
      return TWIXT_OK;
    }
    DeviceGuard g(b_->device_);
    TW_TRY(GrowLogTable(K_));
    TwixTBatch& b = *b_;
    b.ScratchReset();
    Staged st;
    TW_TRY(b.StageOut(out_leaf_status, static_cast<size_t>(count_ * K_) * sizeof(int32_t), &st, false));
    if (gumbel_)
      TW_CUDA(launch_mcts_gumbel_select(a_, gm_, count_, stream0_, static_cast<uint32_t>(sims_), b.rec(leaf_first),
                                        static_cast<int32_t*>(st.dev), b.stream_));
    else
      TW_CUDA(launch_mcts_select(a_, count_, key_, stream0_, static_cast<uint32_t>(sims_), c_, b.rec(leaf_first),
                                 static_cast<int32_t*>(st.dev), b.stream_));
    b.launches_ += 1;
    pending_ = true;
    leaf_first_ = leaf_first;
    node_bound_ += K_;
    TW_TRY(b.Finish(&st));
    if (st.host) TW_TRY(b.Sync());
    return TWIXT_OK;
  }

  // values [count*K, 2], priors: [count*K, n*n] float32 or nullptr (uniform); host priors are checked before anything
  // is launched
  int Backup(const float* values, const float* priors) {
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_backup: no search begun");
    if (!pending_) return fail(TWIXT_EINVAL, "twixt_mcts_backup without a pending twixt_mcts_select");
    if (values == nullptr && count_ > 0) return fail(TWIXT_EINVAL, "null values pointer");
    if (priors != nullptr && a_.edge_p == nullptr && !gumbel_)
      return fail(TWIXT_EINVAL, "twixt_mcts_backup_priors: priors given to a UCT search (use twixt_mcts_create_puct)");
    const size_t cells = static_cast<size_t>(a_.n) * a_.n;
    if (gumbel_ && priors != nullptr && count_ > 0 && !is_device_pointer(priors)) {
      TW_TRY(CheckHostLogits(priors));
    } else if (priors != nullptr && count_ > 0 && !is_device_pointer(priors)) {
      const size_t total = static_cast<size_t>(count_ * K_) * cells;
      for (size_t i = 0; i < total; ++i)
        if (!std::isfinite(priors[i]) || priors[i] < 0.0f)
          return fail(TWIXT_EINVAL, "prior [%lld, %lld] = %g: priors must be finite and >= 0",
                      static_cast<long long>(i / cells), static_cast<long long>(i % cells),
                      static_cast<double>(priors[i]));
    }
    if (count_ > 0) {
      DeviceGuard g(b_->device_);
      TwixTBatch& b = *b_;
      b.ScratchReset();
      Staged in, pin;
      const size_t rows = static_cast<size_t>(count_ * K_);
      TW_TRY(b.StageIn(values, rows * 2 * sizeof(float), &in));
      TW_TRY(b.StageIn(priors, priors != nullptr ? rows * cells * sizeof(float) : 0, &pin));
      if (gumbel_)
        TW_CUDA(launch_mcts_gumbel_backup(a_, gm_, count_, static_cast<const float*>(in.dev),
                                          static_cast<const float*>(pin.dev), b.stream_));
      else
        TW_CUDA(launch_mcts_backup(a_, count_, static_cast<const float*>(in.dev), static_cast<const float*>(pin.dev),
                                   key_, stream0_, b.stream_));
      b.launches_ += 1;
      if (in.host || pin.host) TW_TRY(b.Sync());  // the staged copies are reused by the next call
    }
    pending_ = false;
    sims_ += K_;
    return TWIXT_OK;
  }

  int RootStats(int32_t* out_visits, double* out_value_sums, int32_t* out_best) {
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_root_stats: no search begun");
    if (count_ == 0) return TWIXT_OK;
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    b.ScratchReset();
    const size_t cells = static_cast<size_t>(a_.n) * a_.n;
    Staged v, w, best;
    TW_TRY(b.StageOut(out_visits, static_cast<size_t>(count_) * cells * sizeof(int32_t), &v, false));
    TW_TRY(b.StageOut(out_value_sums, static_cast<size_t>(count_) * cells * sizeof(double), &w, false));
    TW_TRY(b.StageOut(out_best, static_cast<size_t>(count_) * sizeof(int32_t), &best, false));
    if (gumbel_) {  // visits and value sums as for every kind; the best action is the Gumbel action
      if (v.dev != nullptr || w.dev != nullptr) {
        TW_CUDA(launch_mcts_root_stats(a_, count_, static_cast<int32_t*>(v.dev), static_cast<double*>(w.dev), nullptr,
                                       b.stream_));
        b.launches_ += 1;
      }
      if (best.dev != nullptr) {
        TW_CUDA(launch_mcts_gumbel_stats(a_, gm_, count_, static_cast<int32_t*>(best.dev), nullptr, b.stream_));
        b.launches_ += 1;
      }
    } else {
      TW_CUDA(launch_mcts_root_stats(a_, count_, static_cast<int32_t*>(v.dev), static_cast<double*>(w.dev),
                                     static_cast<int32_t*>(best.dev), b.stream_));
      b.launches_ += 1;
    }
    TW_TRY(b.Finish(&v));
    TW_TRY(b.Finish(&w));
    TW_TRY(b.Finish(&best));
    if (v.host || w.host || best.host) TW_TRY(b.Sync());
    return TWIXT_OK;
  }

  // MCTS-Solver results of a solver search; every output nullable, host or device
  int SolverStats(uint8_t* out_proven, float* out_returns, int8_t* out_edge_values, int32_t* out_simulations) {
    if (a_.root_out == nullptr)
      return fail(TWIXT_EINVAL, "twixt_mcts_solver_stats: the search was not created with TWIXT_MCTS_SOLVE");
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_solver_stats: no search begun");
    if (pending_) return fail(TWIXT_EINVAL, "twixt_mcts_solver_stats while a twixt_mcts_select awaits its backup");
    if (count_ == 0) return TWIXT_OK;
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    b.ScratchReset();
    const size_t cells = static_cast<size_t>(a_.n) * a_.n, cnt = static_cast<size_t>(count_);
    Staged pr, re, ev, sm;
    TW_TRY(b.StageOut(out_proven, cnt, &pr, false));
    TW_TRY(b.StageOut(out_returns, cnt * 2 * sizeof(float), &re, false));
    TW_TRY(b.StageOut(out_edge_values, cnt * cells, &ev, false));
    TW_TRY(b.StageOut(out_simulations, cnt * sizeof(int32_t), &sm, false));
    TW_CUDA(launch_mcts_solver_stats(a_, count_, static_cast<uint8_t*>(pr.dev), static_cast<float*>(re.dev),
                                     static_cast<int8_t*>(ev.dev), static_cast<int32_t*>(sm.dev), b.stream_));
    b.launches_ += 1;
    TW_TRY(b.Finish(&pr));
    TW_TRY(b.Finish(&re));
    TW_TRY(b.Finish(&ev));
    TW_TRY(b.Finish(&sm));
    if (pr.host || re.host || ev.host || sm.host) TW_TRY(b.Sync());
    return TWIXT_OK;
  }

  // Tree reuse: actions [count] int32 (host or device), 1 <= keep_nodes <= S, out_status [count] int32 or nullptr.
  // Illegal actions are reported as twixt_apply reports them: TWIXT_EILLEGAL naming the first one, except with
  // device statuses, where the call returns at once and the caller reads the statuses.
  int Advance(const int32_t* actions, int32_t keep_nodes, int32_t* out_status) {
    if (gumbel_)
      return fail(TWIXT_EINVAL, "twixt_mcts_advance: a Gumbel search does not reuse trees (Sequential Halving needs a "
                                "fresh root); begin it again");
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_advance: no search begun");
    if (pending_) return fail(TWIXT_EINVAL, "twixt_mcts_advance while a twixt_mcts_select awaits its backup");
    if (keep_nodes < 1 || keep_nodes > a_.S)
      return fail(TWIXT_EINVAL, "keep_nodes must be in [1, max_simulations + 1 = %d]: %d", a_.S, keep_nodes);
    if (count_ == 0) return TWIXT_OK;
    if (actions == nullptr) return fail(TWIXT_EINVAL, "null actions pointer");
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    if (map_ == nullptr) {  // old -> new slot map, [num_trees, S] int32, allocated at the first advance
      const size_t bytes = static_cast<size_t>(num_trees_) * a_.S * sizeof(int32_t);
      cudaError_t e = cudaMalloc(&map_, bytes);
      if (e != cudaSuccess) {
        cudaGetLastError();
        map_ = nullptr;
        return fail(TWIXT_ENOMEM, "cudaMalloc of %zu bytes for the twixt_mcts_advance slot map failed: %s", bytes,
                    cudaGetErrorString(e));
      }
    }
    b.ScratchReset();
    Staged in, st;
    TW_TRY(b.StageIn(actions, static_cast<size_t>(count_) * sizeof(int32_t), &in));
    const size_t status_bytes = static_cast<size_t>(count_) * sizeof(int32_t);
    if (out_status == nullptr) b.PinAlloc(status_bytes, &st);  // as twixt_apply: statuses read below
    else TW_TRY(b.StageOut(out_status, status_bytes, &st, false));
    const bool scan_host = st.pin != nullptr;
    if (!scan_host) TW_CUDA(cudaMemsetAsync(&b.d_stats_->illegal_index, 0xFF, sizeof(unsigned int), b.stream_));
    TW_CUDA(launch_mcts_advance(a_, count_, static_cast<const int32_t*>(in.dev), keep_nodes, map_,
                                static_cast<int32_t*>(st.dev), &b.d_stats_->illegal_index, b.stream_));
    b.launches_ += 1;
    advanced_ = true;
    TW_TRY(b.Finish(&st));
    // every tree now holds at most min(keep_nodes, bound) nodes, except one whose action was illegal (unchanged);
    // device statuses are the caller's to read, who must begin again after an illegal one
    const int64_t truncated = keep_nodes < node_bound_ ? keep_nodes : node_bound_;
    if (out_status != nullptr && !st.host) {
      node_bound_ = truncated;
      if (in.host) TW_TRY(b.Sync());  // the staged actions are reused by the next call
      return TWIXT_OK;
    }
    int64_t bad = -1;
    if (scan_host) {
      TW_TRY(b.Sync());
      const int32_t* seen = static_cast<const int32_t*>(st.pin);
      for (int64_t i = 0; i < count_ && bad < 0; ++i)
        if (seen[i] == kRootIllegal) bad = i;
    } else {
      unsigned int flag = 0xFFFFFFFFu;
      TW_CUDA(cudaMemcpyAsync(&flag, &b.d_stats_->illegal_index, sizeof(flag), cudaMemcpyDeviceToHost, b.stream_));
      TW_TRY(b.Sync());
      if (flag != 0xFFFFFFFFu) bad = flag;
    }
    if (bad >= 0) {
      int32_t act = 0;
      if (in.host) act = actions[bad];
      else TW_CUDA(cudaMemcpy(&act, actions + bad, sizeof(act), cudaMemcpyDeviceToHost));
      return fail(TWIXT_EILLEGAL, "Not a legal action: %d", act);  // twixt.h:96, as twixt_apply
    }
    node_bound_ = truncated;
    return TWIXT_OK;
  }

  // PUCT searches: P(a) of every root edge of the trees whose root is expanded, from priors [count, n*n]
  int SetRootPriors(const float* priors) {
    if (gumbel_)
      return fail(TWIXT_EINVAL, "twixt_mcts_set_root_priors: a Gumbel search takes its root logits at its first backup "
                                "and its root noise from twixt_mcts_set_root_gumbel");
    if (a_.edge_p == nullptr)
      return fail(TWIXT_EINVAL, "twixt_mcts_set_root_priors: the search is not a PUCT search");
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_set_root_priors: no search begun");
    if (pending_)
      return fail(TWIXT_EINVAL, "twixt_mcts_set_root_priors while a twixt_mcts_select awaits its backup");
    if (count_ == 0) return TWIXT_OK;
    if (priors == nullptr) return fail(TWIXT_EINVAL, "null priors pointer");
    const size_t cells = static_cast<size_t>(a_.n) * a_.n;
    if (!is_device_pointer(priors)) {
      const size_t total = static_cast<size_t>(count_) * cells;
      for (size_t i = 0; i < total; ++i)
        if (!std::isfinite(priors[i]) || priors[i] < 0.0f)
          return fail(TWIXT_EINVAL, "prior [%lld, %lld] = %g: priors must be finite and >= 0",
                      static_cast<long long>(i / cells), static_cast<long long>(i % cells),
                      static_cast<double>(priors[i]));
    }
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    b.ScratchReset();
    Staged pin;
    TW_TRY(b.StageIn(priors, static_cast<size_t>(count_) * cells * sizeof(float), &pin));
    TW_CUDA(launch_mcts_set_root_priors(a_, count_, static_cast<const float*>(pin.dev), b.stream_));
    b.launches_ += 1;
    if (pin.host) TW_TRY(b.Sync());  // the staged copy is reused by the next call
    return TWIXT_OK;
  }

  // Gumbel searches: the root noise g [count, n*n] float32 (host or device; host values must be finite)
  int SetRootGumbel(const float* gumbel) {
    if (!gumbel_) return fail(TWIXT_EINVAL, "twixt_mcts_set_root_gumbel: the search is not a Gumbel search");
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_set_root_gumbel: no search begun");
    if (pending_) return fail(TWIXT_EINVAL, "twixt_mcts_set_root_gumbel while a twixt_mcts_select awaits its backup");
    if (count_ == 0) return TWIXT_OK;
    if (gumbel == nullptr) return fail(TWIXT_EINVAL, "null gumbel pointer");
    const size_t cells = static_cast<size_t>(a_.n) * a_.n, total = static_cast<size_t>(count_) * cells;
    if (!is_device_pointer(gumbel))
      for (size_t i = 0; i < total; ++i)
        if (!std::isfinite(gumbel[i]))
          return fail(TWIXT_EINVAL, "gumbel [%lld, %lld] = %g: the root noise must be finite",
                      static_cast<long long>(i / cells), static_cast<long long>(i % cells),
                      static_cast<double>(gumbel[i]));
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    b.ScratchReset();
    Staged in;
    TW_TRY(b.StageIn(gumbel, total * sizeof(float), &in));
    TW_CUDA(launch_mcts_set_root_gumbel(a_, gm_, count_, static_cast<const float*>(in.dev), b.stream_));
    b.launches_ += 1;
    if (in.host) TW_TRY(b.Sync());  // the staged copy is reused by the next call
    return TWIXT_OK;
  }

  // Gumbel searches: the action [count] int32 and the improved policy [count, n*n] float32; each nullable, host or
  // device
  int GumbelStats(int32_t* out_action, float* out_policy) {
    if (!gumbel_) return fail(TWIXT_EINVAL, "twixt_mcts_gumbel_stats: the search is not a Gumbel search");
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_gumbel_stats: no search begun");
    if (pending_) return fail(TWIXT_EINVAL, "twixt_mcts_gumbel_stats while a twixt_mcts_select awaits its backup");
    if (count_ == 0) return TWIXT_OK;
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    b.ScratchReset();
    const size_t cells = static_cast<size_t>(a_.n) * a_.n, cnt = static_cast<size_t>(count_);
    Staged ac, po;
    TW_TRY(b.StageOut(out_action, cnt * sizeof(int32_t), &ac, false));
    TW_TRY(b.StageOut(out_policy, cnt * cells * sizeof(float), &po, false));
    TW_CUDA(launch_mcts_gumbel_stats(a_, gm_, count_, static_cast<int32_t*>(ac.dev), static_cast<float*>(po.dev),
                                     b.stream_));
    b.launches_ += 1;
    TW_TRY(b.Finish(&ac));
    TW_TRY(b.Finish(&po));
    if (ac.host || po.host) TW_TRY(b.Sync());
    return TWIXT_OK;
  }

  int64_t count() const { return count_; }
  int64_t simulations() const { return sims_; }

 private:
  // Host logits of a Gumbel backup must be finite on the legal actions of every non-terminal leaf: the leaf records
  // select wrote to envs [leaf_first_, leaf_first_ + count) are read back and their legal lists computed here.
  int CheckHostLogits(const float* logits) {
    DeviceGuard g(b_->device_);
    TwixTBatch& b = *b_;
    const int n = a_.n, rw = a_.rw;
    const size_t cells = static_cast<size_t>(n) * n;
    std::vector<uint32_t> recs(static_cast<size_t>(count_) * rw);
    TW_CUDA(cudaMemcpyAsync(recs.data(), b.rec(leaf_first_), recs.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                            b.stream_));
    TW_TRY(b.Sync());
    for (int64_t t = 0; t < count_; ++t) {
      uint32_t* rec = recs.data() + t * rw;
      Header h;
      unpack_header(rec[0], rec[1], rec[2], rec[3], h);
      if (h.result != kOpen) continue;
      RecordRef<1> rb{rec, n};
      for (int x = 0; x < n; ++x)
        for (uint32_t w = legal_word(rb, h, x); w != 0u; w &= w - 1u) {
          const int a = x * n + tw_ctz(w);
          const float l = logits[t * cells + a];
          if (!std::isfinite(l))
            return fail(TWIXT_EINVAL, "logit [%lld, %d] = %g: logits must be finite on the leaf's legal actions",
                        static_cast<long long>(t), a, static_cast<double>(l));
        }
    }
    return TWIXT_OK;
  }

  // The host's bound on a tree's node count (node_bound_: 1 after begin, min(keep_nodes, bound) after an advance,
  // +K per step) keeps every step inside the S node slots without reading the trees back.  Without an advance this
  // is "at most max_simulations simulations since begin".
  int CheckSimulations(int32_t num, const char* what) const {
    if (!begun_) return fail(TWIXT_EINVAL, "twixt_mcts_%s: no search begun", what);
    if (pending_) return fail(TWIXT_EINVAL, "twixt_mcts_%s while a twixt_mcts_select awaits its backup", what);
    if (num < 0) return fail(TWIXT_EINVAL, "num_simulations must be >= 0: %d", num);
    if (!advanced_ && sims_ + num > max_sims_)
      return fail(TWIXT_EINVAL, "%lld simulations since begin would exceed max_simulations %d",
                  static_cast<long long>(sims_ + num), max_sims_);
    if (advanced_ && node_bound_ + num > a_.S)
      return fail(TWIXT_EINVAL,
                  "twixt_mcts_%s: %d simulations on trees of up to %lld nodes since twixt_mcts_advance would exceed "
                  "the max_simulations + 1 = %d node slots of a tree (advance with a smaller keep_nodes)",
                  what, num, static_cast<long long>(node_bound_), a_.S);
    // the simulation counter k carries on across advances: k*R + r keys the rollout streams and must stay 32-bit
    if (static_cast<uint64_t>(sims_ + num) * static_cast<uint64_t>(a_.R) > (1ull << 32))
      return fail(TWIXT_EINVAL,
                  "twixt_mcts_%s: simulation counter %lld + %d times n_rollouts %d would reach 2^32 (rollout stream "
                  "ids); begin the search again",
                  what, static_cast<long long>(sims_), num, a_.R);
    return TWIXT_OK;
  }

  // ln N(s) for N(s) < sims_ + num: N(s) <= the simulations since begin, which outgrow the S entries of the arena's
  // table once advances keep trees.  A larger table is filled from the host's libm as at create, and the old one is
  // freed in stream order.
  int GrowLogTable(int32_t num) {
    const int64_t need = sims_ + num;
    if (need <= log_size_) return TWIXT_OK;
    const int64_t size = need > 2 * log_size_ ? need : 2 * log_size_;
    std::vector<double> logs(static_cast<size_t>(size));
    for (size_t i = 0; i < logs.size(); ++i) logs[i] = std::log(static_cast<double>(i));
    void* table = nullptr;
    cudaError_t e = cudaMallocAsync(&table, logs.size() * sizeof(double), b_->stream_);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(TWIXT_ENOMEM, "cudaMallocAsync of %zu bytes for the ln N(s) table failed: %s",
                  logs.size() * sizeof(double), cudaGetErrorString(e));
    }
    // pageable source: the copy has taken the data when it returns
    TW_CUDA(cudaMemcpyAsync(table, logs.data(), logs.size() * sizeof(double), cudaMemcpyHostToDevice, b_->stream_));
    if (log_grown_ != nullptr) TW_CUDA(cudaFreeAsync(log_grown_, b_->stream_));
    log_grown_ = static_cast<double*>(table);
    a_.log_table = log_grown_;
    log_size_ = size;
    return TWIXT_OK;
  }

  TwixTBatch* b_ = nullptr;
  void* arena_mem_ = nullptr;
  MctsArena a_{};
  int64_t num_trees_ = 0;
  int32_t max_sims_ = 0;
  int32_t K_ = 1;  // leaves per step
  double c_ = 0.0;
  int64_t count_ = 0;
  uint64_t key_ = 0;
  uint32_t stream0_ = 0;
  int64_t sims_ = 0;
  int64_t node_bound_ = 1;     // bound on every tree's node count (CheckSimulations)
  bool advanced_ = false;      // an advance since begin
  int32_t* map_ = nullptr;     // [num_trees, S] old -> new slots of twixt_mcts_advance
  double* log_grown_ = nullptr;  // the ln table once it outgrew the arena's
  int64_t log_size_ = 0;       // its entries
  bool pending_ = false;
  bool begun_ = false;
  bool gumbel_ = false;        // a Gumbel AlphaZero search (gm_ holds its arrays)
  MctsGumbel gm_{};
  int64_t leaf_first_ = 0;     // the leaf envs of the pending select (host logits are checked against them)
};

}  // namespace twixt

struct twixt_batch {
  twixt::TwixTBatch impl;
};

struct twixt_mcts {
  twixt::TwixTMCTS impl;
};

using twixt::fail;

extern "C" {

const char* twixt_last_error(void) { return twixt::g_last_error.c_str(); }
const char* twixt_version(void) { return "twixt_b200 0.1 (sm_100a)"; }

int twixt_game_info_for(int board_size, twixt_game_info* out) { return twixt::fill_game_info(board_size, out); }

int twixt_create(int board_size, int64_t num_envs, int device, uint64_t seed, twixt_batch** out) {
  if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  *out = nullptr;
  twixt_batch* b = new (std::nothrow) twixt_batch();
  if (b == nullptr) return fail(TWIXT_ENOMEM, "out of host memory");
  int rc = b->impl.Init(board_size, num_envs, device, seed);
  if (rc != TWIXT_OK) {
    std::string keep = twixt::g_last_error;
    delete b;
    twixt::g_last_error = keep;
    return rc;
  }
  *out = b;
  return TWIXT_OK;
}

void twixt_destroy(twixt_batch* b) { delete b; }

#define TW_NEED(b) \
  if ((b) == nullptr) return fail(TWIXT_EINVAL, "null batch handle")

int twixt_get_info(const twixt_batch* b, twixt_game_info* out) {
  TW_NEED(b);
  return twixt::fill_game_info(b->impl.n(), out);
}
int64_t twixt_num_envs(const twixt_batch* b) { return b ? b->impl.num_envs() : 0; }
int twixt_set_stream(twixt_batch* b, uintptr_t s) {
  TW_NEED(b);
  return b->impl.SetStream(reinterpret_cast<cudaStream_t>(s));
}
uintptr_t twixt_get_stream(const twixt_batch* b) { return b ? reinterpret_cast<uintptr_t>(b->impl.stream()) : 0; }
int twixt_synchronize(twixt_batch* b) {
  TW_NEED(b);
  return b->impl.Synchronize();
}
int twixt_set_seed(twixt_batch* b, uint64_t seed) {
  TW_NEED(b);
  b->impl.SetSeed(seed);
  return TWIXT_OK;
}
int twixt_set_stream_base(twixt_batch* b, uint64_t base) {
  TW_NEED(b);
  b->impl.SetStreamBase(base);
  return TWIXT_OK;
}
int twixt_reset(twixt_batch* b, int64_t first, int64_t count) {
  TW_NEED(b);
  return b->impl.Reset(first, count);
}
int twixt_clone(twixt_batch* b, int64_t src_first, int64_t dst_first, int64_t count) {
  TW_NEED(b);
  return b->impl.Clone(src_first, dst_first, count);
}
int twixt_clone_gather(twixt_batch* b, const int64_t* src_ids, int64_t dst_first, int64_t count) {
  TW_NEED(b);
  return b->impl.CloneGather(src_ids, dst_first, count);
}
int twixt_clone_from(twixt_batch* dst, int64_t dst_first, const twixt_batch* src, int64_t src_first, int64_t count) {
  TW_NEED(dst);
  TW_NEED(src);
  return dst->impl.CloneFrom(dst_first, src->impl, src_first, count);
}
int twixt_legal_actions(twixt_batch* b, int64_t first, int64_t count, void* out_actions, int32_t elem_bytes,
                        int64_t stride, int32_t* out_counts) {
  TW_NEED(b);
  return b->impl.LegalActions(first, count, out_actions, elem_bytes, stride, out_counts);
}
int twixt_legal_mask(twixt_batch* b, int64_t first, int64_t count, uint8_t* out_mask) {
  TW_NEED(b);
  return b->impl.LegalMask(first, count, out_mask);
}
int twixt_apply(twixt_batch* b, int64_t first, int64_t count, const int32_t* actions, int32_t* out_status) {
  TW_NEED(b);
  return b->impl.Apply(first, count, actions, out_status);
}
int twixt_current_player(twixt_batch* b, int64_t first, int64_t count, int8_t* out) {
  TW_NEED(b);
  return b->impl.Query(first, count, out, nullptr, nullptr);
}
int twixt_is_terminal(twixt_batch* b, int64_t first, int64_t count, uint8_t* out) {
  TW_NEED(b);
  return b->impl.Query(first, count, nullptr, out, nullptr);
}
int twixt_returns(twixt_batch* b, int64_t first, int64_t count, float* out) {
  TW_NEED(b);
  return b->impl.Query(first, count, nullptr, nullptr, out);
}
int twixt_observation(twixt_batch* b, int64_t first, int64_t count, float* out) {
  TW_NEED(b);
  return b->impl.Observation(first, count, out, nullptr);
}
int twixt_observation_and_mask(twixt_batch* b, int64_t first, int64_t count, float* out_obs, uint8_t* out_mask) {
  TW_NEED(b);
  if (out_mask == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  return b->impl.Observation(first, count, out_obs, out_mask);
}
int twixt_replay(twixt_batch* b, int64_t first, int64_t count, const int32_t* actions, int64_t stride,
                 const int32_t* lengths, int32_t* out_applied) {
  TW_NEED(b);
  return b->impl.Replay(first, count, actions, stride, lengths, out_applied);
}
int twixt_step(twixt_batch* b, int64_t env, int32_t action, twixt_step_result* out, int64_t* out_legal) {
  TW_NEED(b);
  return b->impl.Step(env, action, out, out_legal);
}
int twixt_set_validation(twixt_batch* b, int enabled) {
  TW_NEED(b);
  b->impl.SetValidation(enabled != 0);
  return TWIXT_OK;
}
int twixt_playout(twixt_batch* b, int64_t first, int64_t count, int32_t max_plies, const uint64_t* stream_ids,
                  float* out_returns, int32_t* out_lengths, uint16_t* out_actions, int32_t trace_plies) {
  TW_NEED(b);
  return b->impl.Playout(first, count, max_plies, stream_ids, out_returns, out_lengths, out_actions, trace_plies);
}
int twixt_export_state(twixt_batch* b, int64_t first, int64_t count, uint32_t* out_records) {
  TW_NEED(b);
  return b->impl.Export(first, count, out_records);
}
int twixt_import_state(twixt_batch* b, int64_t first, int64_t count, const uint32_t* records) {
  TW_NEED(b);
  return b->impl.Import(first, count, records);
}
// ---- multi-GPU helpers for a host that is not Python (twixt_for_open_spiel_b200/sharding.py restated) ----
int twixt_shard_range(int64_t global_envs, int32_t world, int32_t rank, int64_t* out_first, int64_t* out_count) {
  if (world < 1 || rank < 0 || rank >= world || global_envs < 0)
    return fail(TWIXT_EINVAL, "bad shard arguments: %lld envs, world %d, rank %d", static_cast<long long>(global_envs),
                world, rank);
  if (out_first == nullptr || out_count == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  const int64_t base = global_envs / world, extra = global_envs % world;
  *out_first = rank * base + (rank < extra ? rank : extra);
  *out_count = base + (rank < extra ? 1 : 0);
  return TWIXT_OK;
}
int twixt_stats_accumulate(twixt_stats* acc, const twixt_stats* part) {
  if (acc == nullptr || part == nullptr) return fail(TWIXT_EINVAL, "null pointer");
  acc->plies += part->plies;
  acc->games += part->games;
  acc->red_wins += part->red_wins;
  acc->blue_wins += part->blue_wins;
  acc->draws += part->draws;
  acc->swaps += part->swaps;
  acc->kernel_launches += part->kernel_launches;
  if (part->max_length > acc->max_length) acc->max_length = part->max_length;
  return TWIXT_OK;
}

// ---- batched MCTS (class TwixTMCTS above, kernels in twixt_mcts.cu) ----
#define TW_NEED_MCTS(m) \
  if ((m) == nullptr) return fail(TWIXT_EINVAL, "null mcts handle")

static int mcts_create(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                       double uct_c, uint32_t flags, int32_t leaves_per_step, double virtual_loss, twixt_mcts** out) {
  TW_NEED(b);
  if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  *out = nullptr;
  if ((flags & ~static_cast<uint32_t>(TWIXT_MCTS_PUCT | TWIXT_MCTS_SOLVE)) != 0u)
    return fail(TWIXT_EINVAL, "unknown twixt_mcts_create_ex flags 0x%x", flags);
  const bool puct = (flags & TWIXT_MCTS_PUCT) != 0u, solve = (flags & TWIXT_MCTS_SOLVE) != 0u;
  if (leaves_per_step < 1 || leaves_per_step > 4096)
    return fail(TWIXT_EINVAL, "leaves_per_step must be in [1, 4096]: %d", leaves_per_step);
  if (leaves_per_step > 1 && leaves_per_step > max_simulations)
    return fail(TWIXT_EINVAL, "leaves_per_step %d exceeds max_simulations %d", leaves_per_step, max_simulations);
  if (!std::isfinite(virtual_loss) || virtual_loss < 0.0)
    return fail(TWIXT_EINVAL, "virtual_loss must be finite and >= 0: %g", virtual_loss);
  if (solve && leaves_per_step > 1)
    return fail(TWIXT_EINVAL, "TWIXT_MCTS_SOLVE runs one leaf per step: leaves_per_step %d", leaves_per_step);
  twixt_mcts* m = new (std::nothrow) twixt_mcts();
  if (m == nullptr) return fail(TWIXT_ENOMEM, "out of host memory");
  int rc = m->impl.Init(&b->impl, num_trees, max_simulations, n_rollouts, uct_c, puct, solve, leaves_per_step,
                        virtual_loss);
  if (rc != TWIXT_OK) {
    std::string keep = twixt::g_last_error;
    delete m;
    twixt::g_last_error = keep;
    return rc;
  }
  *out = m;
  return TWIXT_OK;
}
int twixt_mcts_create(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts, double uct_c,
                      twixt_mcts** out) {
  return mcts_create(b, num_trees, max_simulations, n_rollouts, uct_c, 0u, 1, 0.0, out);
}
int twixt_mcts_create_puct(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                           double uct_c, twixt_mcts** out) {
  return mcts_create(b, num_trees, max_simulations, n_rollouts, uct_c, TWIXT_MCTS_PUCT, 1, 0.0, out);
}
int twixt_mcts_create_ex(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                         double uct_c, uint32_t flags, twixt_mcts** out) {
  return mcts_create(b, num_trees, max_simulations, n_rollouts, uct_c, flags, 1, 0.0, out);
}
int twixt_mcts_create_parallel(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                               double uct_c, uint32_t flags, int32_t leaves_per_step, double virtual_loss,
                               twixt_mcts** out) {
  return mcts_create(b, num_trees, max_simulations, n_rollouts, uct_c, flags, leaves_per_step, virtual_loss, out);
}
void twixt_mcts_destroy(twixt_mcts* m) { delete m; }
int twixt_mcts_begin(twixt_mcts* m, int64_t root_first, int64_t count) {
  TW_NEED_MCTS(m);
  return m->impl.Begin(root_first, count);
}
int twixt_mcts_run(twixt_mcts* m, int32_t num_simulations) {
  TW_NEED_MCTS(m);
  return m->impl.Run(num_simulations);
}
int twixt_mcts_select(twixt_mcts* m, int64_t leaf_first, int32_t* out_leaf_status) {
  TW_NEED_MCTS(m);
  return m->impl.Select(leaf_first, out_leaf_status);
}
int twixt_mcts_backup(twixt_mcts* m, const float* values) {
  TW_NEED_MCTS(m);
  return m->impl.Backup(values, nullptr);
}
int twixt_mcts_backup_priors(twixt_mcts* m, const float* values, const float* priors) {
  TW_NEED_MCTS(m);
  return m->impl.Backup(values, priors);
}
int twixt_mcts_root_stats(twixt_mcts* m, int32_t* out_visits, double* out_value_sums, int32_t* out_best) {
  TW_NEED_MCTS(m);
  return m->impl.RootStats(out_visits, out_value_sums, out_best);
}
int twixt_mcts_solver_stats(twixt_mcts* m, uint8_t* out_proven, float* out_returns, int8_t* out_edge_values,
                            int32_t* out_simulations) {
  TW_NEED_MCTS(m);
  return m->impl.SolverStats(out_proven, out_returns, out_edge_values, out_simulations);
}
int twixt_mcts_advance(twixt_mcts* m, const int32_t* actions, int32_t keep_nodes, int32_t* out_status) {
  TW_NEED_MCTS(m);
  return m->impl.Advance(actions, keep_nodes, out_status);
}
int twixt_mcts_set_root_priors(twixt_mcts* m, const float* priors) {
  TW_NEED_MCTS(m);
  return m->impl.SetRootPriors(priors);
}
int twixt_mcts_create_gumbel(twixt_batch* b, int64_t num_trees, int32_t max_simulations, int32_t n_rollouts,
                             int32_t max_considered, double c_visit, double c_scale, twixt_mcts** out) {
  TW_NEED(b);
  if (out == nullptr) return fail(TWIXT_EINVAL, "null output pointer");
  *out = nullptr;
  if (max_considered < 1) return fail(TWIXT_EINVAL, "max_considered must be >= 1: %d", max_considered);
  if (!std::isfinite(c_visit) || c_visit < 0.0)
    return fail(TWIXT_EINVAL, "c_visit must be finite and >= 0: %g", c_visit);
  if (!std::isfinite(c_scale) || c_scale < 0.0)
    return fail(TWIXT_EINVAL, "c_scale must be finite and >= 0: %g", c_scale);
  twixt_mcts* m = new (std::nothrow) twixt_mcts();
  if (m == nullptr) return fail(TWIXT_ENOMEM, "out of host memory");
  int rc = m->impl.Init(&b->impl, num_trees, max_simulations, n_rollouts, 0.0, false, false, 1, 0.0, true,
                        max_considered, c_visit, c_scale);
  if (rc != TWIXT_OK) {
    std::string keep = twixt::g_last_error;
    delete m;
    twixt::g_last_error = keep;
    return rc;
  }
  *out = m;
  return TWIXT_OK;
}
int twixt_mcts_set_root_gumbel(twixt_mcts* m, const float* gumbel) {
  TW_NEED_MCTS(m);
  return m->impl.SetRootGumbel(gumbel);
}
int twixt_mcts_gumbel_stats(twixt_mcts* m, int32_t* out_action, float* out_policy) {
  TW_NEED_MCTS(m);
  return m->impl.GumbelStats(out_action, out_policy);
}

int twixt_get_stats(twixt_batch* b, twixt_stats* out) {
  TW_NEED(b);
  return b->impl.GetStats(out);
}
int twixt_stats_reset(twixt_batch* b) {
  TW_NEED(b);
  return b->impl.ResetStats();
}

}  // extern "C"
