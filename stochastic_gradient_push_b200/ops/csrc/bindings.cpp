// Python bindings + native runtime for the gossip data plane.
//
//  * SymmetricBuffer: cudaMalloc'd, IPC-exportable device memory wrapped as a
//    torch tensor; peers open it with cudaIpcOpenMemHandle and read it with
//    plain loads over NVLink/NVSwitch (one rendezvous replaces the reference's
//    O(world * schedule) two-rank process groups, gossip/graph_manager.py:27).
//  * GossipContext: owns the SgpArgs block for one (parameter arena, peer
//    table, schedule) triple and launches the kernels on the current stream.
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <thread>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "sgp_common.cuh"

namespace py = pybind11;

// every kernel of this extension is launched through one of the two CHECK macros; they count
// the launches (expressions that call a *_launch_* entry point) so that bench.py can report how
// many of OUR kernels one captured training step contains (`launch_count()` delta over a capture)
std::atomic<long long> g_sgp_kernel_launches{0};

#define SGP_CUDA_CHECK(expr)                                                        \
    do {                                                                            \
        if (std::strstr(#expr, "_launch_") != nullptr) ++g_sgp_kernel_launches;     \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess)                                                      \
            throw std::runtime_error(std::string(#expr) + " failed: " +             \
                                     cudaGetErrorString(_e));                       \
    } while (0)

// ---------------------------------------------------------------------------
// symmetric memory
// ---------------------------------------------------------------------------
static py::tuple symm_alloc(int64_t nbytes, int device)
{
    c10::cuda::CUDAGuard guard(device);
    void* ptr = nullptr;
    // round up to 2 MiB so the allocation owns whole pages (IPC exports pages)
    const int64_t gran = 2ll << 20;
    const int64_t padded = (nbytes + gran - 1) / gran * gran;
    SGP_CUDA_CHECK(cudaMalloc(&ptr, padded));
    SGP_CUDA_CHECK(cudaMemset(ptr, 0, padded));
    SGP_CUDA_CHECK(cudaDeviceSynchronize());
    cudaIpcMemHandle_t handle;
    std::string hbytes;
    cudaError_t e = cudaIpcGetMemHandle(&handle, ptr);
    if (e == cudaSuccess) {
        hbytes.assign(reinterpret_cast<const char*>(&handle), sizeof(handle));
    } else {
        (void)cudaGetLastError();   // single-process use still works without IPC
    }
    auto opts = torch::TensorOptions().dtype(torch::kUInt8).device(torch::kCUDA, device);
    auto t = torch::from_blob(ptr, {nbytes}, [device](void* p) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(device);
        cudaFree(p);
        cudaSetDevice(cur);
    }, opts);
    return py::make_tuple(t, py::bytes(hbytes));
}

static torch::Tensor symm_open(const std::string& hbytes, int64_t nbytes, int device)
{
    if (hbytes.size() != sizeof(cudaIpcMemHandle_t))
        throw std::runtime_error("symm_open: bad IPC handle size");
    c10::cuda::CUDAGuard guard(device);
    cudaIpcMemHandle_t handle;
    std::memcpy(&handle, hbytes.data(), sizeof(handle));
    void* ptr = nullptr;
    SGP_CUDA_CHECK(cudaIpcOpenMemHandle(&ptr, handle, cudaIpcMemLazyEnablePeerAccess));
    auto opts = torch::TensorOptions().dtype(torch::kUInt8).device(torch::kCUDA, device);
    return torch::from_blob(ptr, {nbytes}, [device](void* p) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(device);
        cudaIpcCloseMemHandle(p);
        cudaSetDevice(cur);
    }, opts);
}

// same-process peer (one process driving several GPUs, or loop-back tests)
static bool enable_peer_access(int device, int peer)
{
    if (device == peer) return true;
    c10::cuda::CUDAGuard guard(device);
    int can = 0;
    SGP_CUDA_CHECK(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can) return false;
    cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { (void)cudaGetLastError(); return true; }
    SGP_CUDA_CHECK(e);
    return true;
}

// pinned host word the probe kernel can write (AD-PSGD passive poll)
static torch::Tensor pinned_flag()
{
    return torch::zeros({16}, torch::TensorOptions().dtype(torch::kInt32).pinned_memory(true));
}

// ---------------------------------------------------------------------------
// GossipContext
// ---------------------------------------------------------------------------
class GossipContext {
public:
    GossipContext(torch::Tensor z, c10::optional<torch::Tensor> g, c10::optional<torch::Tensor> m,
                  c10::optional<torch::Tensor> shadow, c10::optional<torch::Tensor> residual,
                  torch::Tensor pad_ptrs, c10::optional<torch::Tensor> outbox_ptrs,
                  torch::Tensor table, torch::Tensor wtable, int rank, int world,
                  torch::Tensor state, torch::Tensor hyper, double timeout_s)
    {
        TORCH_CHECK(z.is_cuda() && z.scalar_type() == torch::kFloat32 && z.is_contiguous(),
                    "z must be a contiguous fp32 CUDA tensor");
        TORCH_CHECK(z.numel() % SGP_CHUNK == 0, "arena length must be a multiple of ", SGP_CHUNK);
        TORCH_CHECK(world >= 1 && world <= SGP_MAX_RANKS, "world size out of range");
        TORCH_CHECK(table.scalar_type() == torch::kInt32 && table.size(1) == SGP_TABLE_ROW);
        TORCH_CHECK(wtable.scalar_type() == torch::kFloat32 && wtable.size(1) == SGP_WTABLE_ROW);
        TORCH_CHECK(table.size(0) == wtable.size(0));
        TORCH_CHECK(pad_ptrs.scalar_type() == torch::kInt64 && pad_ptrs.numel() == world);
        TORCH_CHECK(state.numel() * state.element_size() >= (int64_t)sizeof(SgpState));
        TORCH_CHECK(hyper.numel() * hyper.element_size() >= (int64_t)sizeof(SgpHyper));
        device_ = z.get_device();
        std::memset(&args_, 0, sizeof(args_));
        args_.z = z.data_ptr<float>();
        args_.n = z.numel();
        keep_.push_back(z);
        if (g.has_value() && g->defined()) {
            TORCH_CHECK(g->numel() == z.numel() && g->is_contiguous());
            TORCH_CHECK(g->scalar_type() == torch::kFloat32 || g->scalar_type() == torch::kBFloat16);
            args_.g = g->data_ptr();
            grad_bf16_ = g->scalar_type() == torch::kBFloat16;
            keep_.push_back(*g);
        }
        if (m.has_value() && m->defined()) {
            TORCH_CHECK(m->numel() == z.numel() && m->scalar_type() == torch::kFloat32);
            args_.m = m->data_ptr<float>();
            keep_.push_back(*m);
        }
        if (shadow.has_value() && shadow->defined()) {
            TORCH_CHECK(shadow->numel() == z.numel() && shadow->scalar_type() == torch::kBFloat16);
            args_.shadow = reinterpret_cast<__nv_bfloat16*>(shadow->data_ptr());
            keep_.push_back(*shadow);
        }
        if (residual.has_value() && residual->defined()) {
            TORCH_CHECK(residual->numel() == z.numel() && residual->scalar_type() == torch::kFloat32);
            args_.residual = residual->data_ptr<float>();
            keep_.push_back(*residual);
        }
        args_.pads = reinterpret_cast<SgpSignalPad* const*>(pad_ptrs.data_ptr<int64_t>());
        keep_.push_back(pad_ptrs);
        if (outbox_ptrs.has_value() && outbox_ptrs->defined()) {
            TORCH_CHECK(outbox_ptrs->scalar_type() == torch::kInt64 && outbox_ptrs->numel() == world);
            args_.outboxes = reinterpret_cast<float* const*>(outbox_ptrs->data_ptr<int64_t>());
            keep_.push_back(*outbox_ptrs);
        }
        set_schedule(table, wtable);
        args_.rank = rank;
        args_.world = world;
        args_.st = reinterpret_cast<SgpState*>(state.data_ptr());
        args_.hyper = reinterpret_cast<const SgpHyper*>(hyper.data_ptr());
        args_.timeout_ns = (unsigned long long)(timeout_s * 1e9);
        keep_.push_back(state);
        keep_.push_back(hyper);
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_preload_kernels());      // no first launch may wait for a spinning kernel
        max_grid_ = sgp_max_resident_ctas(device_);
        // the warp-specialised TMA step kernel (default for the full SGP / D-PSGD step) is bound by
        // its dynamic shared memory; the grid has to be co-resident for BOTH kernels because the
        // ranks of a job may mix them (flags are matched by CTA index)
        const int pipe_grid = sgp_max_resident_ctas_pipe(device_);
        if (pipe_grid > 0 && (max_grid_ == 0 || pipe_grid < max_grid_)) max_grid_ = pipe_grid;
        const char* env = std::getenv("SGP_B200_PIPE");
        use_pipe_ = !(env && env[0] == '0');
        args_.segments = 4;
    }

    void set_schedule(torch::Tensor table, torch::Tensor wtable)
    {
        TORCH_CHECK(table.is_cuda() && wtable.is_cuda() && table.is_contiguous() && wtable.is_contiguous());
        args_.table = table.data_ptr<int>();
        args_.wtable = wtable.data_ptr<float>();
        args_.period = (int)table.size(0);
        sched_keep_ = {table, wtable};
    }

    void set_grad(torch::Tensor g)
    {
        TORCH_CHECK(g.numel() == args_.n && g.is_contiguous());
        TORCH_CHECK(g.scalar_type() == torch::kFloat32 || g.scalar_type() == torch::kBFloat16);
        args_.g = g.data_ptr();
        grad_bf16_ = g.scalar_type() == torch::kBFloat16;
        grad_keep_ = g;
    }

    void set_grad2(c10::optional<torch::Tensor> g2)
    {
        if (g2.has_value() && g2->defined()) {
            TORCH_CHECK(g2->numel() == args_.n && g2->scalar_type() == torch::kFloat32 && g2->is_contiguous());
            args_.g2 = g2->data_ptr<float>();
            grad2_keep_ = *g2;
        } else {
            args_.g2 = nullptr;
            grad2_keep_ = torch::Tensor();
        }
    }

    void set_sgd_buffers(torch::Tensor g, torch::Tensor m)
    {
        set_grad(g);
        TORCH_CHECK(m.numel() == args_.n && m.scalar_type() == torch::kFloat32 && m.is_contiguous());
        args_.m = m.data_ptr<float>();
        mom_keep_ = m;
    }

    int max_grid() const { return max_grid_; }

    void step(unsigned int flags, int grid)
    {
        check_grid(grid);
        SgpArgs a = prepare(flags);
        if (a.flags & SGP_F_SGD) TORCH_CHECK(a.g && a.m, "SGD needs grad + momentum buffers");
        if (a.flags & SGP_F_FOLD_RES) TORCH_CHECK(a.residual, "fold needs a residual buffer");
        if (a.flags & SGP_F_PUBLISH) TORCH_CHECK(a.outboxes, "publish needs outboxes");
        if (a.flags & SGP_F_PHASE2) TORCH_CHECK(a.flags & SGP_F_PUBLISH, "phase 2 needs publish");
        c10::cuda::CUDAGuard guard(device_);
        const unsigned int full = SGP_F_PHASE1 | SGP_F_PUBLISH | SGP_F_PHASE2;
        const unsigned int not_piped = SGP_F_FOLD_RES | SGP_F_NO_ROTATE | SGP_F_KEEP_Z | SGP_F_SELF_FROM_Z;
        if (use_pipe_ && (a.flags & full) == full && (a.flags & not_piped) == 0)
            SGP_CUDA_CHECK(sgp_launch_step_pipe(&a, grid, at::cuda::getCurrentCUDAStream()));
        else
            SGP_CUDA_CHECK(sgp_launch_step(&a, grid, at::cuda::getCurrentCUDAStream()));
    }

    // ---- AD-PSGD building blocks (all stream-ordered, no host decisions) ----
    void bilat_decide(int pub_grid, bool passive, double max_wait_us, c10::optional<torch::Tensor> host_fb)
    {
        SgpArgs a = prepare(0);
        uint32_t* fb = nullptr;
        if (host_fb.has_value() && host_fb->defined()) {
            void* dev = nullptr;
            SGP_CUDA_CHECK(cudaHostGetDevicePointer(&dev, host_fb->data_ptr(), 0));
            fb = reinterpret_cast<uint32_t*>(dev);
        }
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_bilat_decide(&a, pub_grid, passive ? 1 : 0,
                                               (unsigned long long)(max_wait_us * 1e3), fb,
                                               at::cuda::getCurrentCUDAStream()));
    }
    void bilat_work(int grid)
    {
        check_grid(grid);
        SgpArgs a = prepare(SGP_F_FROM_STATE | (args_.shadow ? SGP_F_SHADOW : 0u));
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_step(&a, grid, at::cuda::getCurrentCUDAStream()));
    }
    void bilat_ctl(int budget, int enabled)
    {
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_bilat_ctl(args_.st, budget, enabled, at::cuda::getCurrentCUDAStream()));
    }
    // raw access for the native gossip daemon
    SgpArgs raw_args(unsigned int flags) const { return prepare(flags); }
    int device() const { return device_; }

    void set_pipe(bool on) { use_pipe_ = on; }
    bool pipe() const { return use_pipe_; }

    void gather(int grid, int pub_grid, bool tma)
    {
        check_grid(grid);
        SgpArgs a = prepare(0);
        TORCH_CHECK(a.residual && a.outboxes);
        c10::cuda::CUDAGuard guard(device_);
        if (tma)
            SGP_CUDA_CHECK(sgp_launch_gather_tma(&a, grid, pub_grid, at::cuda::getCurrentCUDAStream()));
        else
            SGP_CUDA_CHECK(sgp_launch_gather(&a, grid, pub_grid, at::cuda::getCurrentCUDAStream()));
    }

    // Overlap-SGP gather on the copy engines: flag wait (1 CTA) -> cudaMemcpyAsync(peer outbox ->
    // residual) -> ack (1 thread).  `src_ptr`: address of the in-neighbour's outbox half of this step.
    void gather_dma(int pub_grid, int64_t src_ptr)
    {
        SgpArgs a = prepare(0);
        TORCH_CHECK(a.residual && a.outboxes && src_ptr != 0);
        c10::cuda::CUDAGuard guard(device_);
        auto st = at::cuda::getCurrentCUDAStream();
        SGP_CUDA_CHECK(sgp_launch_gather_wait(&a, pub_grid, st));
        SGP_CUDA_CHECK(cudaMemcpyAsync(a.residual, reinterpret_cast<const void*>(src_ptr),
                                       (size_t)a.n * sizeof(float), cudaMemcpyDefault, st));
        SGP_CUDA_CHECK(sgp_launch_gather_ack(&a, st));
    }

    void probe(int pub_grid, c10::optional<torch::Tensor> host_flag)
    {
        SgpArgs a = prepare(0);
        uint32_t* hf = nullptr;
        if (host_flag.has_value() && host_flag->defined()) {
            void* dev = nullptr;
            SGP_CUDA_CHECK(cudaHostGetDevicePointer(&dev, host_flag->data_ptr(), 0));
            hf = reinterpret_cast<uint32_t*>(dev);
        }
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_probe(&a, pub_grid, hf, at::cuda::getCurrentCUDAStream()));
    }

    void allreduce_sgd(torch::Tensor grad_ptrs, unsigned int flags, int grid)
    {
        check_grid(grid);
        SgpArgs a = prepare(flags);
        TORCH_CHECK(a.m, "allreduce_sgd needs a momentum buffer");
        TORCH_CHECK(grad_ptrs.scalar_type() == torch::kInt64 && grad_ptrs.numel() == a.world);
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_allreduce_sgd(
            &a, reinterpret_cast<void* const*>(grad_ptrs.data_ptr<int64_t>()), grid,
            at::cuda::getCurrentCUDAStream()));
    }

    void barrier()
    {
        c10::cuda::CUDAGuard guard(device_);
        SGP_CUDA_CHECK(sgp_launch_barrier(args_.pads, args_.st, args_.rank, args_.world,
                                          args_.timeout_ns, at::cuda::getCurrentCUDAStream()));
    }

    void set_timeout(double seconds) { args_.timeout_ns = (unsigned long long)(seconds * 1e9); }
    void set_segments(int k) { TORCH_CHECK(k >= 1 && k < SGP_SEQ_STRIDE); args_.segments = k; }
    int segments() const { return args_.segments; }

private:
    SgpArgs prepare(unsigned int flags) const
    {
        SgpArgs a = args_;
        a.flags = flags;
        if (grad_bf16_) a.flags |= SGP_F_GRAD_BF16; else a.flags &= ~SGP_F_GRAD_BF16;
        if (!a.shadow) a.flags &= ~SGP_F_SHADOW;
        return a;
    }
    void check_grid(int grid) const
    {
        TORCH_CHECK(grid >= 1 && grid <= SGP_MAX_CTAS, "grid out of range");
        TORCH_CHECK(max_grid_ == 0 || grid <= max_grid_,
                    "grid ", grid, " exceeds the co-resident capacity ", max_grid_,
                    " (flag-waiting CTAs must all be resident)");
    }

    SgpArgs args_;
    int device_ = 0;
    int max_grid_ = 0;
    bool grad_bf16_ = false;
    bool use_pipe_ = true;
    std::vector<torch::Tensor> keep_;
    std::vector<torch::Tensor> sched_keep_;
    torch::Tensor grad_keep_;
    torch::Tensor grad2_keep_;
    torch::Tensor mom_keep_;
};

// ---------------------------------------------------------------------------
// BilatDaemon: the AD-PSGD gossip loop as a NATIVE thread.
//
// The reference runs its gossip loop in a separate *process* with its own process group
// (gossip/ad_psgd.py:253-366).  Here it is a C++ thread inside the training process that never
// touches the Python interpreter (no GIL): it keeps enqueueing {decide, work} kernel pairs on a
// dedicated lowest-priority stream, at most `depth` pairs ahead of the GPU (throttled with a ring
// of events, cudaEventSynchronize -- not a stream synchronize, and never from Python), and backs
// off while the device-side state machine reports "nothing to do" through a pinned feedback word.
// The training thread takes the daemon's mutex (lock()/unlock(), exposed to Python as a context
// manager) to enqueue its own work on the same stream -- gradient application + model pull -- so
// those are ordered against whole gossip rounds exactly like the reference's gossip_lock.
// ---------------------------------------------------------------------------
class BilatDaemon {
public:
    BilatDaemon(std::shared_ptr<GossipContext> ctx, int grid, bool passive, double max_wait_us, int depth,
                double idle_sleep_us)
        : ctx_(std::move(ctx)), grid_(grid), passive_(passive), max_wait_us_(max_wait_us),
          depth_(depth < 1 ? 1 : (depth > 8 ? 8 : depth)), idle_sleep_us_(idle_sleep_us)
    {
        device_ = ctx_->device();
        c10::cuda::CUDAGuard guard(device_);
        int lo = 0, hi = 0;
        SGP_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        SGP_CUDA_CHECK(cudaStreamCreateWithPriority(&stream_, cudaStreamNonBlocking, lo));
        void* hp = nullptr;
        SGP_CUDA_CHECK(cudaHostAlloc(&hp, 8 * 4 * sizeof(uint32_t), cudaHostAllocMapped));
        std::memset(hp, 0, 8 * 4 * sizeof(uint32_t));
        fb_host_ = reinterpret_cast<volatile uint32_t*>(hp);
        void* dp = nullptr;
        SGP_CUDA_CHECK(cudaHostGetDevicePointer(&dp, hp, 0));
        fb_dev_ = reinterpret_cast<uint32_t*>(dp);
        for (int i = 0; i < 8; ++i) SGP_CUDA_CHECK(cudaEventCreateWithFlags(&events_[i], cudaEventDisableTiming));
    }
    // (the stream, the 8 events and the 128-byte pinned feedback block are deliberately NOT released
    // here: the destructor runs whenever Python's garbage collector gets to the object -- possibly
    // while another stream of this thread is being captured into a CUDA graph, where cudaFreeHost
    // (which synchronises the device) is illegal and would invalidate the capture)
    ~BilatDaemon() { stop(); }

    void start()
    {
        if (running_.exchange(true)) return;
        stop_ = false;
        thread_ = std::thread([this] { loop(); });
    }
    void stop()
    {
        stop_ = true;
        if (thread_.joinable()) thread_.join();
        running_ = false;
    }
    void lock() { mu_.lock(); }
    void unlock() { mu_.unlock(); }
    int64_t stream_handle() const { return reinterpret_cast<int64_t>(stream_); }
    long long pairs_enqueued() const { return pairs_.load(); }
    long long rounds_completed() const { return rounds_.load(); }
    long long idle_polls() const { return idle_.load(); }
    int last_status() const { return status_.load(); }
    std::string error() const { std::lock_guard<std::mutex> g(err_mu_); return error_; }

private:
    void loop()
    {
        cudaSetDevice(device_);
        long long i = 0;
        bool recorded[8] = {};
        while (!stop_) {
            const int slot = (int)(i % depth_);
            if (recorded[slot]) {
                // the pair enqueued `depth` iterations ago must have run before its slot is reused
                cudaError_t e = cudaEventSynchronize(events_[slot]);
                if (e != cudaSuccess) { fail(std::string("cudaEventSynchronize: ") + cudaGetErrorString(e)); return; }
                const uint32_t cmd = fb_host_[slot * 4 + 0];
                rounds_ = (long long)fb_host_[slot * 4 + 1];
                status_ = (int)fb_host_[slot * 4 + 2];
                if (cmd == 0u) {
                    ++idle_;
                    std::this_thread::sleep_for(std::chrono::microseconds((long long)idle_sleep_us_));
                }
            }
            {
                std::lock_guard<std::mutex> g(mu_);
                SgpArgs a = ctx_->raw_args(0);
                cudaError_t e = sgp_launch_bilat_decide(&a, grid_, passive_ ? 1 : 0,
                                                        (unsigned long long)(max_wait_us_ * 1e3),
                                                        fb_dev_ + slot * 4, stream_);
                if (e == cudaSuccess) {
                    SgpArgs w = ctx_->raw_args(SGP_F_FROM_STATE | (a.shadow ? SGP_F_SHADOW : 0u));
                    e = sgp_launch_step(&w, grid_, stream_);
                }
                if (e == cudaSuccess) e = cudaEventRecord(events_[slot], stream_);
                if (e != cudaSuccess) { fail(std::string("gossip launch: ") + cudaGetErrorString(e)); return; }
                g_sgp_kernel_launches += 2;
            }
            recorded[slot] = true;
            ++pairs_;
            ++i;
        }
        cudaStreamSynchronize(stream_);
    }
    void fail(const std::string& what)
    {
        std::lock_guard<std::mutex> g(err_mu_);
        error_ = what;
    }

    std::shared_ptr<GossipContext> ctx_;
    int grid_;
    bool passive_;
    double max_wait_us_;
    int depth_;
    double idle_sleep_us_;
    int device_ = 0;
    cudaStream_t stream_ = nullptr;
    cudaEvent_t events_[8] = {};
    volatile uint32_t* fb_host_ = nullptr;
    uint32_t* fb_dev_ = nullptr;
    std::thread thread_;
    std::mutex mu_;
    mutable std::mutex err_mu_;
    std::string error_;
    std::atomic<bool> stop_{false}, running_{false};
    std::atomic<long long> pairs_{0}, rounds_{0}, idle_{0};
    std::atomic<int> status_{0};
};

static void scale_(torch::Tensor x, torch::Tensor scalar, bool invert,
                   c10::optional<torch::Tensor> shadow)
{
    TORCH_CHECK(x.is_cuda() && x.scalar_type() == torch::kFloat32 && x.is_contiguous());
    TORCH_CHECK(x.numel() % 4 == 0);
    TORCH_CHECK(scalar.is_cuda() && scalar.scalar_type() == torch::kFloat32);
    __nv_bfloat16* sh = nullptr;
    if (shadow.has_value() && shadow->defined())
        sh = reinterpret_cast<__nv_bfloat16*>(shadow->data_ptr());
    c10::cuda::CUDAGuard guard(x.get_device());
    SGP_CUDA_CHECK(sgp_launch_scale(x.data_ptr<float>(), x.numel(), scalar.data_ptr<float>(),
                                    invert ? 1 : 0, sh, at::cuda::getCurrentCUDAStream()));
}

// dst = scale * sum(srcs): flat fp32 buffers of equal length, possibly on peer GPUs of this process
static void peer_reduce_(torch::Tensor dst, std::vector<torch::Tensor> srcs, double scale)
{
    TORCH_CHECK(dst.is_cuda() && dst.scalar_type() == torch::kFloat32 && dst.is_contiguous());
    TORCH_CHECK(!srcs.empty() && (int)srcs.size() <= SGP_MAX_RANKS && dst.numel() % 4 == 0);
    std::vector<const float*> ptrs;
    for (auto& t : srcs) {
        TORCH_CHECK(t.is_cuda() && t.scalar_type() == torch::kFloat32 && t.is_contiguous() &&
                    t.numel() == dst.numel());
        if (t.get_device() != dst.get_device())
            TORCH_CHECK(enable_peer_access(dst.get_device(), t.get_device()), "no peer access");
        ptrs.push_back(t.data_ptr<float>());
    }
    c10::cuda::CUDAGuard guard(dst.get_device());
    SGP_CUDA_CHECK(sgp_launch_peer_reduce(dst.data_ptr<float>(), ptrs.data(), (int)ptrs.size(), dst.numel(),
                                          (float)scale, at::cuda::getCurrentCUDAStream()));
}

// ---------------------------------------------------------------------------
// NVLS collectives (csrc/nvls_kernels.cu)
// ---------------------------------------------------------------------------
struct NvlsArgs {
    float* z; float* z_mc; void* g_mc; float* m; SgpSignalPad* const* pads; SgpState* st; const SgpHyper* hyper;
    long long n; int rank, world; unsigned long long timeout_ns; int grad_bf16; float scale;
};
extern "C" {
cudaError_t sgp_launch_nvls_allreduce(const NvlsArgs* a, int fused_sgd, int grid, cudaStream_t stream);
cudaError_t sgp_launch_nvls_bcast(float* dst_mc, const float* src, long long n, SgpSignalPad* const* pads,
                                  SgpState* st, int rank, int world, int root, unsigned long long timeout_ns,
                                  int grid, cudaStream_t stream);
int sgp_nvls_max_grid(int device);
}

// grads (multicast view, fp32 / bf16) -> switch-reduced slice -> [fused SGD-momentum on the slice ->
// multicast of the new parameters] or [scaled sum multicast back into the gradient buffers]
static void nvls_allreduce(c10::optional<torch::Tensor> z, c10::optional<torch::Tensor> z_mc, torch::Tensor g_mc,
                           c10::optional<torch::Tensor> m, torch::Tensor pad_ptrs, torch::Tensor state,
                           torch::Tensor hyper, int rank, int world, double timeout_s, double scale, bool fused_sgd,
                           int grid)
{
    TORCH_CHECK(g_mc.is_cuda() && (g_mc.scalar_type() == torch::kFloat32 || g_mc.scalar_type() == torch::kBFloat16));
    TORCH_CHECK(g_mc.numel() % SGP_CHUNK == 0, "buffer length must be a multiple of ", SGP_CHUNK);
    TORCH_CHECK(pad_ptrs.scalar_type() == torch::kInt64 && pad_ptrs.numel() == world);
    NvlsArgs a;
    std::memset(&a, 0, sizeof(a));
    a.g_mc = g_mc.data_ptr();
    a.grad_bf16 = g_mc.scalar_type() == torch::kBFloat16 ? 1 : 0;
    a.n = g_mc.numel();
    if (fused_sgd) {
        TORCH_CHECK(z.has_value() && z_mc.has_value() && m.has_value(), "fused SGD needs z, z_mc and momentum");
        TORCH_CHECK(z->numel() == a.n && z_mc->numel() == a.n && m->numel() == a.n);
        TORCH_CHECK(z->scalar_type() == torch::kFloat32 && m->scalar_type() == torch::kFloat32);
        a.z = z->data_ptr<float>();
        a.z_mc = z_mc->data_ptr<float>();
        a.m = m->data_ptr<float>();
    } else {
        TORCH_CHECK(!a.grad_bf16, "the plain NVLS all-reduce is fp32");
    }
    a.pads = reinterpret_cast<SgpSignalPad* const*>(pad_ptrs.data_ptr<int64_t>());
    a.st = reinterpret_cast<SgpState*>(state.data_ptr());
    a.hyper = reinterpret_cast<const SgpHyper*>(hyper.data_ptr());
    a.rank = rank;
    a.world = world;
    a.timeout_ns = (unsigned long long)(timeout_s * 1e9);
    a.scale = (float)scale;
    c10::cuda::CUDAGuard guard(g_mc.get_device());
    SGP_CUDA_CHECK(sgp_launch_nvls_allreduce(&a, fused_sgd ? 1 : 0, grid, at::cuda::getCurrentCUDAStream()));
}

static void nvls_bcast(torch::Tensor dst_mc, torch::Tensor src, torch::Tensor pad_ptrs, torch::Tensor state,
                       int rank, int world, int root, double timeout_s, int grid)
{
    TORCH_CHECK(dst_mc.is_cuda() && dst_mc.scalar_type() == torch::kFloat32 && dst_mc.numel() % 4 == 0);
    TORCH_CHECK(src.numel() == dst_mc.numel() && src.scalar_type() == torch::kFloat32 && src.is_contiguous());
    c10::cuda::CUDAGuard guard(dst_mc.get_device());
    SGP_CUDA_CHECK(sgp_launch_nvls_bcast(dst_mc.data_ptr<float>(), src.data_ptr<float>(), dst_mc.numel(),
                                         reinterpret_cast<SgpSignalPad* const*>(pad_ptrs.data_ptr<int64_t>()),
                                         reinterpret_cast<SgpState*>(state.data_ptr()), rank, world, root,
                                         (unsigned long long)(timeout_s * 1e9), grid,
                                         at::cuda::getCurrentCUDAStream()));
}

static void zero_(torch::Tensor x)
{
    TORCH_CHECK(x.is_cuda() && x.is_contiguous());
    const int64_t bytes = x.numel() * x.element_size();
    TORCH_CHECK(bytes % 16 == 0);
    c10::cuda::CUDAGuard guard(x.get_device());
    SGP_CUDA_CHECK(sgp_launch_zero(x.data_ptr(), bytes, at::cuda::getCurrentCUDAStream()));
}

void bind_bn(py::module& mod);   // bn_bindings.cpp
void bind_vmm(py::module& mod);  // vmm_symm.cpp
void bind_data(py::module& mod); // data_loader.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, mod)
{
    bind_bn(mod);
    bind_vmm(mod);
    bind_data(mod);
    mod.doc() = "sm_100a gossip kernels + symmetric-memory runtime";
    mod.def("symm_alloc", &symm_alloc, "allocate IPC-exportable device memory -> (uint8 tensor, handle)");
    mod.def("symm_open", &symm_open, "map a peer's allocation -> uint8 tensor");
    mod.def("enable_peer_access", &enable_peer_access);
    mod.def("pinned_flag", &pinned_flag);
    mod.def("scale_", &scale_, py::arg("x"), py::arg("scalar"), py::arg("invert"),
            py::arg("shadow") = py::none());
    mod.def("zero_", &zero_);
    mod.def("nvls_allreduce", &nvls_allreduce, py::arg("z"), py::arg("z_mc"), py::arg("g_mc"), py::arg("m"),
            py::arg("pad_ptrs"), py::arg("state"), py::arg("hyper"), py::arg("rank"), py::arg("world"),
            py::arg("timeout_s"), py::arg("scale"), py::arg("fused_sgd"), py::arg("grid"));
    mod.def("nvls_bcast", &nvls_bcast);
    mod.def("nvls_max_grid", &sgp_nvls_max_grid);
    mod.def("peer_reduce_", &peer_reduce_, py::arg("dst"), py::arg("srcs"), py::arg("scale") = 1.0);
    mod.def("launch_count", []() { return (long long)g_sgp_kernel_launches.load(); },
            "kernels of this extension launched (or captured) so far by this process");
    mod.def("max_resident_ctas", &sgp_max_resident_ctas);

    mod.attr("CHUNK") = (int)SGP_CHUNK;
    mod.attr("MAX_PEERS") = (int)SGP_MAX_PEERS;
    mod.attr("MAX_RANKS") = (int)SGP_MAX_RANKS;
    mod.attr("MAX_CTAS") = (int)SGP_MAX_CTAS;
    mod.attr("TABLE_ROW") = (int)SGP_TABLE_ROW;
    mod.attr("WTABLE_ROW") = (int)SGP_WTABLE_ROW;
    mod.attr("PAD_BYTES") = (int)sizeof(SgpSignalPad);
    mod.attr("STATE_BYTES") = (int)sizeof(SgpState);
    mod.attr("HYPER_FLOATS") = (int)(sizeof(SgpHyper) / sizeof(float));
    mod.attr("STATE_OFF_STEP") = (int)offsetof(SgpState, step);
    mod.attr("STATE_OFF_STATUS") = (int)offsetof(SgpState, status);
    mod.attr("STATE_OFF_PSW") = (int)offsetof(SgpState, ps_weight);
    mod.attr("STATE_OFF_RESW") = (int)offsetof(SgpState, res_weight);
    mod.attr("STATE_OFF_PHASE_BASE") = (int)offsetof(SgpState, phase_base);
    mod.attr("STATE_OFF_ACK_FROM") = (int)offsetof(SgpState, ack_from);
    mod.attr("STATE_OFF_BILAT_DONE") = (int)offsetof(SgpState, bilat_done);
    mod.attr("F_SGD") = (unsigned)SGP_F_SGD;
    mod.attr("F_SHADOW") = (unsigned)SGP_F_SHADOW;
    mod.attr("F_ZERO_GRAD") = (unsigned)SGP_F_ZERO_GRAD;
    mod.attr("F_PHASE1") = (unsigned)SGP_F_PHASE1;
    mod.attr("F_PHASE2") = (unsigned)SGP_F_PHASE2;
    mod.attr("F_FOLD_RES") = (unsigned)SGP_F_FOLD_RES;
    mod.attr("F_NO_ROTATE") = (unsigned)SGP_F_NO_ROTATE;
    mod.attr("F_PUBLISH") = (unsigned)SGP_F_PUBLISH;
    mod.attr("F_IN_NUMER") = (unsigned)SGP_F_IN_NUMER;
    mod.attr("F_KEEP_Z") = (unsigned)SGP_F_KEEP_Z;
    mod.attr("F_SELF_FROM_Z") = (unsigned)SGP_F_SELF_FROM_Z;

    py::class_<BilatDaemon>(mod, "BilatDaemon")
        .def(py::init<std::shared_ptr<GossipContext>, int, bool, double, int, double>(), py::arg("ctx"),
             py::arg("grid"), py::arg("passive"), py::arg("max_wait_us") = 50.0, py::arg("depth") = 2,
             py::arg("idle_sleep_us") = 100.0)
        .def("start", &BilatDaemon::start)
        .def("stop", &BilatDaemon::stop, py::call_guard<py::gil_scoped_release>())
        .def("lock", &BilatDaemon::lock, py::call_guard<py::gil_scoped_release>())
        .def("unlock", &BilatDaemon::unlock)
        .def("stream_handle", &BilatDaemon::stream_handle)
        .def("pairs_enqueued", &BilatDaemon::pairs_enqueued)
        .def("rounds_completed", &BilatDaemon::rounds_completed)
        .def("idle_polls", &BilatDaemon::idle_polls)
        .def("last_status", &BilatDaemon::last_status)
        .def("error", &BilatDaemon::error);

    mod.attr("STATE_OFF_RES_SCALE") = (int)offsetof(SgpState, res_scale);
    mod.attr("STATE_OFF_SOFT_TIMEOUT_US") = (int)offsetof(SgpState, soft_timeout_us);
    mod.attr("STATE_OFF_SOFT_TIMEOUTS") = (int)offsetof(SgpState, soft_timeouts);
    mod.attr("STATE_OFF_BILAT_ROUND") = (int)offsetof(SgpState, bilat_round);
    mod.attr("STATE_OFF_BILAT_BUDGET") = (int)offsetof(SgpState, bilat_budget);
    mod.attr("STATE_OFF_BILAT_ENABLED") = (int)offsetof(SgpState, bilat_enabled);
    mod.attr("F_FROM_STATE") = (unsigned)SGP_F_FROM_STATE;

    py::class_<GossipContext, std::shared_ptr<GossipContext>>(mod, "GossipContext")
        .def(py::init<torch::Tensor, c10::optional<torch::Tensor>, c10::optional<torch::Tensor>,
                      c10::optional<torch::Tensor>, c10::optional<torch::Tensor>, torch::Tensor,
                      c10::optional<torch::Tensor>, torch::Tensor, torch::Tensor, int, int,
                      torch::Tensor, torch::Tensor, double>(),
             py::arg("z"), py::arg("g"), py::arg("m"), py::arg("shadow"), py::arg("residual"),
             py::arg("pad_ptrs"), py::arg("outbox_ptrs"), py::arg("table"), py::arg("wtable"),
             py::arg("rank"), py::arg("world"), py::arg("state"), py::arg("hyper"),
             py::arg("timeout_s") = 30.0)
        .def("set_schedule", &GossipContext::set_schedule)
        .def("set_grad", &GossipContext::set_grad)
        .def("set_sgd_buffers", &GossipContext::set_sgd_buffers)
        .def("set_grad2", &GossipContext::set_grad2)
        .def("set_timeout", &GossipContext::set_timeout)
        .def("set_segments", &GossipContext::set_segments)
        .def("bilat_decide", &GossipContext::bilat_decide, py::arg("pub_grid"), py::arg("passive"),
             py::arg("max_wait_us") = 50.0, py::arg("host_fb") = py::none())
        .def("bilat_work", &GossipContext::bilat_work)
        .def("bilat_ctl", &GossipContext::bilat_ctl, py::arg("budget") = -1, py::arg("enabled") = -1)
        .def("set_pipe", &GossipContext::set_pipe)
        .def("pipe", &GossipContext::pipe)
        .def("segments", &GossipContext::segments)
        .def("max_grid", &GossipContext::max_grid)
        .def("step", &GossipContext::step, py::arg("flags"), py::arg("grid"))
        .def("gather", &GossipContext::gather, py::arg("grid"), py::arg("pub_grid"), py::arg("tma") = false)
        .def("gather_dma", &GossipContext::gather_dma, py::arg("pub_grid"), py::arg("src_ptr"))
        .def("probe", &GossipContext::probe, py::arg("pub_grid"), py::arg("host_flag") = py::none())
        .def("allreduce_sgd", &GossipContext::allreduce_sgd)
        .def("barrier", &GossipContext::barrier);
}
