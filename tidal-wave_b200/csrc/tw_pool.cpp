// tw_pool.cpp -- the dispatcher: a B200-native re-design of the reference's Manager + Consumer pool
// (/root/reference/src/manager.cpp:40-98, src/consumer.cpp:12-94, src/message_queue.h:50-118).
//
// Reference semantics kept: N consumers block on ONE shared request queue; consumer i is bound to one
// device for its whole life; options are fixed per pool; a response is produced for every request that a
// consumer popped; stop() drops whatever is still queued and joins the consumers; Report counts
// {request, data, error}.  Changed for the GPU: a consumer pops up to `batch` same-size requests at once and
// runs them through one batched launch sequence; there is no CPU worker; results are kept in per-id slots
// so the output does not depend on GPU count or completion order.
#include "../../include/tidalwave_b200.h"

#include <cuda_runtime_api.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

namespace {

struct Request { // Request, src/message_queue.h:13-18 (decoded images; `own` holds them for path-based requests)
    long long id;
    const uint8_t *expect, *target;
    int ew, eh, tw, th;
    std::shared_ptr<uint8_t> own_e, own_t; // pinned buffers of the pool's image store, returned to it when the request is done
    std::vector<tw_rect> ignore;           // ignore regions, copied at submit time
    const uint8_t *mask = nullptr;         // ignore mask (ew x eh) or NULL; caller-owned, or held by own_m for path-based requests
    std::shared_ptr<uint8_t> own_m;
};

struct FileJob { // Request as the reference has it: two paths (src/message_queue.h:13-18)
    long long id;
    std::string expect, target;
    std::vector<tw_rect> ignore;
    std::string mask; // "" = no mask
};

struct Slot {
    bool done = false, dropped = false;
    tw_result res{};
    std::vector<tw_vector> vectors;
    std::vector<tw_change_region> regions; // the first TW_MAX_CHANGE_REGIONS of n_regions (pools with change regions)
    int n_regions = 0;
    std::vector<tw_intensity_cell> cells;  // the first TW_MAX_INTENSITY_CELLS of n_cells (pools with intensity cells)
    int n_cells = 0;
};

} // namespace

struct tw_pool {
    tw_flow_param param{};
    double threshold = 5.0;
    int span = 10, batch = 1, vector_cap = 0, max_w = 0, max_h = 0;
    std::vector<int> devices;
    std::vector<std::thread> consumers;
    std::mutex mu;
    std::condition_variable cv_req, cv_res;
    std::deque<Request> queue;
    std::deque<FileJob> files;            // path-based requests waiting for a decoder thread
    std::vector<std::thread> decoders;
    std::condition_variable cv_file;
    int decoding = 0;                     // jobs a decoder thread is working on
    int n_decoders = 0;                   // 0: one per host core (at most 32)
    bool change_regions = false;          // fixed by the first submit (tw_pool_set_change_regions)
    int intensity = 0;                    // "intensity_threshold", fixed likewise (tw_pool_set_intensity)
    std::unordered_map<long long, Slot> slots;
    bool running = true;
    long long next_id = 0;
    int request_count = 0, data_count = 0, error_count = 0; // Report, src/message_queue.h:44-48
    std::atomic<int> ready{0};
    std::string init_error;
    // image store of the path-based requests: page-locked host buffers (tw_host_alloc) recycled between requests, so a decoded
    // image is written once, straight into memory the copy engine reads -- no 2 MB allocation + page faults per image, no
    // staging of a pageable buffer inside cudaMemcpyAsync on the consumer's thread
    struct ImageStore {
        std::mutex mu;
        std::vector<std::pair<uint8_t *, size_t>> free; // (buffer, capacity)
        ~ImageStore() { for (auto &b : free) tw_host_free(b.first); }
    };
    std::shared_ptr<ImageStore> images = std::make_shared<ImageStore>();
};

namespace {

void fill_error(tw_result *r, int code, const char *msg)
{
    memset(r, 0, sizeof *r);
    r->code = code;
    r->status = TW_STATUS_ERROR;
    snprintf(r->reason, sizeof r->reason, "%s", msg);
}

void publish(tw_pool *p, long long id, const tw_result &res, const tw_vector *vec, int nvec, const tw_change_region *reg = nullptr,
             int n_regions = 0, const tw_intensity_cell *cells = nullptr, int n_cells = 0)
{
    std::lock_guard<std::mutex> lk(p->mu);
    Slot &s = p->slots[id];
    s.res = res;
    if (nvec > 0) s.vectors.assign(vec, vec + nvec);
    if (reg && n_regions > 0) {
        s.n_regions = n_regions;
        s.regions.assign(reg, reg + std::min(n_regions, TW_MAX_CHANGE_REGIONS));
    }
    if (cells && n_cells > 0) {
        s.n_cells = n_cells;
        s.cells.assign(cells, cells + std::min(n_cells, TW_MAX_INTENSITY_CELLS));
    }
    s.done = true;
    if (res.status == TW_STATUS_ERROR) p->error_count++; else p->data_count++; // Manager::notify, src/manager.cpp:109-114
}

// The frame-independent checks of an ignore-region list (tw_compare_ignore clips to the frame): "" if it is good, else the reason.
std::string check_ignore(const tw_rect *r, int n)
{
    if (n < 0 || n > TW_MAX_IGNORE) return "bad ignore region: 0 to " + std::to_string(TW_MAX_IGNORE) + " regions per pair";
    if (n > 0 && !r) return "bad ignore region: NULL list with a count > 0";
    for (int i = 0; i < n; i++)
        if (r[i].width < 1 || r[i].height < 1) return "bad ignore region: width and height must be >= 1";
    return "";
}

std::string bad_mask_size(int mw, int mh, int ew, int eh)
{
    return "bad ignore mask: " + std::to_string(mw) + "x" + std::to_string(mh) + " mask for a " + std::to_string(ew) + "x" +
           std::to_string(eh) + " expected image";
}

// Registers a new request (p->mu held).  A bad ignore-region list answers it at once with TW_BAD_PARAMETER; returns false then.
bool new_request(tw_pool *p, long long &id, const std::string &bad_ignore)
{
    id = p->next_id++;
    Slot &s = p->slots[id];
    p->request_count++; // Manager::request, src/manager.cpp:75-76
    if (bad_ignore.empty()) return true;
    fill_error(&s.res, TW_BAD_PARAMETER, bad_ignore.c_str());
    s.done = true;
    p->error_count++;
    return false;
}

// imread of both paths (src/opticalflow.cpp:20-49) on a decoder thread, then the request joins the compute queue.
bool read_file(const std::string &path, std::vector<uint8_t> &out)
{
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return false;
    out.clear();
    if (fseek(f, 0, SEEK_END) == 0) { // regular file: one read of its size
        const long size = ftell(f);
        if (size > 0 && fseek(f, 0, SEEK_SET) == 0) {
            out.resize((size_t)size);
            out.resize(fread(out.data(), 1, (size_t)size, f));
            fclose(f);
            return !out.empty();
        }
        rewind(f);
    }
    uint8_t buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) out.insert(out.end(), buf, buf + n);
    fclose(f);
    return !out.empty();
}

std::shared_ptr<uint8_t> take_image(const std::shared_ptr<tw_pool::ImageStore> &st, size_t bytes)
{
    uint8_t *buf = nullptr;
    size_t cap = 0;
    {
        std::lock_guard<std::mutex> lk(st->mu);
        for (size_t i = 0; i < st->free.size(); i++)
            if (st->free[i].second >= bytes && st->free[i].second <= 2 * bytes + 4096) { // no 8 MB buffer behind a thumbnail
                buf = st->free[i].first; cap = st->free[i].second;
                st->free[i] = st->free.back();
                st->free.pop_back();
                break;
            }
    }
    if (!buf) {
        cap = (bytes + 4095) & ~(size_t)4095;
        buf = (uint8_t *)tw_host_alloc(cap);
        if (!buf) { // no page-locked memory to be had: an ordinary buffer, not recycled
            buf = (uint8_t *)malloc(cap);
            return std::shared_ptr<uint8_t>(buf, [](uint8_t *b) { free(b); });
        }
    }
    // the deleter keeps the store alive: a request can outlive tw_pool_destroy only inside this translation unit, but the order of
    // member destruction must not matter
    return std::shared_ptr<uint8_t>(buf, [st, cap](uint8_t *b) {
        std::lock_guard<std::mutex> lk(st->mu);
        if (st->free.size() < 256) st->free.emplace_back(b, cap); else tw_host_free(b);
    });
}

bool imread_gray(tw_pool *p, const std::string &path, std::vector<uint8_t> &raw, std::shared_ptr<uint8_t> &img, int &w, int &h)
{
    if (!read_file(path, raw)) return false;
    if (tw_decode_gray(raw.data(), raw.size(), nullptr, 0, &w, &h) != TW_OK || w < 1 || h < 1) return false;
    img = take_image(p->images, (size_t)w * h);
    return img && tw_decode_gray(raw.data(), raw.size(), img.get(), (size_t)w * h, &w, &h) == TW_OK;
}

void decoder_main(tw_pool *p)
{
    std::vector<uint8_t> raw;
    if (!p->devices.empty()) cudaSetDevice(p->devices[0]); // page-locked allocations come from a context the pool uses anyway
    for (;;) {
        FileJob job;
        {
            std::unique_lock<std::mutex> lk(p->mu);
            // back-pressure: decoders stay at most a few batches ahead of the consumers, so the decoded images waiting in page-locked
            // memory are bounded however many paths have been submitted
            const size_t ahead = std::max<size_t>(64, (size_t)4 * p->batch * std::max<size_t>(1, p->devices.size()));
            p->cv_file.wait(lk, [&] { return (!p->files.empty() && p->queue.size() + (size_t)p->decoding < ahead) || !p->running; });
            if (!p->running) return;
            job = std::move(p->files.front());
            p->files.pop_front();
            p->decoding++;
        }
        Request r{};
        r.id = job.id;
        r.ignore = std::move(job.ignore);
        tw_result e;
        bool ok = true;
        // src/opticalflow.cpp:20-49: empty paths are BadParameter, unreadable / undecodable files BadImageFormat "Can't open <path>"
        if (job.expect.empty()) { fill_error(&e, TW_BAD_PARAMETER, "ExpectImagePath is empty."); ok = false; }
        else if (job.target.empty()) { fill_error(&e, TW_BAD_PARAMETER, "TargetImagePath is empty."); ok = false; }
        else if (!imread_gray(p, job.expect, raw, r.own_e, r.ew, r.eh)) { fill_error(&e, TW_BAD_IMAGE_FORMAT, ("Can't open " + job.expect).c_str()); ok = false; }
        else if (!imread_gray(p, job.target, raw, r.own_t, r.tw, r.th)) { fill_error(&e, TW_BAD_IMAGE_FORMAT, ("Can't open " + job.target).c_str()); ok = false; }
        else if (!job.mask.empty()) { // the ignore mask: a gray image of the expected image's size, into the same image store
            int mw = 0, mh = 0;
            if (!imread_gray(p, job.mask, raw, r.own_m, mw, mh)) { fill_error(&e, TW_BAD_IMAGE_FORMAT, ("Can't open " + job.mask).c_str()); ok = false; }
            else if (mw != r.ew || mh != r.eh) { fill_error(&e, TW_BAD_PARAMETER, bad_mask_size(mw, mh, r.ew, r.eh).c_str()); ok = false; }
            else r.mask = r.own_m.get();
        }
        if (!ok) {
            publish(p, job.id, e, nullptr, 0);
            std::lock_guard<std::mutex> lk(p->mu);
            p->decoding--;
            p->cv_res.notify_all();
            continue;
        }
        r.expect = r.own_e.get(); r.target = r.own_t.get();
        {
            std::lock_guard<std::mutex> lk(p->mu);
            p->decoding--;
            if (!p->running) { p->slots[r.id].dropped = true; p->cv_res.notify_all(); return; }
            p->queue.push_back(std::move(r));
        }
        p->cv_req.notify_one();
    }
}

// Consumer::run, src/consumer.cpp:42-94
void consumer_main(tw_pool *p, int idx)
{
    char err[256] = {0};
    tw_ctx *ctx = tw_create(p->devices[idx], p->max_w, p->max_h, p->batch, err, sizeof err);
    // The dispatcher only ever reports status + sampled vectors (Response, src/message_queue.h:27-40): its contexts evaluate
    // the last iteration of the finest scale at the sampled positions only (bit-identical vectors, no dense field).
    // TW_SPARSE_LAST=0 keeps the dense last iteration.
    if (ctx) {
        const char *e = getenv("TW_SPARSE_LAST");
        tw_set_option(ctx, "sparse_last", (e && atoi(e) == 0) ? 0 : 1);
    }
    {
        std::lock_guard<std::mutex> lk(p->mu);
        if (!ctx) p->init_error = err;
        p->ready.fetch_add(1);
    }
    p->cv_res.notify_all();
    // vector_cap > 0: at most that many vectors are kept per request; vector_cap == 0: every vector of every request (the
    // reference returns them all, src/consumer.cpp:60-76) -- the capacity then follows each request's own sampling grid
    std::vector<tw_vector> vec;
    std::vector<tw_result> res(p->batch);
    std::vector<Request> work;
    std::vector<const uint8_t *> ex(p->batch), tg(p->batch);
    std::vector<const tw_rect *> ig(p->batch);
    std::vector<int> nig(p->batch);
    std::vector<const uint8_t *> mk(p->batch);
    // change regions and the intensity threshold: the pool's settings are fixed once a request exists, so they are applied before
    // this consumer's first batch
    bool regions = false, regions_set = false;
    int intensity = 0;
    std::vector<tw_change_region> reg(TW_MAX_CHANGE_REGIONS);
    std::vector<tw_intensity_cell> cells(TW_MAX_INTENSITY_CELLS);
    // publishes pair i of the batch the context answered last, with its change regions and intensity cells
    auto publish_pair = [&](long long id, int i, const tw_result &r, const tw_vector *v, int nv) {
        int nreg = 0, ncell = 0;
        if (regions && tw_change_regions(ctx, i, reg.data(), TW_MAX_CHANGE_REGIONS, &nreg) != TW_OK) nreg = 0;
        if (intensity && tw_intensity_cells(ctx, i, cells.data(), TW_MAX_INTENSITY_CELLS, &ncell) != TW_OK) ncell = 0;
        publish(p, id, r, v, nv, reg.data(), nreg, cells.data(), ncell);
    };
    // Up to two batches are in flight on the context (tw_pipe_*): while batch k runs, this thread pops and uploads batch k + 1
    // and then collects batch k - 1 -- one consumer thread per GPU keeps the device busy (src/consumer.cpp:18-24).
    struct InFlight { std::vector<Request> work; int cap = 0; };
    std::deque<InFlight> inflight;
    auto collect_oldest = [&]() {
        InFlight f = std::move(inflight.front());
        inflight.pop_front();
        const int n = (int)f.work.size();
        if (vec.size() < (size_t)n * f.cap) vec.resize((size_t)n * f.cap);
        tw_pipe_collect(ctx, vec.data(), f.cap, res.data());
        for (int i = 0; i < n; i++) publish_pair(f.work[i].id, i, res[i], vec.data() + (size_t)i * f.cap, std::min(res[i].n_vectors, f.cap));
        p->cv_res.notify_all();
    };
    for (;;) {
        work.clear();
        {
            // MessageQueue::tryPop, src/message_queue.h:67-85: wait for a request or the stop notice; with batches in flight do
            // not block -- their results are due
            std::unique_lock<std::mutex> lk(p->mu);
            if (inflight.empty()) p->cv_req.wait(lk, [&] { return !p->queue.empty() || !p->running; });
            if (!p->running) break;
            if (!p->queue.empty()) {
                work.push_back(p->queue.front());
                p->queue.pop_front();
                // batch: take the following requests while they are compute-ready and have the same size; while the GPU is
                // still busy with an earlier batch there is time to let a short queue fill up (until that batch is done, at most 20 x 50 us)
                const Request h = work[0];
                const bool head_ok = h.expect && h.target && h.ew == h.tw && h.eh == h.th;
                for (int spins = 0; head_ok && (int)work.size() < p->batch; ) {
                    if (p->queue.empty()) {
                        if (inflight.empty() || spins++ >= 20 || !p->running || tw_pipe_ready(ctx)) break;
                        p->cv_req.wait_for(lk, std::chrono::microseconds(50));
                        continue;
                    }
                    const Request &q = p->queue.front();
                    if (!(q.expect && q.target && q.ew == h.ew && q.eh == h.eh && q.tw == h.ew && q.th == h.eh)) break;
                    work.push_back(q);
                    p->queue.pop_front();
                }
                if (!p->files.empty()) p->cv_file.notify_all(); // room for the decoders again
            }
        }
        if (work.empty()) { // nothing new: deliver the oldest batch in flight
            collect_oldest();
            continue;
        }
        if (!ctx) {
            for (auto &r : work) {
                tw_result e;
                fill_error(&e, TW_CUDA_ERROR, err);
                publish(p, r.id, e, nullptr, 0);
            }
            p->cv_res.notify_all();
            continue;
        }
        if (!regions_set) {
            {
                std::lock_guard<std::mutex> lk(p->mu);
                regions = p->change_regions;
                intensity = p->intensity;
            }
            tw_set_option(ctx, "change_regions", regions ? 1 : 0); // nothing in flight yet
            tw_set_option(ctx, "intensity_threshold", intensity);
            regions_set = true;
        }
        int cap = p->vector_cap;
        if (cap <= 0) cap = std::max(1, ((work[0].ew + p->span - 1) / p->span) * ((work[0].eh + p->span - 1) / p->span));
        const Request &r0 = work[0];
        const bool same = r0.expect && r0.target && r0.ew == r0.tw && r0.eh == r0.th;
        if (!same) {
            // error cases and the +-5 px resize path of OpticalFlow::calculate (src/opticalflow.cpp:37-68): synchronous, pipe drained
            while (!inflight.empty()) collect_oldest();
            if (vec.size() < (size_t)cap) vec.resize(cap);
            tw_compare_mask(ctx, r0.expect, r0.ew, r0.eh, r0.target, r0.tw, r0.th, &p->param, p->threshold, p->span, r0.ignore.data(),
                            (int)r0.ignore.size(), r0.mask, vec.data(), cap, &res[0]);
            publish_pair(r0.id, 0, res[0], vec.data(), std::min(res[0].n_vectors, cap));
            p->cv_res.notify_all();
            continue;
        }
        const int n = (int)work.size();
        // pairs with and without regions / masks share a batch; one with regions runs the ignore form, one with a mask the mask form
        bool any_ignore = false, any_mask = false;
        for (int i = 0; i < n; i++) {
            ex[i] = work[i].expect; tg[i] = work[i].target;
            ig[i] = work[i].ignore.data(); nig[i] = (int)work[i].ignore.size();
            mk[i] = work[i].mask;
            any_ignore |= nig[i] > 0;
            any_mask |= mk[i] != nullptr;
        }
        if (!inflight.empty() && (inflight.back().work[0].ew != r0.ew || inflight.back().work[0].eh != r0.eh))
            while (!inflight.empty()) collect_oldest(); // a new size rebuilds the plan: nothing may be in flight
        if (tw_pipe_pending(ctx) >= 2) collect_oldest();
        int rc = tw_pipe_submit_mask(ctx, n, ex.data(), tg.data(), r0.ew, r0.eh, r0.ew, &p->param, p->threshold, p->span, ig.data(),
                                     any_ignore ? nig.data() : nullptr, any_mask ? mk.data() : nullptr);
        if (rc != TW_OK) {
            tw_result e;
            fill_error(&e, rc, tw_last_error(ctx));
            for (auto &r : work) publish(p, r.id, e, nullptr, 0);
            p->cv_res.notify_all();
            continue;
        }
        InFlight f;
        f.work = work; f.cap = cap;
        inflight.push_back(std::move(f));
    }
    while (ctx && !inflight.empty()) collect_oldest(); // stop: requests already on the device are still answered
    if (ctx) tw_destroy(ctx);
}

int take(tw_pool *p, std::unordered_map<long long, Slot>::iterator it, tw_vector *out, int cap, tw_result *res,
         tw_change_region *regions = nullptr, int region_cap = 0, int *n_regions = nullptr, tw_intensity_cell *cells = nullptr,
         int cell_cap = 0, int *n_cells = nullptr)
{
    Slot &s = it->second;
    if (s.dropped) { p->slots.erase(it); return -1; }
    if (res) *res = s.res;
    int n = std::min<int>((int)s.vectors.size(), cap);
    if (out && n > 0) memcpy(out, s.vectors.data(), sizeof(tw_vector) * n);
    const int k = std::min<int>((int)s.regions.size(), region_cap);
    if (regions && k > 0) memcpy(regions, s.regions.data(), sizeof(tw_change_region) * k);
    if (n_regions) *n_regions = s.n_regions;
    const int kc = std::min<int>((int)s.cells.size(), cell_cap);
    if (cells && kc > 0) memcpy(cells, s.cells.data(), sizeof(tw_intensity_cell) * kc);
    if (n_cells) *n_cells = s.n_cells;
    int code = s.res.code;
    p->slots.erase(it);
    return code;
}

} // namespace

extern "C" {

tw_pool *tw_pool_create(const int *devices, int n_devices, int max_w, int max_h, int batch, const tw_flow_param *param,
                        double threshold, int span, int vector_cap, char *err, int errlen)
{
    auto fail = [&](const char *m) -> tw_pool * {
        if (err && errlen > 0) snprintf(err, errlen, "%s", m);
        return nullptr;
    };
    if (!devices || n_devices < 1 || !param || span < 1 || batch < 1 || vector_cap < 0) return fail("bad pool parameter");
    if (tw_device_count() < 1) return fail("no CUDA device (there is no CPU fallback worker)");
    tw_pool *p = new tw_pool();
    p->param = *param; p->threshold = threshold; p->span = span; p->batch = batch; p->vector_cap = vector_cap;
    p->max_w = max_w; p->max_h = max_h;
    p->devices.assign(devices, devices + n_devices);
    // Manager::start, src/manager.cpp:55-59: one consumer per device entry
    for (int i = 0; i < n_devices; i++) p->consumers.emplace_back(consumer_main, p, i);
    {
        std::unique_lock<std::mutex> lk(p->mu);
        p->cv_res.wait(lk, [&] { return p->ready.load() == n_devices; });
        if (!p->init_error.empty()) {
            std::string m = p->init_error;
            lk.unlock();
            tw_pool_stop(p);
            tw_pool_destroy(p);
            return fail(m.c_str());
        }
    }
    return p;
}

long long tw_pool_submit_mask(tw_pool *p, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_,
                              const tw_rect *ignore, int n_ignore, const uint8_t *mask)
{
    if (!p) return -1;
    const std::string bad = check_ignore(ignore, n_ignore);
    long long id;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        if (!p->running) return -1;
        if (!new_request(p, id, bad)) { p->cv_res.notify_all(); return id; }
        Request r{id, expect, target, ew, eh, tw_, th_};
        if (n_ignore > 0) r.ignore.assign(ignore, ignore + n_ignore);
        r.mask = mask;
        p->queue.push_back(std::move(r));
    }
    p->cv_req.notify_one();
    return id;
}

long long tw_pool_submit_ignore(tw_pool *p, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_,
                                const tw_rect *ignore, int n_ignore)
{
    return tw_pool_submit_mask(p, expect, ew, eh, target, tw_, th_, ignore, n_ignore, nullptr);
}

long long tw_pool_submit(tw_pool *p, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_)
{
    return tw_pool_submit_ignore(p, expect, ew, eh, target, tw_, th_, nullptr, 0);
}

// Manager::request as the reference has it (src/manager.cpp:68-78): two image PATHS.  The files are read and decoded on the pool's
// decoder threads (cv::imread(IMREAD_GRAYSCALE), src/opticalflow.cpp:37,44 -> tw_decode_gray), started on first use.
long long tw_pool_submit_files_mask(tw_pool *p, const char *expect_path, const char *target_path, const char *mask_path,
                                    const tw_rect *ignore, int n_ignore)
{
    if (!p) return -1;
    const std::string bad = check_ignore(ignore, n_ignore);
    long long id;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        if (!p->running) return -1;
        if (p->decoders.empty()) {
            int n = p->n_decoders > 0 ? p->n_decoders : (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
            for (int i = 0; i < n; i++) p->decoders.emplace_back(decoder_main, p);
        }
        if (!new_request(p, id, bad)) { p->cv_res.notify_all(); return id; }
        FileJob job{id, expect_path ? expect_path : "", target_path ? target_path : "", {}, mask_path ? mask_path : ""};
        if (n_ignore > 0) job.ignore.assign(ignore, ignore + n_ignore);
        p->files.push_back(std::move(job));
    }
    p->cv_file.notify_one();
    return id;
}

long long tw_pool_submit_files_ignore(tw_pool *p, const char *expect_path, const char *target_path, const tw_rect *ignore, int n_ignore)
{
    return tw_pool_submit_files_mask(p, expect_path, target_path, nullptr, ignore, n_ignore);
}

long long tw_pool_submit_files(tw_pool *p, const char *expect_path, const char *target_path)
{
    return tw_pool_submit_files_ignore(p, expect_path, target_path, nullptr, 0);
}

int tw_pool_set_decoders(tw_pool *p, int n)
{
    if (!p || n < 1) return TW_BAD_PARAMETER;
    std::lock_guard<std::mutex> lk(p->mu);
    if (!p->decoders.empty()) return TW_BAD_PARAMETER; // already started
    p->n_decoders = n;
    return TW_OK;
}

int tw_pool_set_change_regions(tw_pool *p, int on)
{
    if (!p) return TW_BAD_PARAMETER;
    std::lock_guard<std::mutex> lk(p->mu);
    if (p->next_id > 0) return TW_BAD_PARAMETER; // a consumer may already run with the old setting
    p->change_regions = on != 0;
    return TW_OK;
}

int tw_pool_set_intensity(tw_pool *p, int t)
{
    if (!p || t < 0 || t > 255) return TW_BAD_PARAMETER;
    std::lock_guard<std::mutex> lk(p->mu);
    if (p->next_id > 0) return TW_BAD_PARAMETER; // a consumer may already run with the old setting
    p->intensity = t;
    return TW_OK;
}

int tw_pool_wait_intensity(tw_pool *p, long long id, tw_vector *out, int cap, tw_result *res, tw_change_region *regions, int region_cap,
                           int *n_regions, tw_intensity_cell *cells, int cell_cap, int *n_cells)
{
    if (!p) return -1;
    std::unique_lock<std::mutex> lk(p->mu);
    auto it = p->slots.find(id);
    if (it == p->slots.end()) return -1;
    p->cv_res.wait(lk, [&] { it = p->slots.find(id); return it == p->slots.end() || it->second.done || it->second.dropped; });
    if (it == p->slots.end()) return -1;
    return take(p, it, out, cap, res, regions, region_cap, n_regions, cells, cell_cap, n_cells);
}

int tw_pool_wait_regions(tw_pool *p, long long id, tw_vector *out, int cap, tw_result *res, tw_change_region *regions, int region_cap,
                         int *n_regions)
{
    return tw_pool_wait_intensity(p, id, out, cap, res, regions, region_cap, n_regions, nullptr, 0, nullptr);
}

int tw_pool_wait(tw_pool *p, long long id, tw_vector *out, int cap, tw_result *res)
{
    return tw_pool_wait_regions(p, id, out, cap, res, nullptr, 0, nullptr);
}

// Blocks until request `id` is answered and copies its tw_result WITHOUT taking it: res->n_vectors tells the caller how many
// vectors tw_pool_wait will need room for (path-based requests: the caller does not know the image size beforehand).
int tw_pool_peek(tw_pool *p, long long id, tw_result *res)
{
    if (!p || !res) return -1;
    std::unique_lock<std::mutex> lk(p->mu);
    auto it = p->slots.find(id);
    if (it == p->slots.end()) return -1;
    p->cv_res.wait(lk, [&] { it = p->slots.find(id); return it == p->slots.end() || it->second.done || it->second.dropped; });
    if (it == p->slots.end() || it->second.dropped) return -1;
    *res = it->second.res;
    return res->code;
}

int tw_pool_poll(tw_pool *p, long long id, tw_vector *out, int cap, tw_result *res)
{
    if (!p) return -1;
    std::lock_guard<std::mutex> lk(p->mu);
    auto it = p->slots.find(id);
    if (it == p->slots.end()) return -1;
    if (it->second.dropped) { p->slots.erase(it); return -1; }
    if (!it->second.done) return 0;
    take(p, it, out, cap, res);
    return 1;
}

void tw_pool_report(tw_pool *p, int *request_count, int *data_count, int *error_count)
{
    if (!p) return;
    std::lock_guard<std::mutex> lk(p->mu);
    if (request_count) *request_count = p->request_count;
    if (data_count) *data_count = p->data_count;
    if (error_count) *error_count = p->error_count;
}

void tw_pool_stop(tw_pool *p)
{
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        if (!p->running && p->consumers.empty() && p->decoders.empty()) return;
        p->running = false;
        // pending requests are dropped (tryPop returns false once stopped, src/message_queue.h:75-78)
        for (auto &r : p->queue) p->slots[r.id].dropped = true;
        p->queue.clear();
        for (auto &f : p->files) p->slots[f.id].dropped = true;
        p->files.clear();
    }
    p->cv_req.notify_all();
    p->cv_file.notify_all();
    p->cv_res.notify_all();
    for (auto &t : p->decoders) if (t.joinable()) t.join();
    p->decoders.clear();
    {   // a decoder that was mid-job when the pool stopped may have queued its request: drop it like the others
        std::lock_guard<std::mutex> lk(p->mu);
        for (auto &r : p->queue) p->slots[r.id].dropped = true;
        p->queue.clear();
    }
    for (auto &t : p->consumers) if (t.joinable()) t.join();
    p->consumers.clear();
    p->cv_res.notify_all();
}

void tw_pool_destroy(tw_pool *p)
{
    if (!p) return;
    tw_pool_stop(p);
    delete p;
}

} // extern "C"
