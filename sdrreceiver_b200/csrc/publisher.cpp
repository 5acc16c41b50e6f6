// ZMQ output, wire-compatible with ZmqPublisher (zmqpublisher.cpp:15-96): one PUB socket,
// the same keepalive / reconnect socket options, and per message three frames
//   [topic, exactly 5 bytes][sample rate, uint32 little endian][int16 LE mono PCM].
// libzmq has no headers in this image, so the eight entry points are resolved at run time
// from SDRB_LIBZMQ, the system libzmq, or the copy bundled with pyzmq.
#include <dlfcn.h>
#include <glob.h>

#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <string>
#include <set>
#include <thread>
#include <vector>

#include "plan.hpp"

struct sdrb_plan { sdrb::HostPlan h; };

namespace {
struct ZmqApi {
    void *lib = nullptr;
    void *(*ctx_new)() = nullptr;
    int (*ctx_term)(void *) = nullptr;
    void *(*socket)(void *, int) = nullptr;
    int (*close)(void *) = nullptr;
    int (*setsockopt)(void *, int, const void *, size_t) = nullptr;
    int (*bind)(void *, const char *) = nullptr;
    int (*connect)(void *, const char *) = nullptr;
    int (*send)(void *, const void *, size_t, int) = nullptr;
    int (*err)() = nullptr;
};
ZmqApi g_zmq;

bool load_zmq() {
    if (g_zmq.lib) return true;
    std::string cands[8];
    int n = 0;
    if (const char *e = getenv("SDRB_LIBZMQ")) cands[n++] = e;
    cands[n++] = "libzmq.so.5";
    cands[n++] = "libzmq.so";
    glob_t g;
    const char *pats[] = {"/opt/prime-rl/.venv/lib/python3*/site-packages/pyzmq.libs/libzmq-*.so*",
                          "/usr/lib/python3/dist-packages/pyzmq.libs/libzmq-*.so*",
                          "/usr/local/lib/python3*/site-packages/pyzmq.libs/libzmq-*.so*"};
    for (const char *pat : pats)
        if (n < 8 && glob(pat, 0, nullptr, &g) == 0) {
            if (g.gl_pathc > 0) cands[n++] = g.gl_pathv[0];
            globfree(&g);
        }
    for (int i = 0; i < n && !g_zmq.lib; i++) g_zmq.lib = dlopen(cands[i].c_str(), RTLD_NOW | RTLD_LOCAL);
    if (!g_zmq.lib) { sdrb::set_error("libzmq not found (set SDRB_LIBZMQ to its path)"); return false; }
#define SYM(field, name) g_zmq.field = (decltype(g_zmq.field))dlsym(g_zmq.lib, name)
    SYM(ctx_new, "zmq_ctx_new"); SYM(ctx_term, "zmq_ctx_term"); SYM(socket, "zmq_socket"); SYM(close, "zmq_close");
    SYM(setsockopt, "zmq_setsockopt"); SYM(bind, "zmq_bind"); SYM(connect, "zmq_connect"); SYM(send, "zmq_send");
    SYM(err, "zmq_errno");
#undef SYM
    if (!g_zmq.ctx_new || !g_zmq.socket || !g_zmq.setsockopt || !g_zmq.bind || !g_zmq.connect || !g_zmq.send) {
        sdrb::set_error("libzmq is missing required symbols");
        dlclose(g_zmq.lib); g_zmq.lib = nullptr;
        return false;
    }
    return true;
}
// libzmq 4.x constants (zmq.h)
constexpr int kPUB = 1, kSNDMORE = 2, kRECONNECT_IVL = 18, kRECONNECT_IVL_MAX = 21;
constexpr int kKEEPALIVE = 34, kKEEPALIVE_CNT = 35, kKEEPALIVE_IDLE = 36, kKEEPALIVE_INTVL = 37, kLINGER = 17, kSNDHWM = 23;
}  // namespace

struct sdrb_publisher {
    void *ctx = nullptr, *sock = nullptr;
};

// default_sndhwm: 0 = leave libzmq's default (what the reference does), > 0 = the pool's mark
static int publisher_open(const char *address, int bind, int default_sndhwm, sdrb_publisher **out) {
    if (!address || !out) { sdrb::set_error("sdrb_publisher_open: NULL argument"); return SDRB_E_INVALID; }
    *out = nullptr;
    if (!load_zmq()) return SDRB_E_ZMQ;
    sdrb_publisher *p = new sdrb_publisher();
    p->ctx = g_zmq.ctx_new();
    p->sock = p->ctx ? g_zmq.socket(p->ctx, kPUB) : nullptr;
    if (!p->sock) { sdrb::set_error("zmq_socket failed"); delete p; return SDRB_E_ZMQ; }
    // same options, same values as ZmqPublisher::connect (zmqpublisher.cpp:24-37). One addition, documented in
    // include/sdrb200.h: ZMQ_LINGER. The reference never closes its sockets -- they die with the process and whatever is
    // still queued is dropped; sdrb_publisher_close() reproduces that with linger 0 unless SDRB_ZMQ_LINGER_MS asks it to
    // wait (-1 = libzmq's default, wait for ever).
    const int keepalive = 1, cnt = 10, idle = 1, intvl = 1, reconnect = 1000, reconnect_max = 0;
    int linger = 0;
    if (const char *e = getenv("SDRB_ZMQ_LINGER_MS")) linger = atoi(e);
    g_zmq.setsockopt(p->sock, kKEEPALIVE, &keepalive, sizeof(int));
    g_zmq.setsockopt(p->sock, kKEEPALIVE_CNT, &cnt, sizeof(int));
    g_zmq.setsockopt(p->sock, kKEEPALIVE_IDLE, &idle, sizeof(int));
    g_zmq.setsockopt(p->sock, kKEEPALIVE_INTVL, &intvl, sizeof(int));
    g_zmq.setsockopt(p->sock, kRECONNECT_IVL, &reconnect, sizeof(int));
    g_zmq.setsockopt(p->sock, kRECONNECT_IVL_MAX, &reconnect_max, sizeof(int));
    g_zmq.setsockopt(p->sock, kLINGER, &linger, sizeof(int));
    // Send high-water mark: the reference keeps libzmq's default (1000 messages per subscriber), enough for one receiver's 27
    // messages per callback. A pool socket carries the callbacks of a whole call for its share of the receivers in one burst
    // (1728 messages for 25E, 128 receivers, 4 callbacks, 8 sockets): everything past the mark would be dropped before the I/O
    // thread has had a chance to write it. SDRB_ZMQ_SNDHWM overrides both (0 = no limit).
    int sndhwm = default_sndhwm;
    if (const char *e = getenv("SDRB_ZMQ_SNDHWM")) sndhwm = atoi(e);
    if (sndhwm > 0 || getenv("SDRB_ZMQ_SNDHWM")) g_zmq.setsockopt(p->sock, kSNDHWM, &sndhwm, sizeof(int));
    const int rc = bind ? g_zmq.bind(p->sock, address) : g_zmq.connect(p->sock, address);
    if (rc < 0) {
        sdrb::set_error(std::string("ZeroMQ could not ") + (bind ? "bind to " : "connect to ") + address +
                        " error code: " + std::to_string(g_zmq.err ? g_zmq.err() : -1));
        if (g_zmq.close) g_zmq.close(p->sock);
        if (g_zmq.ctx_term) g_zmq.ctx_term(p->ctx);
        delete p;
        return SDRB_E_ZMQ;
    }
    *out = p;
    return SDRB_OK;
}

extern "C" int sdrb_publisher_open(const char *address, int bind, sdrb_publisher **out) { return publisher_open(address, bind, 0, out); }

extern "C" int sdrb_publisher_send(sdrb_publisher *p, const char *topic, uint32_t rate, const void *payload, uint32_t len) {
    if (!p || !topic || (!payload && len)) { sdrb::set_error("sdrb_publisher_send: NULL argument"); return SDRB_E_INVALID; }
    if (len == 0) return SDRB_OK;                                 // zmqpublisher.cpp:88
    char t[SDRB_TOPIC_LEN] = {0, 0, 0, 0, 0};                     // always 5 bytes on the wire (line 91)
    memcpy(t, topic, strnlen(topic, SDRB_TOPIC_LEN));
    unsigned char r[4];
    memcpy(r, &rate, 4);
    if (g_zmq.send(p->sock, t, SDRB_TOPIC_LEN, kSNDMORE) < 0 || g_zmq.send(p->sock, r, 4, kSNDMORE) < 0 ||
        g_zmq.send(p->sock, payload, len, 0) < 0) {
        sdrb::set_error("zmq_send failed, errno " + std::to_string(g_zmq.err ? g_zmq.err() : -1));
        return SDRB_E_ZMQ;
    }
    return SDRB_OK;
}

extern "C" int sdrb_publisher_send_block(sdrb_publisher *p, const sdrb_plan *plan, const int16_t *rec) {
    if (!p || !plan || !rec) { sdrb::set_error("sdrb_publisher_send_block: NULL argument"); return SDRB_E_INVALID; }
    for (const sdrb::SubVfo &s : plan->h.subs) {                  // vfo::transmitData, vfo.cpp:426-437
        const int rc = sdrb_publisher_send(p, s.topic.c_str(), (uint32_t)s.out_rate, rec + s.pcm_offset,
                                           (uint32_t)s.samples_out * 2u);
        if (rc != SDRB_OK) return rc;
    }
    return SDRB_OK;
}

extern "C" void sdrb_publisher_close(sdrb_publisher *p) {
    if (!p) return;
    if (p->sock && g_zmq.close) g_zmq.close(p->sock);
    if (p->ctx && g_zmq.ctx_term) g_zmq.ctx_term(p->ctx);
    delete p;
}

// ---- a pool of publishers: one PUB socket and one sender thread per stream group ----
// A reference deployment runs one SDRReceiver process -- one ZmqPublisher, one address -- per dongle; a bank holds hundreds of
// receivers, and one socket fed by one thread caps the publish leg far below the GPU path (profiles/r02_experiments.md section 6:
// zmq_send copies every payload, 224 MB per bench step). The pool keeps the reference's wire format per message
// (zmqpublisher.cpp:82-96) and the per-receiver order of callbacks; receiver s goes out on socket s % n_sockets.
struct sdrb_publisher_pool {
    std::vector<sdrb_publisher *> pubs;
    std::vector<std::string> addrs;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    unsigned long long gen = 0;
    int pending = 0, failed = 0;
    bool quit = false;
    // the job of the current generation
    const sdrb_plan *plan = nullptr;
    const int16_t *pcm = nullptr;
    const int32_t *streams = nullptr;   // send_streams: record i belongs to receiver streams[i] (send_call: to receiver i)
    int n_streams = 0, n_blocks = 0;
    std::string error;
};

namespace {
std::string pool_address(const char *address, int k) {
    std::string a(address);
    const size_t at = a.find("%d");
    if (at != std::string::npos) return a.substr(0, at) + std::to_string(k) + a.substr(at + 2);
    // tcp://host:port -> port + k; anything else (ipc, inproc): ".k" appended
    const size_t colon = a.rfind(':');
    if (a.compare(0, 6, "tcp://") == 0 && colon != std::string::npos && colon > 5) {
        char *end = nullptr;
        const long port = strtol(a.c_str() + colon + 1, &end, 10);
        if (end && *end == 0 && port > 0) return a.substr(0, colon + 1) + std::to_string(port + k);
    }
    return a + "." + std::to_string(k);
}

void pool_worker(sdrb_publisher_pool *pool, int k) {
    unsigned long long seen = 0;
    for (;;) {
        const sdrb_plan *plan; const int16_t *pcm; const int32_t *list; int ns, nb;
        {
            std::unique_lock<std::mutex> lk(pool->mu);
            pool->cv_go.wait(lk, [&] { return pool->quit || pool->gen != seen; });
            if (pool->quit) return;
            seen = pool->gen;
            plan = pool->plan; pcm = pool->pcm; list = pool->streams; ns = pool->n_streams; nb = pool->n_blocks;
        }
        int rc = SDRB_OK;
        const size_t rec = (size_t)plan->h.pcm_per_block;
        const int n = (int)pool->pubs.size();
        for (int i = list ? 0 : k; i < ns && rc == SDRB_OK; i += list ? 1 : n) {
            if (list && list[i] % n != k) continue;
            for (int cb = 0; cb < nb && rc == SDRB_OK; ++cb)
                rc = sdrb_publisher_send_block(pool->pubs[(size_t)k], plan, pcm + ((size_t)i * nb + cb) * rec);
        }
        {
            std::lock_guard<std::mutex> lk(pool->mu);
            if (rc != SDRB_OK) { pool->failed = rc; pool->error = sdrb_last_error(); }
            if (--pool->pending == 0) pool->cv_done.notify_all();
        }
    }
}
}  // namespace

extern "C" int sdrb_publisher_pool_open(const char *address, int bind, int n_sockets, sdrb_publisher_pool **out) {
    if (!address || !out || n_sockets < 1 || n_sockets > 256) { sdrb::set_error("sdrb_publisher_pool_open: bad argument"); return SDRB_E_INVALID; }
    *out = nullptr;
    sdrb_publisher_pool *pool = new sdrb_publisher_pool();
    for (int k = 0; k < n_sockets; ++k) {
        pool->addrs.push_back(n_sockets == 1 ? std::string(address) : pool_address(address, k));
        sdrb_publisher *p = nullptr;
        const int rc = publisher_open(pool->addrs.back().c_str(), bind, 65536, &p);
        if (rc != SDRB_OK) {
            for (sdrb_publisher *q : pool->pubs) sdrb_publisher_close(q);
            delete pool;
            return rc;
        }
        pool->pubs.push_back(p);
    }
    for (int k = 0; k < n_sockets; ++k) pool->workers.emplace_back(pool_worker, pool, k);
    *out = pool;
    return SDRB_OK;
}

extern "C" int sdrb_publisher_pool_sockets(const sdrb_publisher_pool *pool) { return pool ? (int)pool->pubs.size() : 0; }

extern "C" int sdrb_publisher_pool_address(const sdrb_publisher_pool *pool, int k, char *buf, size_t len) {
    if (!pool || !buf || len == 0 || k < 0 || k >= (int)pool->addrs.size()) { sdrb::set_error("sdrb_publisher_pool_address: bad argument"); return SDRB_E_INVALID; }
    snprintf(buf, len, "%s", pool->addrs[(size_t)k].c_str());
    return SDRB_OK;
}

// One job for every sender thread; returns when all of them are done.
static int pool_run(sdrb_publisher_pool *pool, const sdrb_plan *plan, const int16_t *h_pcm, const int32_t *streams, int n_streams,
                    int n_blocks) {
    std::unique_lock<std::mutex> lk(pool->mu);
    pool->plan = plan; pool->pcm = h_pcm; pool->streams = streams; pool->n_streams = n_streams; pool->n_blocks = n_blocks;
    pool->pending = (int)pool->workers.size();
    pool->failed = 0;
    ++pool->gen;
    pool->cv_go.notify_all();
    pool->cv_done.wait(lk, [&] { return pool->pending == 0; });
    if (pool->failed) { sdrb::set_error(pool->error); return pool->failed; }
    return SDRB_OK;
}

extern "C" int sdrb_publisher_pool_send_call(sdrb_publisher_pool *pool, const sdrb_plan *plan, const int16_t *h_pcm, int n_streams, int n_blocks) {
    if (!pool || !plan || (!h_pcm && n_streams > 0 && n_blocks > 0)) { sdrb::set_error("sdrb_publisher_pool_send_call: NULL argument"); return SDRB_E_INVALID; }
    if (n_streams <= 0 || n_blocks <= 0) return SDRB_OK;
    return pool_run(pool, plan, h_pcm, nullptr, n_streams, n_blocks);
}

extern "C" int sdrb_publisher_pool_send_streams(sdrb_publisher_pool *pool, const sdrb_plan *plan, const int16_t *h_pcm,
                                                const int32_t *streams, int n, int n_blocks) {
    static const char *who = "sdrb_publisher_pool_send_streams";
    if (!pool || !plan || !h_pcm || !streams) { sdrb::set_error(std::string(who) + ": NULL argument"); return SDRB_E_INVALID; }
    if (n <= 0 || n_blocks <= 0) { sdrb::set_error(std::string(who) + ": n and n_blocks must be positive"); return SDRB_E_INVALID; }
    std::set<int32_t> seen;
    for (int k = 0; k < n; k++) {
        const char *bad = streams[k] < 0 ? "is negative" : (!seen.insert(streams[k]).second ? "is listed twice" : nullptr);
        if (bad) {
            sdrb::set_error(std::string(who) + ": streams[" + std::to_string(k) + "] = " + std::to_string(streams[k]) + " " + bad);
            return SDRB_E_INVALID;
        }
    }
    return pool_run(pool, plan, h_pcm, streams, n, n_blocks);
}

extern "C" void sdrb_publisher_pool_close(sdrb_publisher_pool *pool) {
    if (!pool) return;
    {
        std::lock_guard<std::mutex> lk(pool->mu);
        pool->quit = true;
    }
    pool->cv_go.notify_all();
    for (std::thread &t : pool->workers) t.join();
    for (sdrb_publisher *p : pool->pubs) sdrb_publisher_close(p);
    delete pool;
}
