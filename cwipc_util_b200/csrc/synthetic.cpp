// synthetic.cpp -- the synthetic source (the universal fake camera of the reference's tests), generating INTO HBM.
// Geometry restated from src/cwipc_synthetic.cpp:182-222: a sqrt(N) x sqrt(N) surface of revolution,
// tile 1/2 by the sign of z, colours driven by a phase angle.  The host computes, once, the 3 * sqrt(N) libm values the
// geometry needs (radius per row, sin / cos per column); get() uploads those few kilobytes and a kernel expands them to
// the N points on the device (pointops.cu: synthetic_kernel) -- no host-to-device copy of points.  The host generator is
// kept behind auxiliary_operation("cuda-host-generate") as the checker of the device one.
#include <chrono>
#include <cinttypes>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "kernels.hpp"
#include "pointcloud.hpp"

using namespace cwcu;

namespace {

using sysclock = std::chrono::system_clock;

class SyntheticSource : public cwipc_activesource {
    int m_side;
    int m_fps;
    float m_angle = 0.f;
    bool m_started = false;
    std::vector<float> m_radius;        // per row
    std::vector<double> m_sin, m_cos;   // per column
    sysclock::time_point m_t0, m_next;
    bool m_have_next = false;

public:
    SyntheticSource(int fps, int npoints) : m_fps(fps) {
        if (npoints == 0) npoints = 160000;
        m_side = (int)std::sqrt((double)npoints); // ref: :45-47, N is rounded down to a square
        const float pi = 3.14159265358979f;
        const float dh = 2.0f / m_side, da = 2 * pi / m_side;
        m_radius.resize(m_side);
        m_sin.resize(m_side);
        m_cos.resize(m_side);
        for (int i = 0; i < m_side; i++) {
            const float h = i * dh, a = i * da;
            m_radius[i] = (float)(0.3 * std::pow(std::cos((double)(h * pi / 3 - pi / 6)), 0.71));
            m_sin[i] = std::sin((double)a);
            m_cos[i] = std::cos((double)a);
        }
    }
    ~SyntheticSource() override {}

    void free() override {}
    bool reload_config(const char *) override {
        log(CWIPC_LOG_LEVEL_WARNING, "cwipc_synthetic", "reload_config() not implemented (nor needed)");
        return false;
    }
    size_t get_config(char *, size_t) override { return 0; }
    bool start() override {
        if (m_started) {
            log(CWIPC_LOG_LEVEL_WARNING, "cwipc_synthetic", "start() called when already started");
            return true;
        }
        m_t0 = sysclock::now();
        m_have_next = false;
        m_started = true;
        return true;
    }
    void stop() override { m_started = false; }
    bool eof() override { return false; }
    bool seek(uint64_t) override { return false; }
    bool available(bool wait) override {
        if (!m_started) {
            log(CWIPC_LOG_LEVEL_ERROR, "cwipc_synthetic", "available() called before start()");
            return false;
        }
        if (!wait && m_fps != 0 && m_have_next && sysclock::now() < m_next) return false;
        return true;
    }
    cwipc_pointcloud *get() override {
        if (!m_started) {
            log(CWIPC_LOG_LEVEL_ERROR, "cwipc_synthetic", "get() called before start()");
            return nullptr;
        }
        if (m_fps != 0 && m_have_next) std::this_thread::sleep_until(m_next);
        const auto now = sysclock::now();
        const uint64_t timestamp = (uint64_t)std::chrono::duration_cast<std::chrono::milliseconds>(now.time_since_epoch()).count();
        if (m_fps != 0) {
            m_next = now + std::chrono::milliseconds(1000 / m_fps);
            m_have_next = true;
        }
        if (!m_angle_forced) m_angle = std::chrono::duration<float>(now - m_t0).count();
        cwipc_pointcloud *rv = generate_on_device(timestamp);
        if (rv) {
            rv->_set_cellsize((float)(2.0 / m_side)); // ref: :131
            if (is_metadata_requested("test-angle")) {
                void *mem = malloc(sizeof(m_angle));
                memcpy(mem, &m_angle, sizeof(m_angle));
                rv->access_metadata()->_add("test-angle", "", mem, sizeof(m_angle), ::free);
            }
        }
        return rv;
    }
    int maxtile() override { return 3; }
    bool get_tileinfo(int tilenum, struct cwipc_tileinfo *tileinfo) override {
        static cwipc_tileinfo info[3] = {
            {{0, 0, 0}, (char *)"synthetic", 2, 0},
            {{0, 0, 1}, (char *)"synthetic-right", 1, 1},
            {{0, 0, -1}, (char *)"synthetic-left", 1, 2},
        };
        if (tilenum < 0 || tilenum > 2) return false;
        if (tileinfo) *tileinfo = info[tilenum];
        return true;
    }
    bool auxiliary_operation(const std::string op, const void *inbuf, size_t insize, void *outbuf, size_t outsize) override {
        if (op == "cuda-host-generate") {
            // the HOST generator for the angle given in inbuf (float), into outbuf (N points): the checker of the device path;
            // the next get() uses the same angle instead of the wall clock
            const size_t n = (size_t)m_side * m_side;
            if (!inbuf || insize != sizeof(float) || !outbuf || outsize != n * sizeof(cwipc_point)) return false;
            memcpy(&m_angle, inbuf, sizeof(float));
            m_angle_forced = true;
            generate(static_cast<cwipc_point *>(outbuf));
            return true;
        }
        if (op != "test-setangle") return false;
        if (!inbuf || insize != sizeof(float) || !outbuf || outsize != sizeof(float)) return false;
        memcpy(&m_angle, inbuf, sizeof(float));
        memcpy(outbuf, &m_angle, sizeof(float));
        return true;
    }

private:
    bool m_angle_forced = false;

    // the cloud of the current angle, made on the device.  ref: src/cwipc_synthetic.cpp:122-131 (get) + :182-222 (generate_points)
    cwipc_pointcloud *generate_on_device(uint64_t timestamp) {
        return guarded<cwipc_pointcloud *>("cwipc_synthetic", nullptr, [&]() -> cwipc_pointcloud * {
            if (device_count() <= 0) throw CudaError{cudaErrorNoDevice, "libcwipc_util_cuda needs a CUDA device and found none (there is no CPU fallback)"};
            const int dev = current_device();
            DeviceGuard g(dev);
            cudaStream_t s = thread_stream(dev);
            const size_t n = (size_t)m_side * m_side;
            const float pi = 3.14159265358979f;
            const float dh = 2.0f / m_side, da = 2 * pi / m_side;
            const bool eyes_lit = std::fmod(m_angle, pi / 2) > 0.08;
            StoragePtr store = new_storage(dev, n, s, [&](Storage &out) {
                Scratch rad(m_side * sizeof(float), s), sn(m_side * sizeof(double), s), cs(m_side * sizeof(double), s);
                if (m_side) {
                    CWCU_CHECK(cudaMemcpyAsync(rad.p, m_radius.data(), m_side * sizeof(float), cudaMemcpyHostToDevice, s));
                    CWCU_CHECK(cudaMemcpyAsync(sn.p, m_sin.data(), m_side * sizeof(double), cudaMemcpyHostToDevice, s));
                    CWCU_CHECK(cudaMemcpyAsync(cs.p, m_cos.data(), m_side * sizeof(double), cudaMemcpyHostToDevice, s));
                    synthetic_points(out.d_pts, m_side, dh, da, rad.as<float>(), sn.as<double>(), cs.as<double>(), m_angle, eyes_lit, s);
                }
                return n;
            });
            auto *pc = new DevicePointcloud(store, timestamp, 0.f);
            pc->set_exact_size(true); // the reference builds this cloud with cwipc_from_points (:127)
            return pc;
        });
    }

    void generate(cwipc_point *out) {
        const float pi = 3.14159265358979f;
        const float dh = 2.0f / m_side, da = 2 * pi / m_side;
        const bool eyes_lit = std::fmod(m_angle, pi / 2) > 0.08;
        for (int hi = 0; hi < m_side; hi++) {
            const float h = hi * dh;
            const float radius = (float)(0.3 * std::pow(std::cos((double)(h * pi / 3 - pi / 6)), 0.71));
            for (int ai = 0; ai < m_side; ai++, out++) {
                const float a = ai * da;
                const float px = (float)(radius * std::sin((double)a));
                const float pz = (float)(radius * std::cos((double)a));
                int c[3];
                for (int k = 0; k < 3; k++) {
                    const float v = (float)((1 + std::sin((double)((k + 2) * pi * h + m_angle + a))) / 2);
                    c[k] = (int)(v * 255.0);
                }
                const bool in_eye = h > 1.7f && h < 1.8f && ((a > pi * 0.083 && a < pi * 0.1667) || (a > pi * 1.833 && a < pi * 1.917));
                if (in_eye && eyes_lit) c[0] = c[1] = c[2] = 255;
                out->x = -px;
                out->y = h;
                out->z = pz;
                out->r = (uint8_t)c[0];
                out->g = (uint8_t)c[1];
                out->b = (uint8_t)c[2];
                out->tile = pz < 0 ? 1 : 2;
            }
        }
    }
};

} // namespace

extern "C" cwipc_activesource *cwipc_synthetic(int fps, int npoints, char **errorMessage, uint64_t apiVersion) {
    if (apiVersion < CWIPC_API_VERSION_OLD || apiVersion > CWIPC_API_VERSION) {
        if (errorMessage) {
            char *msg = (char *)malloc(1024);
            snprintf(msg, 1024, "cwipc_synthetic: incorrect apiVersion 0x%08" PRIx64 " expected 0x%08" PRIx64 "..0x%08" PRIx64 "", apiVersion, (uint64_t)CWIPC_API_VERSION_OLD,
                     (uint64_t)CWIPC_API_VERSION);
            *errorMessage = msg;
        }
        return nullptr;
    }
    return new SyntheticSource(fps, npoints);
}
