// kernel_timer.cuh -- the reference's per-kernel timer (ARAP/API/src/util.t:404-510: Timer:startEvent / endEvent /
// evaluate), switched on by Opt_InitializationParameters.collectPerKernelTimingInfo (createwrapper.t:145-146,
// util.t:828-840) and printed when verbosityLevel > 0.  One CUDA event pair per launch, aggregated by kernel name in
// first-seen order at the end of a solve; same table layout and the same two summary lines.
#pragma once
#include "devmem.cuh"
#include <string>
#include <vector>

namespace arapb200 {

class KernelTimer {
public:
    // returns the index of the new event pair (for stop_at)
    size_t start(const char* name, cudaStream_t s)
    {
        Ev e;
        e.name = name;
        e.a = make_event();
        e.b = make_event();
        ARAP_CUDA_CHECK(cudaEventRecord(e.a.get(), s));
        ev_.push_back(std::move(e));
        return ev_.size() - 1;
    }
    void stop_at(size_t idx, cudaStream_t s)
    {
        if (idx < ev_.size()) { ARAP_CUDA_CHECK(cudaEventRecord(ev_[idx].b.get(), s)); ev_[idx].ended = true; }
    }
    void stop(cudaStream_t s) { stop_at(ev_.size() - 1, s); }
    bool empty() const { return ev_.empty(); }

    struct Row {
        std::string name;
        int count;
        float total_ms;
    };
    // Timer:evaluate (util.t:451-510) without the printing: aggregate, then forget the events
    std::vector<Row> aggregate()
    {
        std::vector<Row> rows;
        for (Ev& e : ev_) {
            if (!e.ended) continue;
            float ms = 0.f;
            ARAP_CUDA_CHECK(cudaEventSynchronize(e.b.get()));
            ARAP_CUDA_CHECK(cudaEventElapsedTime(&ms, e.a.get(), e.b.get()));
            size_t i = 0;
            for (; i < rows.size(); ++i)
                if (rows[i].name == e.name) break;
            if (i == rows.size()) rows.push_back(Row{e.name, 0, 0.f});
            rows[i].count += 1;
            rows[i].total_ms += ms;
        }
        ev_.clear();
        return rows;
    }
    // the reference's table + "TIMING" + "Per-iter times" lines (util.t:469-508)
    static std::string format(const std::vector<Row>& rows)
    {
        std::string out;
        char buf[256];
        out += "--------------------------------------------------------\n";
        out += "        Kernel        |   Count  |   Total   | Average \n";
        out += "----------------------+----------+-----------+----------\n";
        for (const Row& r : rows) {
            out += "----------------------+----------+-----------+----------\n";
            snprintf(buf, sizeof(buf), " %-20s |   %4d   | %8.3fms| %7.4fms\n", r.name.c_str(), r.count, r.total_ms,
                     r.total_ms / (float)r.count);
            out += buf;
        }
        out += "--------------------------------------------------------\n";
        out += "TIMING ";
        int linIters = 0, nonLinIters = 0;
        for (const Row& r : rows) {
            const bool init1 = r.name.rfind("PCGInit1", 0) == 0, step1 = r.name.rfind("PCGStep1", 0) == 0;
            if (init1 || step1 || r.name.rfind("overall", 0) == 0) {
                snprintf(buf, sizeof(buf), "%f ", r.total_ms);
                out += buf;
            }
            if (init1) linIters = r.count;   // (sic: the reference's names for the two counters are swapped, :488-497)
            if (step1) nonLinIters = r.count;
        }
        out += "\n";
        float linAggregate = 0.f, nonLinAggregate = 0.f;
        for (const Row& r : rows) {
            if (r.count == linIters) linAggregate += r.total_ms;
            if (r.count == nonLinIters) nonLinAggregate += r.total_ms;
        }
        snprintf(buf, sizeof(buf), "Per-iter times ms (nonlinear,linear): %7.4f\t%7.4f\n", linAggregate, nonLinAggregate);
        out += buf;
        return out;
    }

private:
    struct Ev {
        EventHandle a, b;
        const char* name = "";
        bool ended = false;
    };
    std::vector<Ev> ev_;
};

// wrap one launch: ARAP_TIMED(timer_, "PCGStep1", stream, kernel<<<...>>>(...));
#define ARAP_TIMED(timer, name, stream, launch)                     \
    do {                                                            \
        KernelTimer* t__ = (timer);                                 \
        if (t__) t__->start((name), (stream));                      \
        launch;                                                     \
        if (t__) t__->stop((stream));                               \
    } while (0)

} // namespace arapb200
