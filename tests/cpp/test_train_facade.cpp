// The training half of the C++ TensorCoreQModel (include/ql_cuda.hpp): weights() returns the f32 masters set at creation bit
// for bit, train_replay() on replay transitions by index returns a finite loss and moves the weights, and set_weights() of
// an earlier weights() restores them exactly. Exit code 0 = all checks passed. Needs a B200 (there is no CPU fallback).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "ql_cuda.hpp"

#define CHECK(c, ...) do { if (!(c)) { std::printf("FAIL %s:%d: ", __FILE__, __LINE__); std::printf(__VA_ARGS__); std::printf("\n"); return 1; } } while (0)

using W = ql::TensorCoreQModel::Weights;
static bool same_bits(const W& a, const W& b) {
    const std::vector<float>* x[] = {&a.conv1_kernel, &a.conv1_bias, &a.conv2_kernel, &a.conv2_bias, &a.conv3_kernel, &a.conv3_bias, &a.dense1_kernel, &a.dense1_bias, &a.dense2_kernel, &a.dense2_bias};
    const std::vector<float>* y[] = {&b.conv1_kernel, &b.conv1_bias, &b.conv2_kernel, &b.conv2_bias, &b.conv3_kernel, &b.conv3_bias, &b.dense1_kernel, &b.dense1_bias, &b.dense2_kernel, &b.dense2_bias};
    for (int i = 0; i < 10; ++i) if (x[i]->size() != y[i]->size() || std::memcmp(x[i]->data(), y[i]->data(), x[i]->size() * 4) != 0) return false;
    return true;
}

int main() {
    using namespace ql;
    try {
        BreakoutEnvironment environment(84, 84, /*history_buffer_len=*/4096, /*seed=*/7);
        environment.reset();
        uint64_t r = 5;
        for (int i = 0; i < 200; ++i) {
            r = r * 6364136223846793005ULL + 1442695040888963407ULL;
            auto [s, reward, done] = environment.step(BreakoutActionTrait::try_from_numeric((ModelActionType)((r >> 33) % 3)));
            (void)s; (void)reward;
            if (done) environment.reset();
        }
        W w0;
        auto fill = [&](std::vector<float>& v, float scale) { for (float& x : v) { r = r * 6364136223846793005ULL + 1442695040888963407ULL; x = scale * ((float)((r >> 40) & 0xFFFF) / 32768.0f - 1.0f); } };
        fill(w0.conv1_kernel, 0.02f); fill(w0.conv2_kernel, 0.05f); fill(w0.conv3_kernel, 0.05f); fill(w0.dense1_kernel, 0.02f); fill(w0.dense2_kernel, 0.05f);
        fill(w0.conv1_bias, 0.01f); fill(w0.dense1_bias, 0.01f);
        TensorCoreQModel model(environment, w0.view());
        CHECK(same_bits(model.weights(), w0), "weights() differs from the weights given at creation");
        std::vector<uint32_t> idx(32);
        std::vector<float> targets(32);
        for (uint32_t i = 0; i < 32; ++i) { idx[i] = 5 * i + 3; targets[i] = (float)(i % 3) - 1.0f; }
        const float loss = model.train_replay(idx, targets);
        CHECK(std::isfinite(loss) && loss > 0.0f, "loss %f", loss);
        const W w1 = model.weights();
        CHECK(!same_bits(w1, w0), "an update left every weight unchanged");
        for (float v : w1.dense1_kernel) CHECK(std::isfinite(v), "non-finite weight");
        model.set_weights(w0.view());
        CHECK(same_bits(model.weights(), w0), "set_weights(weights()) is not a round trip");
        bool threw = false;
        try { model.train_replay({100000u}, {0.0f}); } catch (const QlError&) { threw = true; }
        CHECK(threw, "an index beyond the replay was accepted");
        std::printf("train facade ok: loss %.6f\n", loss);
    } catch (const std::exception& e) {
        std::printf("exception: %s\n", e.what());
        return std::strstr(e.what(), "no CUDA device") ? 2 : 1;
    }
    return 0;
}
