// host/sampling.h -- Distribution1D with the reference's surface (/root/reference/sampling.h:20-69):
// piecewise-constant 1D distribution.  The constructor builds the running integral and the CDF
// with the reference's float arithmetic (sequential sums of func[i]/n, then division by the
// total); sampling it (SampleContinuous, :38-53) is device code.
#pragma once

#include <vector>        // (no precomp.h: the library's CUDA translation unit builds its light tables with this too)

struct Distribution1D {
	Distribution1D(const float* f, int n) : func(f, f + n), cdf(n + 1) {
		cdf[0] = 0;
		for (int i = 1; i < n + 1; i++) cdf[i] = cdf[i - 1] + func[i - 1] / n;
		funcInt = cdf[n];
		if (funcInt == 0) { for (int i = 1; i < n + 1; i++) cdf[i] = float(i) / float(n); }
		else { for (int i = 1; i < n + 1; i++) cdf[i] /= funcInt; }
	}
	int Count() const { return (int)func.size(); }
	std::vector<float> func, cdf;
	float funcInt;
};
