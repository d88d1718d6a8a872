// main_cli.cpp — headless command line, drop-in for the reference executable's headless branch
// (reference main.cpp: processArgs :22-178, main :201-295, saveImage :180-199): same options, same stdout lines,
// same output files.  The windowed branch (-window / -enable_controls, main.cpp:298-437) needs GLFW/OpenGL and is
// out of scope on a headless B200 server: the flags are parsed and reported, then refused.
// Extra options use a double dash so they cannot collide with the reference's: --device N, --seed S, --slice N,
// --true-mean, --stats, --env-is (sky importance sampling, pt_set_option "env_is"), --light-is (emitter importance sampling,
// pt_set_option "light_is"), --bvh sah|lbvh|auto, and for several GPUs of one box (the reference is fixed to device 0, Pathtracer.cpp:40):
// --gpus N (devices 0..N-1) or --devices MASK, --partition pixels|samples, --exchange p2p|nccl (pt_create_multi).
#include "../../include/pt_b200.h"
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

struct Params // reference Params.h:4-14
{
	unsigned int m_width = 1024;
	unsigned int m_height = 1024;
	unsigned int m_spp = 1024;
	const char *m_inputFilepath = nullptr;
	const char *m_outputFilepath = nullptr;
	bool m_showWindow = false;
	bool m_enableControls = false;
	bool m_outputHdr = false;
	// extensions
	int device = 0;
	unsigned long long seed = 1984;
	unsigned int slice = 0; // samples per launch; 0 = all in one launch
	bool trueMean = false;
	bool stats = false;
	bool envIS = false;
	bool lightIS = false;
	int bvhBuilder = 2; // pt_set_option "bvh_builder": 0 sah, 1 lbvh, 2 auto (the library's default)
	unsigned int deviceMask = 0; // != 0: multi-GPU context over these CUDA ordinals
	int partition = 0;           // 0 pixels, 1 samples
	int exchange = -1;           // -1 auto, 0 nccl, 1 p2p
};

static bool processArgs(int argc, char *argv[], Params &params)
{
	params = Params();
	bool displayHelp = false;
	int i = 1;
	for (; i < (argc - 1);)
	{
		const char *a = argv[i];
		auto numeric = [&](const char *opt, unsigned int &dst)
		{
			if (i + 1 < argc)
			{
				dst = (unsigned int)atoi(argv[i + 1]);
				if (dst == 0) { printf("Invalid input for %s!\n", opt); displayHelp = true; }
			}
			else { printf("Missing argument to %s!\n", opt); displayHelp = true; }
			i += 2;
		};
		if (strcmp(a, "-help") == 0) { displayHelp = true; ++i; }
		else if (strcmp(a, "-w") == 0) numeric("-w", params.m_width);
		else if (strcmp(a, "-h") == 0) numeric("-h", params.m_height);
		else if (strcmp(a, "-spp") == 0) numeric("-spp", params.m_spp);
		else if (strcmp(a, "-window") == 0) { params.m_showWindow = true; ++i; }
		else if (strcmp(a, "-enable_controls") == 0) { params.m_enableControls = true; ++i; }
		else if (strcmp(a, "-ohdr") == 0) { params.m_outputHdr = true; ++i; }
		else if (strcmp(a, "-o") == 0)
		{
			if (i + 1 < argc) params.m_outputFilepath = argv[i + 1];
			else { printf("Missing argument to %s!\n", "-o"); displayHelp = true; }
			i += 2;
		}
		else if (strcmp(a, "--device") == 0 && i + 1 < argc) { params.device = atoi(argv[i + 1]); i += 2; }
		else if (strcmp(a, "--seed") == 0 && i + 1 < argc) { params.seed = strtoull(argv[i + 1], nullptr, 10); i += 2; }
		else if (strcmp(a, "--slice") == 0 && i + 1 < argc) { params.slice = (unsigned int)atoi(argv[i + 1]); i += 2; }
		else if (strcmp(a, "--gpus") == 0 && i + 1 < argc) { const int n = atoi(argv[i + 1]); params.deviceMask = n >= 32 ? 0xffffffffu : (n > 0 ? (1u << n) - 1u : 0u); i += 2; }
		else if (strcmp(a, "--devices") == 0 && i + 1 < argc) { params.deviceMask = (unsigned int)strtoul(argv[i + 1], nullptr, 0); i += 2; }
		else if (strcmp(a, "--partition") == 0 && i + 1 < argc) { params.partition = strcmp(argv[i + 1], "samples") == 0 ? 1 : 0; i += 2; }
		else if (strcmp(a, "--exchange") == 0 && i + 1 < argc) { params.exchange = strcmp(argv[i + 1], "nccl") == 0 ? 0 : (strcmp(argv[i + 1], "p2p") == 0 ? 1 : -1); i += 2; }
		else if (strcmp(a, "--true-mean") == 0) { params.trueMean = true; ++i; }
		else if (strcmp(a, "--env-is") == 0) { params.envIS = true; ++i; }
		else if (strcmp(a, "--light-is") == 0) { params.lightIS = true; ++i; }
		else if (strcmp(a, "--bvh") == 0 && i + 1 < argc) { const char *v = argv[i + 1]; params.bvhBuilder = strcmp(v, "lbvh") == 0 ? 1 : (strcmp(v, "auto") == 0 ? 2 : 0); i += 2; }
		else if (strcmp(a, "--stats") == 0) { params.stats = true; ++i; }
		else
		{
			printf("Can't parse argument: %s\n", a);
			displayHelp = true;
			break;
		}
	}
	if (i < argc && argc > 1) params.m_inputFilepath = argv[argc - 1];
	else if (!(argc == 2 && strcmp(argv[1], "-help") == 0))
	{
		printf("Missing input file argument!\n");
		displayHelp = true;
	}
	if (displayHelp)
	{
		printf("USAGE: PathtracerCUDA.exe [options] <input file>\n\n");
		printf("Options:\n");
		printf("%-30s Display available options\n", "-help");
		printf("%-30s Set width of output image\n", "-w");
		printf("%-30s Set height of output image\n", "-h");
		printf("%-30s Set number of samples per pixel\n", "-spp");
		printf("%-30s Shows a window and displays progressive rendering results\n", "-window");
		printf("%-30s Enables camera controls (WASD to move, RMB+Mouse to rotate). "
		       "If this option is enabled, the result image can only be saved manually by pressing the P key. "
		       "The image is then saved to the filepath specified by %s. %s must be set for this option\n", "-enable_controls", "-o", "-window");
		printf("%-30s Set filepath of output image\n", "-o");
		printf("%-30s Save image as HDR instead of PNG\n", "-ohdr");
		return false;
	}
	params.m_enableControls = params.m_enableControls && params.m_showWindow;
	return true;
}

static void die(const char *what)
{
	// the reference prints the CUDA error and exits with EXIT_FAILURE (Pathtracer.cpp:17-28)
	fprintf(stderr, "%s: %s\n", what, pt_last_error());
	exit(EXIT_FAILURE);
}

static double nowMs()
{
	return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

int main(int argc, char *argv[])
{
	const double t0 = nowMs();
	Params params;
	if (!processArgs(argc, argv, params)) return EXIT_SUCCESS;

	printf("Beginning rendering in configuration:\n");
	printf("Width: %d\n", (int)params.m_width);
	printf("Height: %d\n", (int)params.m_height);
	printf("Samples per Pixel: %d\n", (int)params.m_spp);
	printf("Window: %d\n", (int)params.m_showWindow);
	printf("Controls: %d\n", (int)params.m_enableControls);
	printf("Output HDR: %d\n", (int)params.m_outputHdr);
	printf("Output Filepath: %s\n", params.m_outputFilepath ? params.m_outputFilepath : "");
	printf("Input Filepath: %s\n", params.m_inputFilepath);

	if (params.m_showWindow)
	{
		fprintf(stderr, "-window is not supported by this headless build (no GLFW/OpenGL); run without it.\n");
		return EXIT_FAILURE;
	}

	pt_context *ctx = nullptr;
	if (params.deviceMask != 0)
	{
		if (pt_create_multi(params.m_width, params.m_height, params.deviceMask, &ctx) != PT_OK) die("pt_create_multi");
		pt_set_option(ctx, "partition", (double)params.partition);
		pt_set_option(ctx, "exchange", (double)params.exchange);
	}
	else if (pt_create(params.m_width, params.m_height, params.device, &ctx) != PT_OK) die("pt_create");
	const double tCreate = nowMs();
	pt_set_option(ctx, "seed", (double)params.seed);
	// reference-compatible normalisation: the reference renders 8 samples per render() call and divides by the number
	// of CALLS (quirk Q1); one launch here counts as ceil(spp/8) calls.  --true-mean writes the real mean instead.
	pt_set_option(ctx, "frames_per_spp", 8.0);
	if (params.envIS) pt_set_option(ctx, "env_is", 1.0);
	if (params.lightIS) pt_set_option(ctx, "light_is", 1.0);
	pt_set_option(ctx, "bvh_builder", (double)params.bvhBuilder);

	pt_camera_desc camera;
	const int lr = pt_load_scene_file(ctx, params.m_inputFilepath, &camera);
	if (lr == PT_E_IO) { printf("%s\n", pt_last_error()); return EXIT_FAILURE; }       // "Failed to open input file: ..."
	if (lr == PT_E_PARSE) { printf("%s", pt_last_error()); return EXIT_FAILURE; }      // printf(ex.what())
	if (lr != PT_OK) die("pt_load_scene_file");

	const double tLoad = nowMs();
	const unsigned int slice = params.slice ? params.slice : params.m_spp;
	float totalGpuTime = 0.0f, totalTrace = 0.0f, totalExchange = 0.0f;
	unsigned long long totalRays = 0;
	unsigned int nextReport = 0;
	pt_stats st;
	for (unsigned int i = 0; i < params.m_spp; i += slice)
	{
		const unsigned int spp = std::min(i + slice, params.m_spp) - i;
		// the reference prints progress every 32 samples (main.cpp:282-285): report every multiple of 32 this launch covers
		for (; nextReport < i + spp; nextReport += 32) printf("Accumulated %d samples\n", (int)nextReport);
		if (pt_render(ctx, &camera, spp, i == 0) != PT_OK) die("pt_render");
		totalGpuTime += pt_get_timing_ms(ctx);
		float tr = 0.0f, ex = 0.0f;
		pt_get_multi_info(ctx, nullptr, nullptr, &tr, &ex);
		totalTrace += tr;
		totalExchange += ex;
		pt_get_stats(ctx, &st);
		totalRays += st.rays;
	}
	const double tRender = nowMs();
	printf("Finished accumulating %d samples in %f ms GPU time\n", (int)params.m_spp, totalGpuTime);

	if (params.m_outputFilepath)
	{
		printf("Writing result to %s\n", params.m_outputFilepath);
		int r;
		if (params.m_outputHdr)
		{
			const float *img = params.trueMean ? pt_get_hdr_mean(ctx) : pt_get_hdr(ctx);
			if (!img) die("pt_get_hdr");
			r = pt_write_hdr(params.m_outputFilepath, params.m_width, params.m_height, img);
		}
		else
		{
			if (params.trueMean) pt_set_option(ctx, "frames_per_spp", 1.0);
			const uint8_t *img = pt_get_ldr(ctx);
			if (!img) die("pt_get_ldr");
			r = pt_write_png(params.m_outputFilepath, params.m_width, params.m_height, img);
		}
		if (r != PT_OK) printf("Failed to write file!\n");
	}
	const double tOut = nowMs();
	if (params.stats)
	{
		int devices = 1, p2p = 0;
		pt_get_multi_info(ctx, &devices, &p2p, nullptr, nullptr);
		const unsigned long long imageBytes = (unsigned long long)params.m_width * params.m_height * 16ull;
		printf("{\"rays\": %llu, \"rays_last_launch\": %llu, \"samples_last_launch\": %llu, \"bvh_nodes\": %u, \"bvh_depth\": %u, \"scene_bytes\": %u, \"scene_in_smem\": %u, "
		       "\"devices\": %d, \"partition\": \"%s\", \"exchange\": \"%s\", \"trace_ms\": %f, \"exchange_ms\": %f, \"exchange_bytes_per_device\": %llu, "
		       "\"host_ms\": {\"create\": %.1f, \"load_scene\": %.1f, \"render\": %.1f, \"read_back_and_write\": %.1f}}\n",
		       totalRays, (unsigned long long)st.rays, (unsigned long long)st.samples, st.bvh_nodes, st.bvh_depth, st.scene_bytes, st.scene_in_smem, devices,
		       params.partition ? "samples" : "pixels", devices == 1 ? "none" : (p2p ? "p2p" : "nccl"), totalTrace, totalExchange,
		       devices == 1 ? 0ull : (p2p ? imageBytes / devices : imageBytes), tCreate - t0, tLoad - tCreate, tRender - tLoad, tOut - tRender);
	}
	// The output file is written and closed: leave.  An orderly teardown (pt_destroy: every buffer, texture, stream and event freed
	// one by one, then the CUDA runtime's own atexit work) is for a host that keeps living; a process that ends hands everything back
	// to the driver at once, which is what the user of a command line waits for.  PT_B200_CLI_TEARDOWN=1 asks for the orderly one
	// (leak checkers).
	fflush(stdout);
	fflush(stderr);
	if (getenv("PT_B200_CLI_TEARDOWN")) { pt_destroy(ctx); return EXIT_SUCCESS; }
	_Exit(EXIT_SUCCESS);
}
