# Host build of the product's per-pixel picture code (test harness, see vss_render_emu.cpp).
CXX := $(firstword $(wildcard /usr/bin/g++) g++)
all: libvss_render_emu.so
libvss_render_emu.so: vss_render_emu.cpp ../../rsoccer_isaac_cleanrl_b200/csrc/vss_render.cuh ../../rsoccer_isaac_cleanrl_b200/csrc/vss_lane.cuh ../../include/vss_b200.h
	$(CXX) -O2 -std=c++17 -fPIC -ffp-contract=off -fvisibility=hidden -shared -x c++ -o $@ vss_render_emu.cpp -lm
clean:
	rm -f libvss_render_emu.so
