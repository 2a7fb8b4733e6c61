/* oracle/layout_mirror.c — TEST INFRASTRUCTURE: sizes and offsets of the layout mirrors in include/vdl2_dropin.h, one
 * "name<TAB>value" line each, under the names oracle/layout_check.c gives the reference's own declarations.
 * tests/test_dropin.py compares them with the reference's values stored in tests/golden/dropin_layout.json. */
#include <stdio.h>
#include <stddef.h>
#include "vdl2_dropin.h"

#define SHOW(what, expr) printf("%s\t%zu\n", what, (size_t)(expr))

int main(void) {
	SHOW("sizeof(vdl2_channel_t)", sizeof(vdl2_channel_t));
	SHOW("offsetof(vdl2_channel_t, demod_thread)", offsetof(vdl2_channel_t, demod_thread));
	SHOW("offsetof(vdl2_channel_t, freq)", offsetof(vdl2_channel_t, freq));
	SHOW("offsetof(vdl2_channel_t, oversample)", offsetof(vdl2_channel_t, oversample));
	SHOW("offsetof(vdl2_channel_t, burst_timestamp)", offsetof(vdl2_channel_t, burst_timestamp));
	SHOW("sizeof(octet_string_t)", sizeof(octet_string_t));
	SHOW("offsetof(octet_string_t, len)", offsetof(octet_string_t, len));
	SHOW("sizeof(vdl2_msg_metadata)", sizeof(vdl2_msg_metadata));
	SHOW("offsetof(vdl2_msg_metadata, idx)", offsetof(vdl2_msg_metadata, idx));
	SHOW("offsetof(vdl2_msg_metadata, burst_timestamp)", offsetof(vdl2_msg_metadata, burst_timestamp));
	SHOW("offsetof(vdl2_msg_metadata, ppm_error)", offsetof(vdl2_msg_metadata, ppm_error));
	return 0;
}
